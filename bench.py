#!/usr/bin/env python3
"""Benchmark of the hot path named by BASELINE.json: c32 FFT fast convolution, 2^20-point vectors,
batched, on 1/2/4/8 B200 (weak scaling: every GPU convolves its own rows, no collective).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU algorithm (C port), host cores

One step = one pass of `convolve_signal` (1023-tap raised cosine, SURVEY.md section 8 config C2a-B)
over ROWS = 64 independent 2^20-point complex f32 vectors per GPU (512 MiB in, 512 MiB out: larger than
the 126 MB L2, so no L2 flush is needed between iterations).  Rank 0 prints ONE JSON line.

--dump-outputs DIR writes rank 0's results of the last device-resident step and of the last end-to-end step
as a fixed sample (see output_sample) to DIR/*.npy, float32 (re, im) pairs, 48 MiB in all.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POINTS = 1 << 20
TAPS = 1023
ROWS = 64
METRIC = "Msamples/s c32 FFT fast-conv 2^20 batched"
WORKLOAD = "C2a-B: convolve_signal, %d x 2^20-point c32 vectors per GPU, %d-tap RaisedCosine(0.35) h[k]=RC((k-511)*0.25)" % (ROWS, TAPS)


def make_taps():
    """h[k] = RC_0.35((k - 511) * 0.25) evaluated in f32 like the reference (conv_types.rs:406-423)."""
    k = np.arange(TAPS, dtype=np.float32)
    x = ((k - np.float32(511)) * np.float32(0.25)).astype(np.float32)
    pi = np.float32(np.pi)
    beta = np.float32(0.35)
    with np.errstate(divide="ignore", invalid="ignore"):
        pi_x = pi * x
        arg = np.float32(2) * beta * x
        v = np.sin(pi_x) * np.cos(pi_x * beta) / pi_x / (np.float32(1) - arg * arg)
    v = v.astype(np.float32)
    v[x == 0] = 1.0
    return v.astype(np.complex64)


def make_rows(rows, seed):
    rng = np.random.default_rng(seed)
    out = np.empty((rows, N_POINTS), dtype=np.complex64)
    for r in range(rows):  # re, im i.i.d. uniform [-10, 10) (tests/tools/mod.rs:124-131)
        out[r].real = rng.uniform(-10, 10, N_POINTS).astype(np.float32)
        out[r].imag = rng.uniform(-10, 10, N_POINTS).astype(np.float32)
    return out


def output_sample(y):
    """Fixed sample of a (ROWS, N_POINTS) complex64 result: two whole rows (their edges included) and 2^20 points
    drawn over all rows, as float32 arrays of (re, im) pairs (16 MiB + 8 MiB)."""
    rng = np.random.default_rng(20261020)
    rows = np.sort(rng.choice(ROWS, 2, replace=False))
    flat = np.sort(rng.integers(0, ROWS * N_POINTS, 1 << 20))
    return {"rows": y[rows].view(np.float32).reshape(len(rows), N_POINTS, 2),
            "points": y.reshape(-1)[flat].view(np.float32).reshape(-1, 2)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.time()] + [c.strip() for c in line.split(",")])

    def summary(self, t0=None, t1=None):
        """Median SM clock / throttle reasons of the samples taken in [t0, t1] (all samples when None)."""
        rows = [r[1:] for r in self.rows if (t0 is None or r[0] >= t0 - 0.05) and (t1 is None or r[0] <= t1 + 0.05)]
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        return self.summary()


def cpu_port_rate(rows, threads, steps=1, warmup=0):
    """Msamples/s of the C port of the reference's CPU path on `rows` vectors with `threads` threads."""
    from oracle import ref_port
    x0 = make_rows(rows, 20260102)
    h = make_taps()
    times = []
    for it in range(warmup + steps):
        x = x0.copy()
        t0 = time.perf_counter()
        rc = ref_port.convolve_signal_rows_inplace(x, h, threads)
        dt = time.perf_counter() - t0
        if rc:
            raise RuntimeError("reference port failed: %d" % rc)
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return rows * N_POINTS * len(times) / total / 1e6, total / len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    rows = cores  # bounded sample: one 2^20-point vector per host thread per step (~1 s of CPU each)
    warm = min(args.warmup, 1)
    steps = max(1, min(args.steps, 5))
    rate, sec = cpu_port_rate(rows, cores, steps=steps, warmup=warm)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": "%d rows of 2^20 points per step on %d host threads" % (rows, cores)},
        "cpu_baseline": {"value": rate, "unit": "Msamples/s", "cores": cores, "kind": "port",
                         "sample": "%d x 2^20-point vectors per step, %d steps, C port of overlap_discard incl. its scalar head/tail "
                                   "loops (oracle/ref_port.c), one OpenMP thread per vector" % (rows, steps)},
        "e2e": {"value": rate, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import basic_dsp_b200 as bd

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    # one disjoint slice of the host's CPUs per rank (before the pinned buffers are allocated and first touched): the
    # end-to-end path is bound by the host <-> device link, and ranks that migrate over each other's cores and memory make it worse
    affinity = None
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cpus) >= world:
            per = len(cpus) // world
            affinity = cpus[local * per:(local + 1) * per]
            os.sched_setaffinity(0, affinity)
    except (AttributeError, OSError):
        affinity = None
    L = bd.lib()
    if L.bdsp_set_device(local) != 0:
        raise SystemExit("bdsp_set_device failed: %s" % L.bdsp_last_error())
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        L.bdsp_sync()

    # ---- inputs: this rank's shard (rows [rank*ROWS, (rank+1)*ROWS) of the global batch) ------------
    nbytes = ROWS * N_POINTS * 8
    h = make_taps()
    host_in = L.bdsp_malloc_host(nbytes)
    host_out = L.bdsp_malloc_host(nbytes)
    if not host_in or not host_out:
        raise SystemExit("pinned host allocation failed")
    hin = np.ctypeslib.as_array((ctypes.c_float * (2 * ROWS * N_POINTS)).from_address(host_in))
    hout = np.ctypeslib.as_array((ctypes.c_float * (2 * ROWS * N_POINTS)).from_address(host_out))
    dumps = {}
    from basic_dsp_b200.sharding import row_shard
    row0, row1 = row_shard(world * ROWS, world, rank)     # weak scaling: ROWS rows per GPU, contiguous blocks
    assert row1 - row0 == ROWS
    hin[:] = make_rows(ROWS, 20260102 + row0).view(np.float32).ravel()
    d_in, d_out, d_h = L.bdsp_malloc(nbytes), L.bdsp_malloc(nbytes), L.bdsp_malloc(TAPS * 8)
    if not d_in or not d_out or not d_h:
        raise SystemExit("device allocation failed: %s" % L.bdsp_last_error())
    L.bdsp_memcpy_h2d(d_in, host_in, nbytes)
    L.bdsp_memcpy_h2d(d_h, h.ctypes.data, TAPS * 8)
    L.bdsp_sync()
    plan = L.bdsp_conv_plan_create_c32(d_h, TAPS)
    if not plan:
        raise SystemExit("conv plan failed: %s" % L.bdsp_last_error())

    def step():
        rc = L.bdsp_convolve_signal_rows_c32(d_in, d_out, N_POINTS, ROWS, plan)
        if rc:
            raise SystemExit("bdsp_convolve_signal_rows_c32 -> %d (%s)" % (rc, L.bdsp_last_error()))

    # ---- device-resident throughput ---------------------------------------------------------------------------
    # nvidia-smi samples every ~25 ms while the K timed steps last a few milliseconds: the clock record therefore covers
    # the window from the warm-up through the K timed steps to the end of the end-to-end steps (both timed regions of
    # this line), without any artificial load (a sustained load of this kernel runs into the 1000 W power cap after
    # ~0.2 s - 1837 MHz, 5 % slower - which a run of K = 20 steps never reaches).
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.1)
    t_load0 = time.time()
    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = bd.kernel_launch_count()
    evs = [L.bdsp_event_create() for _ in range(args.steps + 1)]
    barrier()
    L.bdsp_event_record(evs[0])
    for i in range(args.steps):
        step()
        L.bdsp_event_record(evs[i + 1])
    barrier()
    total_ms = L.bdsp_event_elapsed_ms(evs[0], evs[args.steps])
    per_launch_ms = [L.bdsp_event_elapsed_ms(evs[i], evs[i + 1]) for i in range(args.steps)]
    launches = bd.kernel_launch_count() - launches0
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    samples = world * ROWS * N_POINTS * args.steps
    value = samples / (total_ms_max * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        L.bdsp_memcpy_d2h(host_out, d_out, nbytes)
        L.bdsp_sync()
        for k_, a in output_sample(hout.view(np.complex64).reshape(ROWS, N_POINTS)).items():
            dumps["device_" + k_] = a

    # ---- end to end through the C ABI with HOST buffers: upload -> convolve_signal32 -> download, every step --------
    # Rows are pipelined over DEPTH (stream, vector handle) pairs so that the upload of row r+1, the kernel
    # of row r and the download of row r-1 overlap (PCIe is full duplex); every call is the reference's
    # per-vector C-ABI entry point.
    DEPTH = int(os.environ.get("BDSP_E2E_DEPTH", "3"))
    hv = bd.DspVec(h)
    hv_warm = bd.DspVec.zeros(2 * N_POINTS, is_complex=True, dtype=np.float32)
    hv_warm.convolve_signal(hv)   # builds and caches the impulse-response spectrum inside `hv`
    L.bdsp_sync()
    streams = [L.bdsp_stream_create() for _ in range(DEPTH)]
    vecs = [bd.DspVec.zeros(2 * N_POINTS, is_complex=True, dtype=np.float32) for _ in range(DEPTH)]
    for v_ in vecs:                 # allocate each handle's scratch once, outside the timed region
        v_.convolve_signal(hv)
    L.bdsp_sync()
    fptr = ctypes.POINTER(ctypes.c_float)
    row_floats = 2 * N_POINTS

    def e2e_step():
        for r in range(ROWS):
            k = r % DEPTH
            L.bdsp_set_stream(streams[k])
            vec = vecs[k]
            src = ctypes.cast(host_in + r * row_floats * 4, fptr)
            dst = ctypes.cast(host_out + r * row_floats * 4, fptr)
            if L.bdsp_upload32(vec._h, src, row_floats):
                raise SystemExit("upload failed")
            vec.convolve_signal(hv)
            if L.bdsp_download_async32(vec._h, dst, row_floats):
                raise SystemExit("download failed")
        for st in streams:
            L.bdsp_stream_sync(st)
        L.bdsp_set_stream(None)

    e2e_steps = max(1, min(args.steps, 10))
    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:
        for k_, a in output_sample(hout.view(np.complex64).reshape(ROWS, N_POINTS)).items():
            dumps["e2e_" + k_] = a
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * ROWS * N_POINTS * e2e_steps / float(t.item()) / 1e6
    t_load1 = time.time()
    clocks = sampler.summary(t_load0, t_load1) if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + the K timed steps + the end-to-end steps (%.2f s)" % (t_load1 - t_load0)

    # ---- what the box's host <-> device path allows: the same pinned buffers copied up and down concurrently (two
    # streams, all ranks at once, nothing else running), i.e. the ceiling of any end-to-end number on this machine
    s_up, s_dn = streams[0], streams[1 % DEPTH]

    def copy_step():
        L.bdsp_set_stream(s_up)
        L.bdsp_memcpy_h2d(d_in, host_in, nbytes)
        L.bdsp_set_stream(s_dn)
        L.bdsp_memcpy_d2h(host_out, d_out, nbytes)
        L.bdsp_stream_sync(s_up)
        L.bdsp_stream_sync(s_dn)
        L.bdsp_set_stream(None)

    copy_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        copy_step()
    barrier()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    copy_ceiling_gbs = world * 2.0 * nbytes * 3 / float(t.item()) / 1e9          # aggregate, both directions
    e2e_gbs = e2e_value * 1e6 * 16.0 / 1e9                                       # 8 B up + 8 B down per sample
    # the e2e result of the last row must equal the device-resident result (same kernel, same input)
    chk = np.empty(row_floats, dtype=np.float32)
    L.bdsp_memcpy_d2h(chk.ctypes.data, d_out + (ROWS - 1) * row_floats * 4, row_floats * 4)
    L.bdsp_sync()
    # (the per-vector call and the batched call may pick different block lengths, so equal up to rounding)
    a64, b64 = chk.astype(np.float64), hout[(ROWS - 1) * row_floats:].astype(np.float64)
    rel = float(np.linalg.norm(a64 - b64) / np.linalg.norm(a64))
    if not rel <= 2e-5:
        raise SystemExit("e2e result differs from the device-resident result (rel L2 %.3e)" % rel)

    if rank == 0:
        peak, peak_src = peaks()
        alg_bytes = 16.0 * N_POINTS * ROWS          # SURVEY.md 8(d): 16 B per sample (8 read + 8 write)
        avg_ms = statistics.mean(per_launch_ms)
        achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
        flops = ROWS * N_POINTS * (2 * 5 * 20 + 6)   # 5 N log2 N convention, forward + inverse + multiply
        line = {
            "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "rows_per_gpu": ROWS, "points": N_POINTS, "taps": TAPS,
                       "l2": "inputs larger than L2 (512 MiB in + 512 MiB out per step), no flush",
                       "sharding": "rows, no collective", "cpus_per_rank": len(affinity) if affinity else None},
            "gflops_5nlog2n": flops * world / (total_ms_max / args.steps * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": 1030119424.0, "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch (profiles/r2_ols4096i_ncu.txt)",
                         "kernel": "ols4096i_kernel<true>", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms,
                         "min_launch_ms": min(per_launch_ms)},
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                    "steps": e2e_steps, "path": "per row: bdsp_upload32 -> convolve_signal32 -> bdsp_download_async32, pinned host buffers, 3 streams in flight",
                    "host_link_GBps": e2e_gbs, "copy_ceiling_GBps": copy_ceiling_gbs, "frac_of_copy_ceiling": e2e_gbs / copy_ceiling_gbs,
                    "copy_ceiling": "aggregate over all ranks of concurrent pinned H2D + D2H cudaMemcpyAsync of the same buffers, no kernels"},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if world == 1 and not args.no_configs:
            # every other BASELINE config, device resident, CUDA events, with the clocks sampled while it ran
            import bench_configs
            lines = bench_configs.measure(set("C1,C2a,C2b,C3,C4a,C4b,C5a,C5b".split(",")), 10, emit=False)
            cfgs = {}
            prev_end = time.time()
            for ln in lines:
                key = ln["config"] + (" (L2 flushed)" if "flushed" in ln["what"] else " (L2 warm)" if "warm" in ln["what"] else "")
                cfgs[key] = {"what": ln["what"], "ms": ln["ms_median"], "ms_best": ln["ms_best"], "Msamples_per_s": ln["Msamples_per_s"],
                             "algorithmic_bytes": ln["algorithmic_bytes"], "achieved_GBps": ln["achieved_GBps"], "frac": ln["roofline_frac"]}
            t_cfg1 = time.time()
            ck = sampler.summary(t_load1, t_cfg1)
            for k_ in cfgs:
                cfgs[k_]["clocks"] = ck
            line["configs"] = cfgs
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            rate, sec = cpu_port_rate(cores, cores, steps=3, warmup=1)   # same protocol as --impl reference
            line["cpu_baseline"] = {"value": rate, "unit": "Msamples/s", "cores": cores, "kind": "port",
                                    "sample": "%d x 2^20-point vectors (one per host thread) per step, 1 warm-up + 3 timed steps of %.2f s; "
                                              "C port of the reference's overlap_discard incl. scalar head/tail (oracle/ref_port.c)" % (cores, sec)}
        print(json.dumps(line))
        sampler.stop()
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    barrier()
    L.bdsp_conv_plan_destroy(plan)
    for p in (d_in, d_out, d_h):
        L.bdsp_free(p)
    L.bdsp_free_host(host_in)
    L.bdsp_free_host(host_out)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config measurements (C1 ... C5b) on the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last step's results to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
