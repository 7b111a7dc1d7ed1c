"""CUDA-event times of the elementwise kernels whose code moved onto the shared arithmetic and launch helpers, for two
builds of the library alternated in one session: the binary ops with a shorter operand (smaller_kernel), complex math
(math_complex_kernel), set_real_imag / set_mag_phase (compose_kernel), the row-broadcast spectrum multiply of chirp-z
transforms and of the full-length convolution, and the full-length convolution of real signals (its complex-to-real
pass).  Inputs are 2^26 points (c32 and c64), above the 126 MB L2.  Every in-place call starts from the same input: it
is restored by a device copy outside the timed window.

    python scratch/bench_elementwise.py --lib A.so --lib B.so [--rounds 3] [--iters 15]

Each round runs every library once, in a fresh process, in the order given; the table shows per case and library the
median of the per-round medians and the spread (max - min) of those medians over the rounds."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 1 << 26


def worker(iters):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import basic_dsp_b200 as bd
    L = bd.lib()
    bd.require_device()
    L.bdsp_set_stream(torch.cuda.current_stream().cuda_stream)
    DspVec = bd.DspVec
    res = {}

    class _Cai:   # the vector's device storage, seen by torch as bytes
        def __init__(self, v):
            nbytes = v.len() * np.dtype(v._T).itemsize
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (v._fn("bdsp_device_ptr")(v._h), False),
                                             "version": 2}

    def storage(v):
        return torch.as_tensor(_Cai(v), device="cuda")

    def timed(key, fn, prep=lambda: None, warmup=2):
        for _ in range(warmup):
            prep()
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            prep()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        res[key] = statistics.median(ts)

    def in_place(key, x, call):
        v = DspVec(x)
        saved = storage(v).clone()
        timed(key, lambda: call(v), lambda: storage(v).copy_(saved))
        del v

    rng = np.random.default_rng(0)
    for dtype in (np.float32, np.float64):
        name = "c32" if dtype == np.float32 else "c64"
        ct = np.complex64 if dtype == np.float32 else np.complex128
        z = (rng.uniform(-2, 2, N) + 1j * rng.uniform(-2, 2, N)).astype(ct)
        r = rng.uniform(-10, 10, N).astype(dtype)
        # operands of magnitude 1 keep repeated calls away from overflow
        wz = np.exp(1j * rng.uniform(-3, 3, 4096)).astype(ct)
        wr = rng.choice([-1.0, 1.0], 4096).astype(dtype)
        for op in ("add", "sub", "mul", "div"):
            wv, wzv = DspVec(wr), DspVec(wz)
            in_place("smaller %s real %s" % (name, op), r, lambda v: getattr(v, op + "_smaller")(wv))
            in_place("smaller %s complex %s" % (name, op), z, lambda v: getattr(v, op + "_smaller")(wzv))
        for op in ("sqrt", "square", "exp", "ln", "sin"):
            in_place("math %s complex %s" % (name, op), z, lambda v: v.math(op))
        re, im = DspVec(z.real.copy()), DspVec(z.imag.copy())
        mag, ph = DspVec(np.abs(z).astype(dtype)), DspVec(np.angle(z).astype(dtype))
        out = DspVec(np.zeros(2, dtype=ct))
        out.set_real_imag(re, im)
        timed("compose %s set_real_imag" % name, lambda: out.set_real_imag(re, im))
        timed("compose %s set_mag_phase" % name, lambda: out.set_mag_phase(mag, ph))
        del re, im, mag, ph, out
        # full-length convolution of a real signal: taps beyond the overlap-save blocks, complex-to-real pass at the end
        taps = 9000 if dtype == np.float32 else 5000
        h = DspVec((rng.uniform(-1, 1, taps)).astype(dtype))
        in_place("conv-full real %s N=2^26 L=%d" % (name, taps), r, lambda v: v.convolve_signal(h))
        del h
        torch.cuda.empty_cache()
    # the row-broadcast spectrum multiply: chirp-z rows (M = 16384) and full-length convolution rows of 16384 points
    x = torch.randn(4096 * 4099, dtype=torch.complex64, device="cuda")
    y = torch.empty_like(x)
    timed("chirp-z fft c32 n=4099 x4096 (M=16384)", lambda: L.bdsp_fft_rows_c32(x.data_ptr(), y.data_ptr(), 4099, 4096, 0))
    del x, y
    x = torch.randn(N, dtype=torch.complex64, device="cuda")
    y = torch.empty_like(x)
    hv = DspVec((rng.uniform(-1, 1, 9000) + 1j * rng.uniform(-1, 1, 9000)).astype(np.complex64) / 10)
    plan = L.bdsp_conv_plan_create_c32(hv._fn("bdsp_device_ptr")(hv._h), 9000)
    timed("conv-full rows c32 N=16384 x4096 L=9000", lambda: L.bdsp_convolve_signal_rows_c32(x.data_ptr(), y.data_ptr(), 16384, 4096, plan))
    L.bdsp_conv_plan_destroy(plan)
    print("RESULT " + json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=15)
    ap.add_argument("--worker", action="store_true")
    args = ap.parse_args()
    if args.worker:
        return worker(args.iters)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    print("card: %s" % (smi[0] if smi else "nvidia-smi unavailable"))
    runs = {lib: [] for lib in args.lib}
    for rnd in range(args.rounds):
        for lib in args.lib:
            env = dict(os.environ, BASIC_DSP_B200_LIB=os.path.abspath(lib))
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--iters", str(args.iters)], env=env,
                                 capture_output=True, text=True)
            line = [l for l in out.stdout.splitlines() if l.startswith("RESULT ")]
            if out.returncode or not line:
                print(out.stdout[-3000:], out.stderr[-3000:])
                raise SystemExit("worker failed for %s" % lib)
            runs[lib].append(json.loads(line[0][7:]))
            print("round %d %s done" % (rnd, lib), flush=True)
    keys = list(runs[args.lib[0]][0])
    hdr = "%-44s" % "case (ms, median of round medians / spread)"
    for i, lib in enumerate(args.lib):
        hdr += " | %-22s" % ("lib %d" % i)
    print("\n" + "\n".join("lib %d: %s" % (i, lib) for i, lib in enumerate(args.lib)))
    print(hdr + " | ratio 1/0")
    for k in keys:
        row, meds = "%-44s" % k, []
        for lib in args.lib:
            v = [r[k] for r in runs[lib]]
            meds.append(statistics.median(v))
            row += " | %8.4f  spread %6.4f" % (meds[-1], max(v) - min(v))
        if len(meds) > 1:
            row += " | %.3f" % (meds[1] / meds[0])
        print(row)


if __name__ == "__main__":
    main()
