"""bdsp_welch_c32 / _c64 (Welch's averaged periodogram) against what a caller does without it, on the library's stream:
  (a) bdsp_fft_frames_c32 with BDSP_F_MAGNITUDE (every frame's |X| to HBM), then the square and the mean over frames in torch;
  (b) torch.stft(center=False) with the library's window table, then abs()^2 and the mean.
Median and best of CUDA-event timings after warm-up; algorithmic bytes = the signal read once (hop * frames points; the
L2 re-reads of overlapping frames are not counted) plus the output; the HBM peak is a device-to-device copy measured in
the same run.  Every output is compared with a float64 reference computed on the GPU with torch (relative L2 error).

    python scratch/bench_welch.py [--iters 20] [--fused-only]      (results: profiles/r3_welch.txt)

Workloads (the three of profiles/r3_fft_frames.txt, with their natural frame counts; inputs above the 126 MB L2):
  1. real f32 signal of 2^28 samples, 1024-point Hamming frames, hop 256, one-sided density: 1048573 frames, one frame
     past whole groups of 4 (the fused kernel takes the incomplete group);
  2. c32 signal of 2^26 points, 4096-point Blackman-Harris frames, hop 2048, fftshift order;
  3. c32 signal of 2^26 points, 256-point rectangular frames, hop 128, power spectrum: 15 frames past whole groups of 16;
  4. (general path) real f64 signal of 2^27 samples, 1024-point Hamming frames, hop 256, one-sided density.
--fused-only times the library call alone (for comparing builds, selected with BASIC_DSP_B200_LIB)."""
import argparse
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import basic_dsp_b200 as bd  # noqa: E402

FS = 1.0


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times), min(times)


def hbm_peak(iters):
    a = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    med, best = timed(lambda: b.copy_(a), iters)
    del a, b
    return 2 * (1 << 32) / best / 1e6   # GB/s, read + write


def library_window(kind, points, dtype):
    if kind is None:
        return np.ones(points, dtype=dtype)
    return bd.DspVec(np.ones(points, dtype=dtype), is_complex=False, dtype=dtype).apply_window(kind).to_numpy()


def finish(p, w, frames, flags, points):
    """mean |X|^2 (two-sided, fftfreq order; or one-sided bins 0 .. points/2) -> the bdsp_welch_* output"""
    w = w.double()
    den = w.sum() ** 2 if flags & bd.F_POWER_SPECTRUM else FS * (w * w).sum()
    out = p.double() / den
    if flags & bd.F_ONESIDED:
        out = out[:points // 2 + 1].clone()
        out[1:points // 2 + points % 2] *= 2
    elif flags & bd.F_SHIFT:
        out = torch.roll(out, points // 2)
    return out


def reference(x, points, hop, frames, w, flags):
    """float64 closed form on the GPU, in chunks of frames"""
    xd = x.to(torch.complex128 if x.is_complex() else torch.float64)
    wd = w.double()
    acc = torch.zeros(points, dtype=torch.float64, device="cuda")
    step = max(1, (1 << 25) // points)
    for f0 in range(0, frames, step):
        seg = xd[f0 * hop:].unfold(0, points, hop)[:min(step, frames - f0)]
        acc += (torch.fft.fft(seg * wd).abs() ** 2).sum(0)
    return finish(acc / frames, w, frames, flags, points)


def rel_l2(a, ref):
    return float(torch.linalg.vector_norm(a.double() - ref) / torch.linalg.vector_norm(ref))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--fused-only", action="store_true")
    args = ap.parse_args()
    L = bd.lib()
    bd.require_device()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    print("card: %s (torch: %s)  library: %s" % (smi[0] if smi else "nvidia-smi unavailable", torch.cuda.get_device_name(), bd.LIB_PATH))
    stream = torch.cuda.current_stream()
    L.bdsp_set_stream(stream.cuda_stream)   # torch's kernels and the library's on one stream
    peak = hbm_peak(args.iters)
    print("HBM peak (device-to-device copy, best of %d): %.0f GB/s" % (args.iters, peak))
    print("%-56s %7s %9s %9s %9s %8s %7s %10s" % ("workload", "frames", "path", "median ms", "best ms", "GB/s", "of peak", "rel L2"))
    g = torch.Generator(device="cuda").manual_seed(0)
    R, ONE, PSD, SH = bd.F_REAL_INPUT, bd.F_ONESIDED, bd.F_POWER_SPECTRUM, bd.F_SHIFT
    workloads = [
        ("real 2^28, 1024 Hamming, hop 256, one-sided density", torch.float32, True, 1 << 28, 1024, 256, bd.HAMMING, R | ONE),
        ("c32 2^26, 4096 Blackman-Harris, hop 2048, shift", torch.float32, False, 1 << 26, 4096, 2048, bd.BLACKMAN_HARRIS, SH),
        ("c32 2^26, 256 rectangular, hop 128, power spectrum", torch.float32, False, 1 << 26, 256, 128, None, PSD),
        ("real f64 2^27, 1024 Hamming, hop 256, one-sided (general)", torch.float64, True, 1 << 27, 1024, 256, bd.HAMMING, R | ONE),
    ]
    for name, rdt, real, length, points, hop, kind, flags in workloads:
        c32 = rdt == torch.float32
        npdt = np.float32 if c32 else np.float64
        if real:
            x = torch.rand(length, generator=g, device="cuda", dtype=rdt) * 2 - 1
        else:
            x = torch.view_as_complex(torch.rand(length, 2, generator=g, device="cuda", dtype=rdt) * 2 - 1)
        frames = 1 + (length - points) // hop
        wflag = bd.F_WINDOW(kind) if kind is not None else 0
        w = torch.from_numpy(library_window(kind, points, npdt)).cuda()
        nout = points // 2 + 1 if flags & ONE else points
        out = torch.empty(nout, device="cuda", dtype=rdt)
        welch = L.bdsp_welch_c32 if c32 else L.bdsp_welch_c64

        def fused():
            assert welch(x.data_ptr(), out.data_ptr(), points, hop, frames, flags | wflag, FS) == 0, L.bdsp_last_error()

        esz = x.element_size()
        nbytes = hop * frames * esz + nout * out.element_size()
        ref = reference(x, points, hop, frames, w, flags)
        paths = [("welch", fused, lambda: out)]
        if c32 and not args.fused_only:
            mag = torch.empty(frames, points, device="cuda", dtype=torch.float32)
            res = {}

            def frames_mag():
                f = (flags & R) | wflag | bd.F_MAGNITUDE   # fftshift and fold in finish()
                assert L.bdsp_fft_frames_c32(x.data_ptr(), mag.data_ptr(), points, hop, frames, f) == 0, L.bdsp_last_error()
                res["a"] = finish(mag.square().mean(0), w, frames, flags, points)

            def stft():
                S = torch.stft(x, n_fft=points, hop_length=hop, win_length=points, window=w, center=False,
                               onesided=bool(flags & ONE), return_complex=True)      # bins x frames
                res["b"] = finish(S.abs().square().mean(1), w, frames, flags, points)

            paths += [("(a) frames|X|", frames_mag, lambda: res["a"]), ("(b) stft", stft, lambda: res["b"])]
        for label, run, result in paths:
            med, best = timed(run, args.iters)
            gbs = nbytes / med / 1e6
            torch.cuda.synchronize()
            print("%-56s %7d %9s %9.3f %9.3f %8.0f %6.1f%% %10.2e" % (name, frames, label, med, best, gbs, 100 * gbs / peak,
                                                                    rel_l2(result(), ref)))
        del x
        torch.cuda.empty_cache()
    L.bdsp_set_stream(None)


if __name__ == "__main__":
    main()
