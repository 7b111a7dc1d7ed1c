"""bdsp_ifft_frames_c32/c64 (inverse short-time transform: inverse rows, then a weighted overlap-add kernel) against
torch.istft(center=False, onesided=False, return_complex=True) on the same device spectra with the same window tensor,
and bdsp_fft_rows_*(INVERSE | SHIFT) alone, which is the inverse-transform share of the call.  Median and best of
CUDA-event timings after warm-up; every input is above the 126 MB L2.

    python scratch/bench_ifft_frames.py [--iters 20]      (results: profiles/r3_ifft_frames.txt)

Workloads (the forward benchmark's, scratch/bench_fft_frames.py, with a c64 case added); the spectra are what
bdsp_fft_frames_* writes for a random signal:
  1. 1024-point Hamming frames of a real 2^28-sample signal, hop 256, real output;
  2. 4096-point Blackman-Harris frames of a c32 signal of 2^26 points, hop 1024, shift;
  3. 256-point rectangular frames of a c32 signal of 2^26 points, hop 128;
  4. 1024-point Hamming frames of a c64 signal of 2^25 points, hop 256, shift.
Bytes per call, e = bytes per complex point, o = bytes per output point, P x F spectrum points, len output points:
  two-stage (what the library does: spectra in, frames out, frames in again, signal out) = 3 e P F + o len;
  fused ideal (spectra in, signal out)                                                    = e P F + o len.
GB/s is the two-stage bytes over the median; "of 7.7 TB/s" is that rate over the B200 data-sheet HBM bandwidth, and
"fused x" is the median over the fused ideal's time at 7.7 TB/s."""
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
from oracle import accuracy as acc  # noqa: E402

HBM = 7.7e12   # B/s, HGX B200 data sheet, one GPU


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    L = bd.lib()
    bd.require_device()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    print("card: %s (torch: %s)" % (smi[0] if smi else "nvidia-smi unavailable", torch.cuda.get_device_name()))
    stream = torch.cuda.current_stream()
    L.bdsp_set_stream(stream.cuda_stream)   # torch's kernels and the library's on one stream
    print("%-46s %7s %9s %9s %9s %8s %8s %8s" % ("workload", "frames", "path", "median ms", "best ms", "GB/s", "of 7.7", "fused x"))
    g = torch.Generator(device="cuda").manual_seed(0)
    workloads = [
        ("real 2^28, 1024 Hamming, hop 256, real out", 4, True, 1 << 28, 1024, 256, bd.HAMMING, 0),
        ("c32 2^26, 4096 Blackman-Harris, hop 1024, shift", 4, False, 1 << 26, 4096, 1024, bd.BLACKMAN_HARRIS, bd.F_SHIFT),
        ("c32 2^26, 256 rectangular, hop 128", 4, False, 1 << 26, 256, 128, None, 0),
        ("c64 2^25, 1024 Hamming, hop 256, shift", 8, False, 1 << 25, 1024, 256, bd.HAMMING, bd.F_SHIFT),
    ]
    for name, rsz, real, length, points, hop, kind, shift in workloads:
        rt, ct = (torch.float32, torch.complex64) if rsz == 4 else (torch.float64, torch.complex128)
        s = "c32" if rsz == 4 else "c64"
        x = torch.rand(length if real else 2 * length, generator=g, device="cuda", dtype=rt) * 2 - 1
        if not real:
            x = torch.view_as_complex(x.view(length, 2))
        frames = 1 + (length - points) // hop
        out_len = (frames - 1) * hop + points
        win_flag = bd.F_WINDOW(kind) if kind is not None else 0
        spec = torch.empty(frames, points, device="cuda", dtype=ct)
        fwd = shift | win_flag | (bd.F_REAL_INPUT if real else 0)
        assert getattr(L, "bdsp_fft_frames_" + s)(x.data_ptr(), spec.data_ptr(), points, hop, frames, fwd) == 0, L.bdsp_last_error()
        del x
        inv = shift | win_flag | (bd.F_REAL_OUTPUT if real else 0)
        out = torch.empty(out_len, device="cuda", dtype=rt if real else ct)
        rows_out = torch.empty_like(spec)
        window = torch.from_numpy(acc.window(3 if kind is None else kind, points, np.float32 if rsz == 4 else np.float64)).cuda()
        ifft_frames, fft_rows = getattr(L, "bdsp_ifft_frames_" + s), getattr(L, "bdsp_fft_rows_" + s)
        res = {}

        def ours():
            assert ifft_frames(spec.data_ptr(), out.data_ptr(), points, hop, frames, inv) == 0, L.bdsp_last_error()

        def rows():
            assert fft_rows(spec.data_ptr(), rows_out.data_ptr(), points, frames, bd.F_INVERSE | bd.F_SHIFT) == 0, L.bdsp_last_error()

        def torch_istft():
            X = torch.roll(spec, -(points // 2), dims=1) if shift else spec
            res["torch"] = torch.istft(X.T, n_fft=points, hop_length=hop, win_length=points, window=window, center=False,
                                       normalized=False, onesided=False, return_complex=True)

        e, o = 2 * rsz, rsz if real else 2 * rsz
        two_stage = 3 * e * points * frames + o * out_len
        fused = e * points * frames + o * out_len
        for label, fn, nbytes in (("ifft_frames", ours, two_stage), ("torch.istft", torch_istft, None), ("rows only", rows, None)):
            med, best = timed(fn, args.iters)
            if nbytes:
                gbs = nbytes / med / 1e6
                print("%-46s %7d %9s %9.3f %9.3f %8.0f %7.1f%% %8.2f" % (name, frames, label, med, best, gbs, 100 * gbs * 1e9 / HBM,
                                                                         med / (fused / HBM * 1e3)))
            else:
                print("%-46s %7d %9s %9.3f %9.3f" % (name, frames, label, med, best))
        torch_istft()
        torch.cuda.synchronize()
        ref = res["torch"].real if real else res["torch"]
        rel = (torch.linalg.vector_norm((out - ref).to(torch.complex128)) / torch.linalg.vector_norm(ref.to(torch.complex128))).item()
        print("  (two-stage %d B, fused ideal %d B; relative L2 difference to torch.istft %.2e)" % (two_stage, fused, rel))
        del spec, out, rows_out, res
        torch.cuda.empty_cache()
    L.bdsp_set_stream(None)


if __name__ == "__main__":
    main()
