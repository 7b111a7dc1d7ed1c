"""bdsp_fft_frames_c32 (short-time transforms of overlapping frames of one device signal) against what a caller does
without it: materialise the frames on the device (torch unfold(...).contiguous() on the library's stream), then
bdsp_fft_rows_c32 with the same flags.  Median and best of CUDA-event timings; algorithmic bytes = the signal read once
(hop * frames points) plus the output; the HBM peak is a device-to-device copy measured in the same run.

    python scratch/bench_fft_frames.py [--iters 20]      (results: profiles/r3_fft_frames.txt)

Workloads (inputs above the 126 MB L2):
  1. real f32 signal of 2^28 samples, 1024-point Hamming frames, hop 256, magnitude (spectrogram);
  2. c32 signal of 2^26 points, 4096-point Blackman-Harris frames, hop 2048, fft_shift and magnitude;
  3. c32 signal of 2^26 points, 256-point rectangular frames, hop 128.
frames = 1 + (len - points) / hop leaves 1 and 15 frames past whole groups of 4096 / n frames in 1 and 3: those calls take
the gathering frame pass; each is also run with the frame count rounded down to whole groups (the fused kernel)."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import basic_dsp_b200 as bd  # noqa: E402


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
    L.bdsp_set_stream(stream.cuda_stream)   # torch's copies and the library's kernels on one stream
    peak = hbm_peak(args.iters)
    print("HBM peak (device-to-device copy, best of %d): %.0f GB/s" % (args.iters, peak))
    print("%-58s %7s %9s %9s %9s %8s %7s" % ("workload", "frames", "path", "median ms", "best ms", "GB/s", "of peak"))
    g = torch.Generator(device="cuda").manual_seed(0)
    workloads = [
        ("real 2^28, 1024 Hamming, hop 256, |X|", True, 1 << 28, 1024, 256, bd.F_REAL_INPUT | bd.F_MAGNITUDE | bd.F_WINDOW(bd.HAMMING)),
        ("c32 2^26, 4096 Blackman-Harris, hop 2048, shift |X|", False, 1 << 26, 4096, 2048,
         bd.F_SHIFT | bd.F_MAGNITUDE | bd.F_WINDOW(bd.BLACKMAN_HARRIS)),
        ("c32 2^26, 256 rectangular, hop 128", False, 1 << 26, 256, 128, 0),
    ]
    for name, real, length, points, hop, flags in workloads:
        if real:
            x = torch.rand(length, generator=g, device="cuda", dtype=torch.float32) * 2 - 1
        else:
            x = torch.view_as_complex(torch.rand(length, 2, generator=g, device="cuda", dtype=torch.float32) * 2 - 1)
        full = 1 + (length - points) // hop
        per = 4096 // points if points < 4096 else 1
        counts = [full] if full % per == 0 else [full, full - full % per]
        mag = flags & bd.F_MAGNITUDE
        for frames in counts:
            out_f = torch.empty(frames, points, device="cuda", dtype=torch.float32 if mag else torch.complex64)
            out_r = torch.empty_like(out_f)

            def fused():
                assert L.bdsp_fft_frames_c32(x.data_ptr(), out_f.data_ptr(), points, hop, frames, flags) == 0, L.bdsp_last_error()

            def materialised():
                fr = x.unfold(0, points, hop)[:frames].contiguous()
                assert L.bdsp_fft_rows_c32(fr.data_ptr(), out_r.data_ptr(), points, frames, flags) == 0, L.bdsp_last_error()

            esz_in = 4 if real else 8
            nbytes = hop * frames * esz_in + frames * points * (4 if mag else 8)
            route = "fused" if frames % per == 0 else "gather"
            for label, fn in ((route, fused), ("baseline", materialised)):
                med, best = timed(fn, args.iters)
                gbs = nbytes / med / 1e6
                print("%-58s %7d %9s %9.3f %9.3f %8.0f %6.1f%%" % (name, frames, label, med, best, gbs, 100 * gbs / peak))
            torch.cuda.synchronize()
            same = torch.equal(out_f.view(torch.int32) if mag else torch.view_as_real(out_f).view(torch.int32),
                               out_r.view(torch.int32) if mag else torch.view_as_real(out_r).view(torch.int32))
            print("  (%s: %d B algorithmic; outputs byte-identical: %s)" % (route, nbytes, same))
            del out_f, out_r
        del x
        torch.cuda.empty_cache()
    L.bdsp_set_stream(None)


if __name__ == "__main__":
    main()
