"""bdsp_csd_c32 / _c64 and bdsp_coherence_c32 / _c64 against what a caller does without them, on the library's stream:
  (a) bdsp_fft_frames_* of x and of y into full frame spectra, then the conjugate product and the mean over frames in torch
      (for coherence also the means of |X|^2 and |Y|^2);
  (b) torch.stft(center=False) of x and of y with the library's window table, then the same torch code;
  (c) bdsp_welch_* of x and of y: two fused power sums, a floor for a fused cross sum rather than a competitor.
Median and best of CUDA-event timings after warm-up, every input above the 126 MB L2.  Every output is compared with a
float64 closed form computed on the GPU with torch (relative L2 error).

    python scratch/bench_csd.py [--iters 20]                     (results: profiles/r3_csd.txt)
    python scratch/bench_csd.py --sweep LIB...                   the library calls alone, once per build in LIB (a build of
                                                                 the library with another CSD_CHUNK_POINTS, named *_<log2>.so)

Workloads (those of scratch/bench_welch.py), two signals each: x uniform in [-1, 1), y = 0.6 x + 0.3 x delayed by 3 samples
+ 0.5 independent noise, so that the coherence lies inside (0, 1):
  1. real f32 signals of 2^28 samples, 1024-point Hamming frames, hop 256, one-sided density: 1048573 frames;
  2. c32 signals of 2^26 points, 4096-point Blackman-Harris frames, hop 2048, fftshift order;
  3. c32 signals of 2^26 points, 256-point rectangular frames, hop 128, power spectrum (csd; coherence takes no scaling);
  4. real f64 signals of 2^27 samples, 1024-point Hamming frames, hop 256, one-sided."""
import argparse
import os
import re
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


def library_window(kind, points, dtype):
    if kind is None:
        return np.ones(points, dtype=dtype)
    return bd.DspVec(np.ones(points, dtype=dtype), is_complex=False, dtype=dtype).apply_window(kind).to_numpy()


def finish(sums, w, frames, flags, points, coherence):
    """frame sums (two-sided, fftfreq order): csd -> sum conj(X) Y; coherence -> (sum conj(X) Y, sum |X|^2, sum |Y|^2);
    sliced to bins 0 .. points/2 where one-sided -> the library's output"""
    nout = points // 2 + 1 if flags & bd.F_ONESIDED else points
    if coherence:
        sxy, sxx, syy = (s[:nout].to(torch.complex128 if s.is_complex() else torch.float64) for s in sums)
        out = sxy.abs() ** 2 / (sxx * syy)
    else:
        w = w.double()
        den = w.sum() ** 2 if flags & bd.F_POWER_SPECTRUM else FS * (w * w).sum()
        out = sums[0][:nout].to(torch.complex128) / (frames * den)
        if flags & bd.F_ONESIDED:
            out[1:points // 2 + points % 2] *= 2
    if flags & bd.F_SHIFT:
        out = torch.roll(out, points // 2)
    return out


def torch_sums(X, Y, nout, coherence):
    """frames x bins spectra -> the frame sums of finish(), over the first nout bins"""
    X, Y = X[:, :nout], Y[:, :nout]
    sxy = (X.conj() * Y).sum(0)
    if not coherence:
        return (sxy,)
    return sxy, (X.real.square() + X.imag.square()).sum(0), (Y.real.square() + Y.imag.square()).sum(0)


def reference(x, y, points, hop, frames, w, flags, coherence):
    """float64 closed form on the GPU, in chunks of frames"""
    cdt = torch.complex128 if x.is_complex() else torch.float64
    xd, yd, wd = x.to(cdt), y.to(cdt), w.double()
    sums = None
    step = max(1, (1 << 24) // points)
    for f0 in range(0, frames, step):
        cnt = min(step, frames - f0)
        X = torch.fft.fft(xd[f0 * hop:].unfold(0, points, hop)[:cnt] * wd)
        Y = torch.fft.fft(yd[f0 * hop:].unfold(0, points, hop)[:cnt] * wd)
        part = torch_sums(X, Y, points, coherence)
        sums = part if sums is None else tuple(a + b for a, b in zip(sums, part))
    return finish(sums, w, frames, flags, points, coherence)


def rel_l2(a, ref):
    a = a.to(ref.dtype)
    return float(torch.linalg.vector_norm(a - ref) / torch.linalg.vector_norm(ref))


WORKLOADS = [
    ("1 real 2^28, 1024 Hamming, hop 256, one-sided", torch.float32, True, 1 << 28, 1024, 256, "HAMMING", "R|ONE"),
    ("2 c32 2^26, 4096 Blackman-Harris, hop 2048, shift", torch.float32, False, 1 << 26, 4096, 2048, "BLACKMAN_HARRIS", "SH"),
    ("3 c32 2^26, 256 rectangular, hop 128, power spectrum", torch.float32, False, 1 << 26, 256, 128, None, "PSD"),
    ("4 real f64 2^27, 1024 Hamming, hop 256, one-sided", torch.float64, True, 1 << 27, 1024, 256, "HAMMING", "R|ONE"),
]


def run(args):
    L = bd.lib()
    bd.require_device()
    stream = torch.cuda.current_stream()
    L.bdsp_set_stream(stream.cuda_stream)   # torch's kernels and the library's on one stream
    g = torch.Generator(device="cuda").manual_seed(0)
    names = {"R": bd.F_REAL_INPUT, "ONE": bd.F_ONESIDED, "PSD": bd.F_POWER_SPECTRUM, "SH": bd.F_SHIFT}
    print("%-52s %-9s %8s %-16s %9s %9s %8s %10s" % ("workload", "output", "frames", "path", "median ms", "best ms", "x lib", "rel L2"))
    for name, rdt, real, length, points, hop, kind_name, flag_names in WORKLOADS:
        c32 = rdt == torch.float32
        npdt = np.float32 if c32 else np.float64
        kind = getattr(bd, kind_name) if kind_name else None
        flags = 0
        for f in flag_names.split("|"):
            flags |= names[f]
        shape = (length,) if real else (length, 2)
        x = torch.rand(shape, generator=g, device="cuda", dtype=rdt) * 2 - 1
        e = torch.rand(shape, generator=g, device="cuda", dtype=rdt) * 2 - 1
        y = 0.6 * x + 0.3 * torch.roll(x, 3, 0) + 0.5 * e
        del e
        if not real:
            x, y = torch.view_as_complex(x), torch.view_as_complex(y)
        frames = 1 + (length - points) // hop
        wflag = bd.F_WINDOW(kind) if kind is not None else 0
        w = torch.from_numpy(library_window(kind, points, npdt)).cuda()
        nout = points // 2 + 1 if flags & bd.F_ONESIDED else points
        s = "32" if c32 else "64"
        for coherence in (False, True):
            cflags = flags & ~bd.F_POWER_SPECTRUM if coherence else flags
            out = torch.empty(nout, device="cuda", dtype=rdt if coherence else (torch.complex64 if c32 else torch.complex128))
            if coherence:
                f = getattr(L, "bdsp_coherence_c" + s)

                def lib_call():
                    assert f(x.data_ptr(), y.data_ptr(), out.data_ptr(), points, hop, frames, cflags | wflag) == 0, L.bdsp_last_error()
            else:
                f = getattr(L, "bdsp_csd_c" + s)

                def lib_call():
                    assert f(x.data_ptr(), y.data_ptr(), out.data_ptr(), points, hop, frames, cflags | wflag, FS) == 0, L.bdsp_last_error()

            ref = reference(x, y, points, hop, frames, w, cflags, coherence)
            paths = [("library", lib_call, lambda: out)]
            if not args.library_only:
                res = {}
                X = torch.empty(frames, points, device="cuda", dtype=torch.complex64 if c32 else torch.complex128)
                Y = torch.empty_like(X)
                ff = getattr(L, "bdsp_fft_frames_c" + s)

                def frames_torch():
                    fl = (cflags & bd.F_REAL_INPUT) | wflag   # fftshift and fold in finish()
                    assert ff(x.data_ptr(), X.data_ptr(), points, hop, frames, fl) == 0, L.bdsp_last_error()
                    assert ff(y.data_ptr(), Y.data_ptr(), points, hop, frames, fl) == 0, L.bdsp_last_error()
                    res["a"] = finish(torch_sums(X, Y, nout, coherence), w, frames, cflags, points, coherence)

                def stft():
                    kw = dict(n_fft=points, hop_length=hop, win_length=points, window=w, center=False, onesided=bool(cflags & bd.F_ONESIDED),
                              return_complex=True)
                    SX, SY = torch.stft(x, **kw).T, torch.stft(y, **kw).T   # frames x bins
                    res["b"] = finish(torch_sums(SX, SY, nout, coherence), w, frames, cflags, points, coherence)

                pw = torch.empty(nout, device="cuda", dtype=rdt)
                welch = getattr(L, "bdsp_welch_c" + s)

                def two_welch():
                    for sig in (x, y):
                        assert welch(sig.data_ptr(), pw.data_ptr(), points, hop, frames, flags | wflag, FS) == 0, L.bdsp_last_error()

                paths += [("(a) frames+torch", frames_torch, lambda: res["a"]), ("(b) stft+torch", stft, lambda: res["b"]),
                          ("(c) 2x welch", two_welch, None)]
            lib_med = None
            for label, call, result in paths:
                med, best = timed(call, args.iters)
                torch.cuda.synchronize()
                lib_med = lib_med or med
                err = "%10.2e" % rel_l2(result(), ref) if result else "%10s" % "-"
                print("%-52s %-9s %8d %-16s %9.3f %9.3f %8.2f %s" % (name, "coherence" if coherence else "csd", frames, label, med, best,
                                                                   med / lib_med, err), flush=True)
            if not args.library_only:
                del X, Y
            torch.cuda.empty_cache()
        del x, y
        torch.cuda.empty_cache()
    L.bdsp_set_stream(None)


def sweep(args):
    """the library calls alone, once per build: a fresh process each, the build selected with BASIC_DSP_B200_LIB"""
    rows = {}
    for lib in args.sweep:
        k = int(re.search(r"_(\d+)\.so$", lib).group(1))
        env = dict(os.environ, BASIC_DSP_B200_LIB=os.path.abspath(lib))
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--library-only", "--iters", str(args.iters)], env=env,
                             capture_output=True, text=True, check=True).stdout
        print("CSD_CHUNK_POINTS = 2^%d (%s)\n%s" % (k, os.path.basename(lib), out), flush=True)
        for line in out.splitlines()[2:]:   # past the card and the header
            key = line[:62].rstrip()
            rows.setdefault(key, {})[k] = float(line.split()[-4])   # median ms
    ks = sorted({k for r in rows.values() for k in r})
    print("median ms by CSD_CHUNK_POINTS")
    print("%-62s %s" % ("workload / output", " ".join("%8s" % ("2^%d" % k) for k in ks)))
    for key, r in rows.items():
        print("%-62s %s" % (key, " ".join("%8.3f" % r[k] for k in ks)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--library-only", action="store_true")
    ap.add_argument("--sweep", nargs="*")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    print("card: %s (torch: %s)  library: %s" % (smi[0] if smi else "nvidia-smi unavailable", torch.cuda.get_device_name(), bd.LIB_PATH),
          flush=True)
    if args.sweep:
        sweep(args)
    else:
        run(args)


if __name__ == "__main__":
    main()
