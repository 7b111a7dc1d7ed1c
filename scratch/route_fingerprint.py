"""Path fingerprint of a library build: SHA-256 of the output bytes and the kernel-launch count of every FFT, windowed-FFT
and convolution case of tests/test_gpu_accuracy.py (same seeded inputs), plus seeded c32 / c64 cases of the elementwise
entry points (binary ops with a shorter operand, complex mul / div, complex math, set_real_imag / set_mag_phase), real
signals on the full-length convolution path and chirp-z lengths with the separate spectrum multiply.  Two builds that
take the same paths agree on every case; select the library with BASIC_DSP_B200_LIB.

    python scratch/route_fingerprint.py OUT.json
    python scratch/route_fingerprint.py --compare A.json B.json"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fingerprints():
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    import numpy as np
    import basic_dsp_b200 as bd
    import test_gpu_accuracy as t

    res = {}

    def record(key, run):
        before = bd.kernel_launch_count()
        y = np.ascontiguousarray(run())
        res[key] = [hashlib.sha256(y.tobytes()).hexdigest(), bd.kernel_launch_count() - before]

    for c in t.FFT_CASES:
        dtype, n, rows, flags, variant, *_ = c.values
        rng = np.random.default_rng(n * 131 + rows * 7 + flags)
        x = t.rand_c(rng, (rows, n), dtype)
        if flags & t.REAL:
            x = np.ascontiguousarray(x.real)
        record("fft " + c.id, lambda: t.gpu_fft(x, flags, dtype, 1 if variant == "offset" else 0, variant == "inplace"))
    for dtype, n, rows, branch, _ in t.WINDOWED_CASES:
        x = t.rand_c(np.random.default_rng(n + rows), (rows, n), dtype)
        record("windowed %s-%d-%d" % (np.dtype(dtype).name, n, rows), lambda: t.gpu_fft(x, t.SH, dtype, window=bd.BLACKMAN_HARRIS))
    for dtype, n, rows, taps, api, *_ in t.CONV_CASES:
        rng = np.random.default_rng(n * 17 + taps * 3 + rows)
        x = t.rand_c(rng, (rows, n), dtype)
        h = (t.rand_c(rng, taps, dtype) / 10).astype(x.dtype)
        if api == "vec-real":
            x, h = np.ascontiguousarray(x.real), np.ascontiguousarray(h.real)
        key = "conv %s-%d-x%d-L%d-%s" % (np.dtype(dtype).name, n, rows, taps, api)
        if api.startswith("rows"):
            record(key, lambda: t.gpu_conv_rows(x, h, dtype, 1 if api == "rows-offset" else 0))
        else:
            record(key, lambda: t.gpu_conv_vec(x, h))
    elementwise_cases(record, np, bd, t)
    return res


def elementwise_cases(record, np, bd, t):
    DspVec = bd.DspVec

    def run(key, fn):
        try:
            record(key, fn)
        except bd.DspError as e:   # an error code is part of the fingerprint too
            res_err = "error %s" % (e.args,)
            record(key, lambda: np.frombuffer(res_err.encode(), dtype=np.uint8))

    for dtype in (t.F32, t.F64):
        name = np.dtype(dtype).name
        for cplx in (False, True):
            kind = "complex" if cplx else "real"
            rng = np.random.default_rng(11 + cplx + 2 * (dtype == t.F64))
            n, m = 100003 * 7, 7
            x = t.rand_c(rng, n, dtype) if cplx else rng.uniform(-10, 10, n).astype(dtype)
            w = t.rand_c(rng, m, dtype) if cplx else rng.uniform(1, 10, m).astype(dtype)
            for op in ("add", "sub", "mul", "div"):
                run("smaller %s-%s-%s" % (name, kind, op), lambda: getattr(DspVec(x), op + "_smaller")(DspVec(w)).to_numpy())
        rng = np.random.default_rng(21 + (dtype == t.F64))
        n = 100003
        a, b = t.rand_c(rng, n, dtype), t.rand_c(rng, n, dtype)
        run("binary %s-complex-mul" % name, lambda: DspVec(a).mul(DspVec(b)).to_numpy())
        run("binary %s-complex-div" % name, lambda: DspVec(a).div(DspVec(b)).to_numpy())
        for op in ("sin", "cos", "tan", "asin", "acos", "atan", "sinh", "cosh", "tanh", "asinh", "acosh", "atanh", "sqrt",
                   "square", "ln", "exp", "abs", "ln_approx", "exp_approx", "sin_approx", "cos_approx"):
            run("math %s-complex-%s" % (name, op), lambda: DspVec(a).math(op).to_numpy())
        for op, arg in (("root", 3.0), ("powf", 2.5), ("log", 10.0), ("expf", 3.0), ("wrap", 1.0), ("log_approx", 10.0),
                        ("expf_approx", 3.0), ("powf_approx", 2.5)):
            run("math %s-complex-%s" % (name, op), lambda: DspVec(a).math(op, arg).to_numpy())
        s = np.array([complex(4, 0), complex(-4, 0.0), complex(-4, -0.0), complex(0, 2), complex(0, -2)], dtype=a.dtype)
        run("math %s-complex-sqrt-exact" % name, lambda: DspVec(s).math("sqrt").to_numpy())
        re, im = a.real.copy(), a.imag.copy()
        run("compose %s-set_real_imag" % name, lambda: DspVec(np.zeros(2, dtype=a.dtype)).set_real_imag(DspVec(re), DspVec(im)).to_numpy())
        mag, ph = np.abs(a).astype(dtype), np.angle(a).astype(dtype)
        run("compose %s-set_mag_phase" % name, lambda: DspVec(np.zeros(2, dtype=a.dtype)).set_mag_phase(DspVec(mag), DspVec(ph)).to_numpy())
    # real signals long enough for the full-length convolution (taps beyond the overlap-save blocks)
    for dtype, n, taps in ((t.F32, 16384, 9000), (t.F32, 3 << 14, 9000), (t.F32, 20000, 9000), (t.F64, 40000, 5000), (t.F64, 1 << 15, 4500)):
        rng = np.random.default_rng(n + taps)
        x = rng.uniform(-10, 10, n).astype(dtype)
        h = (rng.uniform(-10, 10, taps) / 10).astype(dtype)
        run("conv-full-real %s-%d-L%d" % (np.dtype(dtype).name, n, taps), lambda: DspVec(x).convolve_signal(DspVec(h)).to_numpy())
    # chirp-z lengths whose padded length M = next_pow2(2n - 1) is 64 .. 16384: c32 keeps a separate spectrum multiply
    for n in (37, 251, 1009, 4099, 8191):
        for rows in (1, 5):
            for flags in (0, t.INV):
                rng = np.random.default_rng(n * 3 + rows + flags)
                x = t.rand_c(rng, (rows, n), t.F32)
                run("chirp c32-%d-x%d-f%d" % (n, rows, flags), lambda: t.gpu_fft(x, flags, t.F32))


def main():
    if sys.argv[1] == "--compare":
        a, b = (json.load(open(p)) for p in sys.argv[2:4])
        diff = sorted(k for k in set(a) | set(b) if a.get(k) != b.get(k))
        for k in diff:
            print("DIFFERS", k, a.get(k), b.get(k))
        print("%d cases, %d differ" % (len(a), len(diff)))
        return 1 if diff or set(a) != set(b) else 0
    res = fingerprints()
    with open(sys.argv[1], "w") as fh:
        json.dump(res, fh, indent=1, sort_keys=True)
    print("%d cases -> %s" % (len(res), sys.argv[1]))
    return 0


if __name__ == "__main__":
    sys.exit(main())
