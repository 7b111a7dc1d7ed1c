"""Table fingerprint of a library build: result code, SHA-256 of the output bytes and kernel-launch count of every entry point
that builds a host table (tap tables, frequency-response tables, callback windows) or maps window / shift flags to a
transform, f32 and f64, on seeded inputs.  Cacheable cases run twice, and a last pass of more than 64 distinct parameter
sets runs the staging fallback behind a full cache.  Two builds that compute the same tables agree on every case; select
the library with BASIC_DSP_B200_LIB.

    python scratch/table_fingerprint.py OUT.json
    python scratch/table_fingerprint.py --compare A.json B.json"""
import ctypes
import hashlib
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fingerprints():
    sys.path[:0] = [ROOT]
    import numpy as np
    import basic_dsp_b200 as bd
    from basic_dsp_b200 import DspVec

    L = bd.lib()
    res = {}

    def sha(a):
        return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    def vec_case(key, x, name, *args, domain=bd.TIME, dtype=np.float32):
        v = DspVec(x, domain=domain, dtype=dtype)
        before = bd.kernel_launch_count()
        rc = v.result_code_of(name, *args)
        launches = bd.kernel_launch_count() - before
        res[key] = [rc, sha(v.to_numpy()), launches]

    def dptr(v):
        return v._fn("bdsp_device_ptr")(v._h)

    for dtype in (np.float32, np.float64):
        s = "32" if dtype == np.float32 else "64"
        ct = np.complex64 if dtype == np.float32 else np.complex128
        rng = np.random.default_rng(2024 + len(s))

        def real(n):
            return rng.uniform(-1, 1, n).astype(dtype)

        def cplx(n):
            return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(ct)

        RFN, WFN = getattr(L, "RealFn" + s), getattr(L, "WindowFn" + s)
        imp = RFN(lambda _d, t: math.exp(-0.1 * t * t) * math.cos(0.7 * t))
        resp = RFN(lambda _d, t: 1.0 / (1.0 + t * t))
        skew = RFN(lambda _d, t: 1.0 / (1.0 + t * t) + 0.25 * t)
        win = WFN(lambda _d, i, p: 0.6 + 0.4 * math.sin(math.pi * (i + 0.5) / p))
        keep = [imp, resp, skew, win]
        if s == "32":
            # {float, float} returned in the low 64 bits of xmm0 (see basic_dsp_b200._declare)
            def _c(_d, t):
                return float(np.array([math.cos(0.3 * t) / (1 + 0.05 * t * t), 0.5 * math.sin(0.3 * t)], dtype=np.float32).view(np.float64)[0])
            cfn = L.ComplexFn32(_c)
            keep.append(cfn)
        p = s + " "

        # convolve: built-in on the SIMD branch (ratio 1, len <= 202, > 2000 scalars) and the convolve_function_priv branch
        x_r, x_c, x_s = real(4096), cplx(3000), cplx(20)
        for rep in (1, 2):
            for kind, roll in ((bd.SINC, 0.0), (bd.RAISED_COSINE, 0.35)):
                vec_case(p + "convolve simd k%d r%d" % (kind, rep), x_r, "convolve", kind, roll, 1.0, 31, dtype=dtype)
                vec_case(p + "convolve priv k%d r%d" % (kind, rep), x_c, "convolve", kind, roll, 0.3, 31, dtype=dtype)
                vec_case(p + "convolve priv taps>points k%d r%d" % (kind, rep), x_s, "convolve", kind, roll, 0.3, 31, dtype=dtype)
        vec_case(p + "convolve_real priv", x_c, "convolve_real", imp, None, 1, 0.3, 31, dtype=dtype)
        vec_case(p + "convolve_real simd", x_r, "convolve_real", imp, None, 1, 1.0, 31, dtype=dtype)
        vec_case(p + "convolve_real taps>points", x_s, "convolve_real", imp, None, 1, 0.3, 31, dtype=dtype)
        if s == "32":
            vec_case(p + "convolve_complex", x_c, "convolve_complex", cfn, None, 0, 0.3, 31, dtype=dtype)
            vec_case(p + "convolve_complex taps>points", x_s, "convolve_complex", cfn, None, 0, 0.3, 31, dtype=dtype)

        # multiply_frequency_response: built-in, real callback, complex callback; even and odd lengths
        for n in (4096, 4095):
            X = cplx(n)
            for kind, roll in ((bd.SINC, 0.0), (bd.RAISED_COSINE, 0.35)):
                vec_case(p + "mul_freq_resp k%d n%d" % (kind, n), X, "multiply_frequency_response", kind, roll, 0.7, domain=bd.FREQ, dtype=dtype)
            vec_case(p + "mul_freq_resp real cb n%d" % n, X, "multiply_frequency_response_real", resp, None, 1, 0.7, domain=bd.FREQ, dtype=dtype)
            if s == "32":
                vec_case(p + "mul_freq_resp complex cb n%d" % n, X, "multiply_frequency_response_complex", cfn, None, 0, 0.7,
                         domain=bd.FREQ, dtype=dtype)

        # callback windows, symmetric and not, even and odd lengths
        for n in (1000, 1001):
            x = cplx(n)
            for sym in (1, 0):
                for name in ("apply_custom_window", "unapply_custom_window", "windowed_custom_fft"):
                    vec_case(p + "%s n%d sym%d" % (name, n, sym), x, name, win, None, sym, dtype=dtype)
                vec_case(p + "windowed_custom_ifft n%d sym%d" % (n, sym), x, "windowed_custom_ifft", win, None, sym, domain=bd.FREQ, dtype=dtype)
        r = real(1001)
        H = cplx(501)
        H[250] = H[250].real   # a half spectrum whose shifted first bin is real
        for sym in (1, 0):
            vec_case(p + "windowed_custom_sfft sym%d" % sym, r, "windowed_custom_sfft", win, None, sym, dtype=dtype)
            vec_case(p + "windowed_custom_sifft sym%d" % sym, H, "windowed_custom_sifft", win, None, sym, domain=bd.FREQ, dtype=dtype)

        # built-in windows: kinds 0..3 and out of range
        for kind in (0, 1, 2, 3, 7, -1):
            x = cplx(1024)
            vec_case(p + "windowed_fft k%d" % kind, x, "windowed_fft", kind, dtype=dtype)
            vec_case(p + "windowed_ifft k%d" % kind, x, "windowed_ifft", kind, domain=bd.FREQ, dtype=dtype)
            vec_case(p + "windowed_sfft k%d" % kind, real(1001), "windowed_sfft", kind, dtype=dtype)
            vec_case(p + "windowed_sifft k%d" % kind, H, "windowed_sifft", kind, domain=bd.FREQ, dtype=dtype)
            vec_case(p + "apply_window k%d" % kind, x, "apply_window", kind, dtype=dtype)

        # fft rows: F_WINDOW(0..3, 7) and F_SHIFT, forward and inverse
        rows_fn = getattr(L, "bdsp_fft_rows_c" + s)
        n, rows = 4096, 3
        xr = DspVec(cplx(n * rows), dtype=dtype)
        for flags in [0, bd.F_SHIFT, bd.F_REAL_INPUT | bd.F_SHIFT, bd.F_MAGNITUDE | bd.F_SHIFT] + \
                     [bd.F_WINDOW(k) | sh for k in (0, 1, 2, 3, 7) for sh in (0, bd.F_SHIFT)]:
            for inv in (0, bd.F_INVERSE):
                out = DspVec.zeros(2 * n * rows, is_complex=True, dtype=dtype)
                before = bd.kernel_launch_count()
                rc = rows_fn(dptr(xr), dptr(out), n, rows, flags | inv)
                launches = bd.kernel_launch_count() - before
                res[p + "fft_rows flags%#x" % (flags | inv)] = [rc, sha(out.to_numpy()), launches]

        # interpolatef: polyphase and per-output paths, custom callbacks, rows API
        x = real(3000)
        for rep in (1, 2):
            for kind, roll in ((bd.SINC, 0.0), (bd.RAISED_COSINE, 0.35)):
                vec_case(p + "interpolatef poly k%d r%d" % (kind, rep), x, "interpolatef", kind, roll, 4.0, 0.25, 12, dtype=dtype)
                vec_case(p + "interpolatef frac k%d r%d" % (kind, rep), x, "interpolatef", kind, roll, 2.5, 0.25, 12, dtype=dtype)
        vec_case(p + "interpolatef poly complex", cplx(3000), "interpolatef", bd.SINC, 0.0, 3.0, 0.0, 20, dtype=dtype)
        vec_case(p + "interpolatef_custom integer", x, "interpolatef_custom", imp, None, 1, 4.0, 0.25, 12, dtype=dtype)
        vec_case(p + "interpolatef_custom non-integer", x, "interpolatef_custom", imp, None, 1, 2.5, 0.25, 12, dtype=dtype)
        irows = getattr(L, "bdsp_interpolatef_rows" + s)
        for rep in (1, 2):
            for cx, factor in ((0, 4.0), (1, 4.0), (0, 2.5), (1, 2.5)):
                pts, rows = 1500, 3
                xin = DspVec(cplx(pts * rows) if cx else real(pts * rows), dtype=dtype)
                out = DspVec.zeros(2 * int(pts * factor + 2) * rows, dtype=dtype)
                npts = ctypes.c_size_t(0)
                before = bd.kernel_launch_count()
                rc = irows(dptr(xin), dptr(out), pts, rows, cx, bd.RAISED_COSINE, 0.35, factor, 0.25, 12, ctypes.byref(npts))
                launches = bd.kernel_launch_count() - before
                y = out.to_numpy()[: (2 if cx else 1) * npts.value * rows]
                res[p + "interpolatef_rows cx%d f%g r%d" % (cx, factor, rep)] = [rc, sha(y), launches, npts.value]

        # interpolatei / interpolate / interpft
        for kind, roll in ((bd.SINC, 0.0), (bd.RAISED_COSINE, 0.35)):
            vec_case(p + "interpolatei k%d" % kind, real(1000), "interpolatei", kind, roll, 3, dtype=dtype)
            vec_case(p + "interpolatei complex k%d" % kind, cplx(1000), "interpolatei", kind, roll, 4, dtype=dtype)
            for dest in (2500, 600):
                vec_case(p + "interpolate k%d d%d" % (kind, dest), real(1000), "interpolate", kind, roll, dest, 0.3, dtype=dtype)
        vec_case(p + "interpolatei_custom sym real", real(1000), "interpolatei_custom", resp, None, 1, 3, dtype=dtype)
        vec_case(p + "interpolatei_custom sym odd", real(999), "interpolatei_custom", resp, None, 1, 3, dtype=dtype)
        vec_case(p + "interpolatei_custom asym complex", cplx(1000), "interpolatei_custom", skew, None, 0, 3, dtype=dtype)
        vec_case(p + "interpolatei_custom asym real", real(1000), "interpolatei_custom", skew, None, 0, 3, dtype=dtype)
        for dest in (2500, 2501, 600):
            vec_case(p + "interpolate_custom sym d%d" % dest, real(1000), "interpolate_custom", resp, None, 1, dest, 0.3, dtype=dtype)
            vec_case(p + "interpolate_custom asym complex d%d" % dest, cplx(1000), "interpolate_custom", skew, None, 0, dest, 0.3, dtype=dtype)
            vec_case(p + "interpft d%d" % dest, cplx(1000), "interpft", dest, dtype=dtype)

        del keep

    # more than 64 distinct built-in parameter sets: the cache fills, the rest are staged
    for dtype in (np.float32, np.float64):
        x = np.random.default_rng(9).uniform(-1, 1, 4096).astype(dtype)
        for i in range(40):
            vec_case("fill %s convolve %d" % (np.dtype(dtype).name, i), x, "convolve", bd.RAISED_COSINE, 0.1 + 0.01 * i, 0.3, 15, dtype=dtype)
            vec_case("fill %s interpolatef %d" % (np.dtype(dtype).name, i), x, "interpolatef", bd.RAISED_COSINE, 0.1 + 0.01 * i, 2.0, 0.0, 8,
                     dtype=dtype)
    return res


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
