"""Path fingerprint of a library build: SHA-256 of the output bytes and the kernel-launch count of every FFT, windowed-FFT
and convolution case of tests/test_gpu_accuracy.py (same seeded inputs).  Two builds that take the same paths agree on
every case; select the library with BASIC_DSP_B200_LIB.

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
