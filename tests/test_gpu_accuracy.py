"""Per-element accuracy of every FFT and convolution dispatch branch against same-precision CPU peers.

Every case names the branch it targets and the condition in the code that selects it.  Each row of a result is checked
with oracle.accuracy.check: relative L2 error and worst element error (relative to the row's RMS), both measured
against a higher-precision reference, within a small factor of what a CPU computation in the kernel's own precision
achieves (and within BASELINE's tolerance).  Each case also runs on 4^k x (k = +-10 for f32, +-100 for f64): scaling by a
power of two commutes with every rounding, so the result must be 4^k times the unscaled result bit for bit (1 ulp for
the sqrt.approx of F_MAGNITUDE); a mismatch means data-dependent behaviour or a race.

Run with -s to see the records (path, n, rows, rel / elmax of GPU and peer, ratios) of profiles/r3_accuracy.txt.
Inputs are uniform in [-10, 10)."""
import numpy as np
import pytest

import basic_dsp_b200 as bd
from basic_dsp_b200 import DspVec
from oracle import accuracy as acc
from oracle.accuracy import F_INVERSE as INV, F_MAGNITUDE as MAG, F_REAL_INPUT as REAL, F_SHIFT as SH

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
ALL_FLAGS = (0, SH, INV, INV | SH, SH | MAG, REAL)


def dptr(v):
    return v._fn("bdsp_device_ptr")(v._h)


def rand_c(rng, shape, dtype):
    return (rng.uniform(-10, 10, shape) + 1j * rng.uniform(-10, 10, shape)).astype(acc.ctype(dtype))


class Buf:
    """Device buffer holding `arr` (complex or real rows) `off` elements after a 256-byte aligned allocation start."""

    def __init__(self, arr, off=0, dtype=F32):
        arr = np.ascontiguousarray(arr).ravel()
        self.cplx = np.iscomplexobj(arr)
        self.dtype, self.off, self.count = dtype, off, arr.size
        host = np.zeros(arr.size + off, dtype=arr.dtype)
        host[off:] = arr
        self.v = DspVec(host, is_complex=self.cplx, dtype=dtype)
        self.esize = np.dtype(dtype).itemsize * (2 if self.cplx else 1)

    @classmethod
    def empty(cls, count, cplx, off=0, dtype=F32):
        return cls(np.zeros(count, dtype=acc.ctype(dtype) if cplx else dtype), off, dtype)

    @property
    def ptr(self):
        return dptr(self.v) + self.off * self.esize

    def get(self, shape):
        return self.v.to_numpy()[self.off:].reshape(shape)


def report(rec):
    print(acc.format_record(rec))


def check_rows(got, ref, peer, dtype, path, k_rel=acc.K_REL, k_el=acc.K_EL, tol_n=None):
    """Every row, then the first and the last row of the batch on their own."""
    rec = acc.check(got, ref, peer, dtype, path=path, k_rel=k_rel, k_el=k_el, tol_n=tol_n)
    got, ref, peer = (np.asarray(a).reshape(-1, np.asarray(got).shape[-1]) for a in (got, ref, peer))
    for r in (0, got.shape[0] - 1):
        acc.check(got[r], ref[r], peer[r], dtype, path="%s row %d" % (path, r), k_rel=k_rel, k_el=k_el, tol_n=tol_n)
    report(rec)
    return rec


def assert_scaled_exact(run, x, base, dtype, ulps=0):
    """run(4^k x) == 4^k run(x) bit for bit (or within `ulps` ulp)."""
    for k in ((10, -10) if dtype == F32 else (100, -100)):
        s = dtype(4.0) ** k
        got = run((x * s).astype(x.dtype))
        want = base * s
        assert got.dtype == want.dtype
        if ulps == 0:
            bad = np.flatnonzero(got.view(dtype).ravel() != want.view(dtype).ravel())
            assert bad.size == 0, "4^%d scaling not exact at %d elements (first flat index %d)" % (k, bad.size, bad[0])
        else:
            assert acc_ulp(got, want, dtype) <= ulps, k


def acc_ulp(a, b, dtype):
    from oracle.dsp_oracle import ulp_diff
    return int(ulp_diff(np.asarray(a).view(dtype).ravel(), np.asarray(b).view(dtype).ravel(), dtype).max())


# Per-path factors above the default K_rel = 4, K_el = 8, each with its measured cause (profiles/r3_accuracy.txt).
#   Chirp-z lengths that pocketfft factors directly (1001 = 7 * 11 * 13; 20000 = 2^5 * 5^4): the GPU runs Bluestein
#   (two chirp products and three M-point transforms), the peer a mixed-radix transform.  Measured on B200: c32 n = 1001
#   rel x3.8 - 4.3, elmax up to x6.1; c64 n = 1001 rel x2.9 - 3.1 (the same ratio in both precisions: the algorithm,
#   not a precision defect); c32 n = 30021, where the peer is a chirp-z transform as well, x1.6.
CHIRP_DIRECT_PEER = (8.0, 12.0)
WIDER = {"chirp-z (M = 2048: separate filter multiply)": CHIRP_DIRECT_PEER, "c64 chirp-z": CHIRP_DIRECT_PEER,
         "full length c32 rows, chirp-z N": CHIRP_DIRECT_PEER}


# ---- transforms ------------------------------------------------------------------------------------------------------
def gpu_fft(x, flags, dtype, off=0, inplace=False, window=None):
    """bdsp_fft_rows_* over the rows of x; off: input (and output) pointer offset in elements; inplace: in == out."""
    L = bd.lib()
    rows, n = x.shape
    fn = getattr(L, "bdsp_fft_rows_" + ("c32" if dtype == F32 else "c64"))
    xin = Buf(x, off, dtype)
    out = xin if inplace else Buf.empty(rows * n, not flags & MAG, off, dtype)
    f = flags | (bd.F_WINDOW(window) if window is not None else 0)
    assert fn(xin.ptr, out.ptr, n, rows, f) == 0, bd.lib().bdsp_last_error()
    return out.get((rows, n))


# (dtype, n, rows, flags, variant, branch, selecting condition, route)
#   variant: "" | "offset" (input and output one element past a 16-byte boundary) | "inplace" (in == out)
#   route: what fft_route (csrc/fft_route.h) picks, level by level ("mul-pass > packed"); a dict maps flags to routes where
#   they differ (None: the other flags).  Checked without a GPU by test_fft_route.py.
FFT_CASES = []


def fc(dtype, n, rows, flags, branch, cond, route, variant=""):
    for f in flags:
        FFT_CASES.append(pytest.param(dtype, n, rows, f, variant, branch, cond, route,
                                      id="%s-%d-x%d-f%d%s" % ("c32" if dtype == F32 else "c64", n, rows, f, "-" + variant if variant else "")))


_SP = {64: "fftp SQ=4", 128: "fftp SQ=8", 256: "fftp NATQ=1", 512: "fftp NATQ=2", 1024: "fftp NATQ=4", 2048: "fftp NATQ=8",
       4096: "fftp R0=1", 8192: "fftp R0=2"}
PACKED = {None: "packed", REAL: "real-rows"}
for n, name in _SP.items():
    # rows = 2^16 / n: a multiple of 4096 / n, and n * rows >= 2^16 for the real-input kernel
    fc(F32, n, 65536 // n, ALL_FLAGS, "packed single pass " + name,
       "fft_route: c32 pow2 64 <= n <= 16384, no in_mul, in != out, in & 15 == 0; n < 4096: rows % (4096/n) == 0; "
       "REAL: real-rows, n*rows >= 2^16", PACKED)
    if n < 4096:
        fc(F32, n, 4096 // n + 1, ALL_FLAGS, "generic fall-back of " + name, "fft_route: rows % (4096/n) != 0 -> block kernel", "block")
    fc(F32, n, 4096 // n if n < 4096 else 2, (0, SH, INV, INV | SH), "generic fall-back of " + name, "fft_route: in == out", "block",
       "inplace")
    fc(F32, n, 4096 // n if n < 4096 else 2, ALL_FLAGS, "generic fall-back of " + name,
       "fft_route: in & 15 (real rows: in & 7) -> generic kernels", "block", "offset")
fc(F32, 16384, 4, ALL_FLAGS, "packed 16384 persistent (fftp16k)", "fft_route: n == 16384 && rows >= 2 -> packed-16k",
   {None: "packed-16k", REAL: "real-rows"})
fc(F32, 16384, 1, ALL_FLAGS[:5], "packed 16384 non-persistent fftp R0=4", "fft_route: n == 16384 && rows == 1", "packed")
fc(F32, 16384, 2, (0, SH, INV, INV | SH), "generic fall-back of 16384", "fft_route: in == out", "block", "inplace")
fc(F32, 16384, 2, ALL_FLAGS, "generic fall-back of 16384", "fft_route: in & 15", "block", "offset")
fc(F32, 1 << 16, 1, (0, SH, INV, INV | SH), "2^16 cluster kernel (fftc)", "fft_route: n == 65536, !real, !mag, rows <= 8, in != out",
   "cluster")
fc(F32, 1 << 16, 8, (0, SH, INV, INV | SH), "2^16 cluster kernel (fftc)", "fft_route: rows <= 8", "cluster")
fc(F32, 1 << 16, 9, ALL_FLAGS, "packed two-pass 2^16 (N1 = 256)", "fft_route: rows > 8 -> two-pass", "two-pass")
fc(F32, 1 << 15, 4, ALL_FLAGS, "packed two-pass 2^15 (N1 = 32)", "fft_route: 2^15 <= n <= 2^20 -> two-pass", "two-pass")
fc(F32, 1 << 19, 2, ALL_FLAGS, "packed two-pass 2^19 (N1 = 512)", "fft_route: two-pass n1 = 512", "two-pass")
fc(F32, 1 << 20, 2, ALL_FLAGS, "packed two-pass 2^20 (N1 = 256, 4096-point rows)", "fft_route: two-pass n1 = 256, log2n2 = 12", "two-pass")
fc(F32, 1 << 20, 1, (0,), "generic column pass + packed 1024-point rows 2^20 (misaligned)",
   "fft_route: in & 15 -> no two-pass; out & 7 == 0, work & 15 == 0 -> hybrid", "hybrid", "offset")
fc(F32, 1 << 21, 2, ALL_FLAGS, "packed three-pass 2^21 (nA = 16)", "fft_route: 2^21 <= n <= 2^24 -> three-pass", "three-pass")
fc(F32, 1 << 23, 1, (0, INV | SH), "packed three-pass 2^23 (nA = 32)", "fft_route: three-pass nA = 32", "three-pass")
fc(F32, 1 << 24, 1, (0, INV | SH), "packed three-pass 2^24 (nA = 256)", "fft_route: three-pass nA = 256", "three-pass")
fc(F32, 3 << 12, 24, (0, SH, INV | SH, SH | MAG), "q = 3: radix-3 pass + packed rows + interleave",
   "fft_route: q <= 31, packed rows: P >= 256, n*batch >= 2^18", "q-rows-interleave > packed")
fc(F32, 15 << 10, 2, (0, SH, INV | SH, SH | MAG), "q = 15: radix-q pass + generic rows", "fft_route: q <= 31, no packed rows", "q-rows")
fc(F32, 31 << 15, 1, (0, SH, INV | SH, SH | MAG), "q = 31: radix-q pass + two-pass rows + interleave", "fft_route: P > fft_block_max_n",
   "q-rows-interleave > two-pass")
fc(F32, 1001, 5, ALL_FLAGS, "chirp-z (M = 2048: separate filter multiply)", "fft_route: q > 31 -> Bluestein, M <= 16384", "bluestein")
fc(F32, 10007 * 3, 2, ALL_FLAGS, "chirp-z (M = 2^16: filter fused into in_mul)", "fft_route: Bluestein, M > 16384", "bluestein")
fc(F64, 512, 8, ALL_FLAGS, "c64 fft_block_kernel", "fft_route: n <= 8192, not 1024/2048/4096 -> block", "block")
fc(F64, 8192, 3, ALL_FLAGS, "c64 fft_block_kernel", "fft_route: n <= 8192", "block")
for n in (1024, 2048, 4096):
    fc(F64, n, 4, ALL_FLAGS, "c64 f64_row_kernel", "fft_route: f64, n in {1024, 2048, 4096} -> c64-rows", "c64-rows")
fc(F64, 1024, 4, (0, INV | SH), "c64 f64_row_kernel (misaligned)", "c64-rows take any alignment", "c64-rows", "offset")
fc(F64, 1 << 15, 2, ALL_FLAGS, "c64 two-pass f64_tile_kernel", "fft_pow2 tiles: n > 8192, ceil(log2 n / 9) == 2", "tiles")
fc(F64, 1 << 18, 1, (0, INV | SH, SH | MAG), "c64 two-pass f64_tile_kernel", "log2 n = 18", "tiles")
fc(F64, 1 << 20, 1, (0, INV | SH, SH | MAG, REAL), "c64 three-pass f64_tile_kernel", "fft_pow2 tiles: ceil(log2 n / 9) == 3", "tiles")
fc(F64, 3 << 16, 1, (0, SH, INV | SH, REAL), "c64 3*2^k, folded radix-3 first pass", "fft_route: f64, P > 8192, !mag -> q-three-pass",
   "q-three-pass")
fc(F64, 15 << 8, 3, (0, SH, INV | SH, SH | MAG), "c64 q*2^k, radix-q pass + block rows", "fft_route: q <= 31, P <= 8192 -> q-rows", "q-rows")
fc(F64, 31 << 10, 2, (0, INV | SH, SH | MAG), "c64 q*2^k, radix-q pass + f64_row rows", "fft_route: q <= 31, P = 1024; rows: c64-rows",
   "q-rows")
fc(F64, 1001, 3, ALL_FLAGS, "c64 chirp-z", "fft_route: q > 31 -> Bluestein", "bluestein")
fc(F64, 10007 * 3, 1, (0, SH, INV | SH), "c64 chirp-z (M = 2^16, tiles)", "Bluestein, M > 8192", "bluestein")


@pytest.mark.parametrize("dtype,n,rows,flags,variant,branch,cond,route", FFT_CASES)
def test_fft_rows_accuracy(dtype, n, rows, flags, variant, branch, cond, route):
    rng = np.random.default_rng(n * 131 + rows * 7 + flags)
    x = rand_c(rng, (rows, n), dtype)
    if flags & REAL:
        x = np.ascontiguousarray(x.real)
    off = 1 if variant == "offset" else 0
    inplace = variant == "inplace"
    got = gpu_fft(x, flags, dtype, off, inplace)
    ref, peer = acc.fft_pair(x, flags, dtype)
    k_rel, k_el = WIDER.get(branch, (acc.K_REL, acc.K_EL))
    check_rows(got, ref, peer, dtype, "%s f%d%s" % (branch, flags, " " + variant if variant else ""), k_rel, k_el)
    assert_scaled_exact(lambda xs: gpu_fft(xs, flags, dtype, off, inplace), x, got, dtype, ulps=1 if flags & MAG else 0)


# windowed_fft (Blackman-Harris through in_mul) on one length of each multi-kernel family: (dtype, n, rows, branch, route)
WINDOWED_CASES = [
    (F32, 4096, 16, "single pass: in_mul_rows_kernel + packed kernel (n*rows >= 2^16)", "mul-pass > packed"),
    (F32, 1 << 16, 2, "packed two-pass, window on the column pass", "two-pass"),
    (F32, 1 << 21, 1, "packed three-pass, window on pass A", "three-pass"),
    (F32, 3 << 15, 1, "q*2^k: window in the radix-q pass", "q-rows-interleave > two-pass"),
    (F32, 10007, 2, "chirp-z: window in bluestein_pre_kernel", "bluestein"),
    (F64, 1 << 15, 2, "c64 tiles", "tiles"),
    (F64, 3 << 14, 1, "c64 folded radix-3", "q-three-pass"),
    (F64, 10007, 1, "c64 chirp-z", "bluestein"),
]


@pytest.mark.parametrize("dtype,n,rows,branch", [c[:4] for c in WINDOWED_CASES],
                         ids=["%s-%d-%d-%s" % (np.dtype(c[0]).name, c[1], c[2], c[3]) for c in WINDOWED_CASES])
def test_windowed_fft_accuracy(dtype, n, rows, branch):
    rng = np.random.default_rng(n + rows)
    x = rand_c(rng, (rows, n), dtype)
    got = gpu_fft(x, SH, dtype, window=bd.BLACKMAN_HARRIS)
    ref = acc.windowed_transform(x, bd.BLACKMAN_HARRIS, acc.ref_ctype(dtype))
    peer = acc.windowed_transform(x, bd.BLACKMAN_HARRIS, acc.ctype(dtype))
    check_rows(got, ref, peer, dtype, "windowed " + branch)
    assert_scaled_exact(lambda xs: gpu_fft(xs, SH, dtype, window=bd.BLACKMAN_HARRIS), x, got, dtype)


# ---- convolution -----------------------------------------------------------------------------------------------------
def gpu_conv_vec(x, h):
    """Per-vector convolve_signal (capi.cu convolve_taps -> conv.cu convolve)."""
    return DspVec(x[0]).convolve_signal(DspVec(h)).to_numpy().reshape(1, -1)


def gpu_conv_rows(x, h, dtype, off=0):
    """bdsp_convolve_signal_rows_* (capi.cu conv_rows -> conv.cu convolve); off: input and output pointers `off` elements past alignment."""
    L = bd.lib()
    rows, n = x.shape
    sfx = "c32" if dtype == F32 else "c64"
    hv = DspVec(h)
    plan = getattr(L, "bdsp_conv_plan_create_" + sfx)(dptr(hv), len(h))
    assert plan
    try:
        xin, out = Buf(x, off, dtype), Buf.empty(rows * n, True, off, dtype)
        assert getattr(L, "bdsp_convolve_signal_rows_" + sfx)(xin.ptr, out.ptr, n, rows, plan) == 0, L.bdsp_last_error()
        return out.get((rows, n))
    finally:
        L.bdsp_conv_plan_destroy(plan)


def conv_peer(x, h, dtype, kind):
    if kind == "fir":
        return acc.fir_peer(x, h, dtype)
    if kind == "full":
        return acc.conv_full(x, h, acc.ctype(dtype) if np.iscomplexobj(x) else dtype)
    M, geo = acc.ols_block(dtype, len(h), np.iscomplexobj(x), x.shape[-1], x.shape[0])
    return acc.ols_peer(x, h, dtype, M, geo)


# (dtype, n, rows, taps, api, peer, branch, selecting condition)
#   api: "vec" (DspVec.convolve_signal), "rows" (plan + rows entry point), "rows-offset" (pointers one element past a
#   16-byte boundary), "vec-real" (real signal and real taps).  Rows with n*rows <= 2^22.
#   The smallest tap count an overlap-save kernel sees through the C ABI is 25 (complex taps; <= 24 run the FIR) and
#   97 (real taps on real signals): 1- and 2-tap responses never reach ols4096i / ols64.
CONV_CASES = [
    (F32, 5000, 1, 24, "vec", "fir", "FIR c32, 24 complex taps, N >= 2048 + L", "convolve: L <= 24 (complex); fir_kernel big"),
    (F32, 2000, 1, 24, "vec", "fir", "FIR c32, 24 complex taps, N < 2048 + L (modulo)", "fir_kernel: N < FIR_TILE + L"),
    (F64, 5000, 1, 24, "vec", "fir", "FIR c64, 24 complex taps", "convolve: L <= 24"),
    (F64, 700, 1, 24, "vec", "fir", "FIR c64, N < 2048 + L (modulo)", "fir_kernel: N < FIR_TILE + L"),
    (F32, 5000, 1, 96, "vec-real", "fir", "FIR f32 real, 96 real taps", "convolve: L <= 96 (real)"),
    (F32, 1000, 1, 96, "vec-real", "fir", "FIR f32 real, 96 taps, modulo", "fir_kernel: N < FIR_TILE + L"),
    (F64, 3000, 1, 96, "vec-real", "fir", "FIR f64 real, 96 real taps", "convolve: L <= 96 (real)"),
    (F32, 5000, 3, 24, "rows", "fir", "FIR rows c32", "convolve: L <= 24 -> fir_convolve batch > 1"),
    (F32, 1500, 4, 17, "rows", "fir", "FIR rows c32, modulo", "convolve: L <= 24, N < FIR_TILE + L"),
    (F64, 5000, 3, 24, "rows", "fir", "FIR rows c64", "convolve: L <= 24"),
    (F32, 20000, 1, 1023, "vec", "ols", "ols4096i<true> even N", "convolve: M == 4096, olsi_applicable(4096), aligned"),
    (F32, 20001, 1, 1023, "vec", "ols", "ols4096i<false> odd N", "ols4096_convolve: N % 2 != 0"),
    (F32, 20000, 1, 25, "vec", "ols", "ols4096i<true> 25 taps", "L > 24 (FIR below)"),
    (F32, 20000, 1, 2046, "vec", "ols", "ols4096i<true> 2046 taps", "ols_block_len: L <= 2046 -> 4096; 8192 blocks*rows < 592"),
    (F32, 20000, 4, 1023, "rows", "ols", "ols4096i<true> rows", "aligned, rows > 1"),
    (F32, 20001, 3, 1023, "rows", "ols", "ols4096i<false> rows, odd N", "N % 2 != 0, rows > 1"),
    (F32, 20000, 3, 1023, "rows-offset", "ols", "ols4096i<false> rows, misaligned", "(x | y) & 15, rows > 1"),
    (F32, 20000, 3, 25, "rows-offset", "ols", "ols4096i<false> rows, misaligned, 25 taps", "(x | y) & 15"),
    (F32, 20001, 2, 2046, "rows", "ols", "ols4096i<false> rows, odd N, 2046 taps", "N % 2 != 0"),
    (F32, 50000, 1, 2047, "vec", "ols", "ols8192i<true> 2047 taps", "ols_block_len: 2047 <= L <= 4094 -> 8192"),
    (F32, 50000, 1, 4094, "vec", "ols", "ols8192i<true> 4094 taps", "olsi_applicable(8192): L <= 4094"),
    (F32, 1 << 20, 4, 1450, "rows", "ols", "ols8192i for 1450 taps, blocks*rows >= 592", "L >= 1450 && olsi_blocks(8192) * batch >= 592"),
    (F32, 1 << 20, 1, 1450, "vec", "ols", "ols4096i for 1450 taps, blocks*rows < 592", "olsi_blocks(8192) * batch < 592"),
    (F32, 50001, 1, 3000, "vec", "ols", "ols8192i<false> odd N", "ols8192_convolve: N % 2 != 0"),
    (F32, 50000, 2, 3000, "rows-offset", "ols", "ols8192i<false> rows, misaligned", "(x | y) & 15"),
    (F64, 30000, 1, 25, "vec", "ols", "ols64 25 taps", "ols64_applicable: M == 4096, L <= 2048, N >= 4096"),
    (F64, 30000, 1, 1023, "vec", "ols", "ols64 1023 taps", "ols64_applicable"),
    (F64, 30000, 1, 2048, "vec", "ols", "ols64 2048 taps", "ols_block_len: c64 L <= 2048 -> 4096"),
    (F64, 30000, 3, 1023, "rows", "ols", "ols64 rows", "convolve: ols plan, batch > 1"),
    (F64, 4096, 3, 1023, "rows", "ols", "ols64 N = 4096 exactly", "ols64_applicable: N >= 4096"),
    (F64, 30000, 2, 2048, "rows-offset", "ols", "ols64 rows, pointers one element into the buffer", "ols64 has no aligned variant"),
    (F32, 30000, 1, 1000, "vec-real", "ols", "ols_conv_kernel<float, REAL>", "convolve_taps: real signal -> plan with complex_signal false, generic"),
    (F64, 30000, 1, 1000, "vec-real", "ols", "ols_conv_kernel<double, REAL>", "real signal, generic"),
    (F32, 3000, 1, 1000, "vec", "ols", "ols_conv_kernel c32, N < 4096", "olsi_applicable(4096): N < 4096"),
    (F32, 1500, 4, 700, "rows", "ols", "ols_conv_kernel c32 rows, N < M/2 (loads wrap twice)", "N < 4096, rows > 1"),
    (F32, 6000, 2, 3000, "rows", "ols", "ols_conv_kernel c32 rows, M = 8192, N < 8192", "olsi_applicable(8192): N < 8192"),
    (F64, 3000, 1, 1000, "vec", "ols", "ols_conv_kernel c64, N < 4096", "ols64_applicable: N < 4096"),
    (F64, 1500, 3, 700, "rows", "ols", "ols_conv_kernel c64 rows, N < M/2", "N < 4096, rows > 1"),
    (F64, 50000, 1, 3000, "vec", "ols", "ols_conv_kernel c64, L > 2048 (M = 8192)", "ols_block_len c64: L > 2048"),
    (F64, 50000, 2, 4000, "rows", "ols", "ols_conv_kernel c64 rows, L > 2048", "ols_block_len c64: L > 2048"),
    (F32, 1 << 16, 1, 5000, "vec", "full", "full length c32, fused spectrum multiply (4095 .. 8192 taps)",
     "convolve: c32, L > 4094, pow2 N >= 2^15 -> fft_convolve_full, in_mul"),
    (F32, 1 << 15, 3, 8000, "rows", "full", "full length c32 rows (4095 .. 8192 taps)", "L > 4094, pow2 N >= 2^15"),
    (F32, 1 << 16, 1, 6000, "vec-real", "ols", "ols_conv_kernel<float, REAL>, M = 16384", "real signal: the 4095 .. 8192-tap full-length path is complex only"),
    (F32, 16384, 1, 9000, "vec", "full", "full length c32 N = 16384, separate spectrum multiply",
     "convolve: L > 8192; fft_convolve_full: pow2 N <= 16384 -> ew_spectrum_mul_rows"),
    (F32, 3 << 14, 1, 9000, "vec", "full", "full length c32, q*2^k N", "L > 8192, not pow2: in_mul"),
    (F32, 20000, 2, 9000, "rows", "full", "full length c32 rows, chirp-z N", "convolve: L > 8192 -> fft_convolve_full"),
    (F32, 20000, 1, 5000, "vec", "ols", "ols_conv_kernel c32, M = 16384 (non-pow2 N, L > 4094)", "L > 4094, !is_pow2(N)"),
    (F64, 40000, 1, 5000, "vec", "full", "full length c64", "convolve: L > ols_max_taps (4096)"),
    (F64, 1 << 15, 2, 4500, "rows", "full", "full length c64 rows", "convolve: L > ols_max_taps, no ols plan"),
]


@pytest.mark.parametrize("dtype,n,rows,taps,api,kind,branch,cond", CONV_CASES,
                         ids=["%s-%d-x%d-L%d-%s" % ("c32" if c[0] == F32 else "c64", c[1], c[2], c[3], c[4]) for c in CONV_CASES])
def test_convolution_accuracy(dtype, n, rows, taps, api, kind, branch, cond):
    rng = np.random.default_rng(n * 17 + taps * 3 + rows)
    x = rand_c(rng, (rows, n), dtype)
    h = (rand_c(rng, taps, dtype) / 10).astype(x.dtype)
    if api == "vec-real":
        x, h = np.ascontiguousarray(x.real), np.ascontiguousarray(h.real)
    if api.startswith("rows"):
        off = 1 if api == "rows-offset" else 0
        run = lambda xs: gpu_conv_rows(xs, h, dtype, off)  # noqa: E731
    else:
        run = lambda xs: gpu_conv_vec(xs, h)  # noqa: E731
    got = run(x)
    ref = acc.conv_ref(x, h, dtype)
    peer = conv_peer(x, h, dtype, kind)
    k_rel, k_el = WIDER.get(branch, (acc.K_REL, acc.K_EL))
    check_rows(got, ref, peer, dtype, "conv %s L=%d %s" % (branch, taps, api), k_rel, k_el, tol_n=max(n, 4096))
    assert_scaled_exact(run, x, got, dtype)
