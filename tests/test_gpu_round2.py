"""Round-2 GPU tests: the fused 8192-point overlap-save kernel, the full-length convolution path with mixed-radix and
chirp-z lengths (ADVICE r1: workspace slot clash), thread safety of shared impulse responses and of the per-thread
workspaces, and the bounded chirp-filter cache.  Everything goes through the C ABI."""
import math
import threading

import numpy as np
import pytest

import basic_dsp_b200 as bd
from basic_dsp_b200 import DspVec
from oracle import dsp_oracle as o

pytestmark = pytest.mark.gpu


def tol(n, dtype):
    return (1e-5 if dtype == np.float32 else 1e-12) * max(1.0, math.log2(max(n, 2)))


def dptr(v):
    return v._fn("bdsp_device_ptr")(v._h)


def rand_c(rng, n, dtype):
    ct = np.complex64 if dtype == np.float32 else np.complex128
    return (rng.uniform(-10, 10, n) + 1j * rng.uniform(-10, 10, n)).astype(ct)


# ---- fused 8192-point blocks (c32, 1450 <= L <= 4094 in the throughput regime; 2047 <= L <= 4094 always) ----------
@pytest.mark.parametrize("n,l", [(8192, 2047), (8192, 4094), (8193, 3000), (20001, 2500), (1 << 16, 4093), (100000, 3333),
                                 (1 << 22, 1500), (1 << 22, 2046), (3 * (1 << 20) + 2, 1451)])
def test_convolve_signal_8192_point_blocks(n, l):
    rng = np.random.default_rng(n + l)
    x = rand_c(rng, n, np.float32)
    h = (rand_c(rng, l, np.float32) / 10).astype(np.complex64)
    got = DspVec(x).convolve_signal(DspVec(h)).to_numpy()
    assert o.rel_l2(got, o.convolve_signal(x, h)) <= tol(8192, np.float32)


@pytest.mark.parametrize("n,rows,l", [(100000, 40, 2000), (1 << 16, 64, 1450), (50001, 33, 4094), (1 << 20, 6, 1023)])
def test_convolve_signal_rows_8192_point_blocks(n, rows, l):
    L = bd.lib()
    rng = np.random.default_rng(n + rows + l)
    x = rand_c(rng, n * rows, np.float32)
    h = (rand_c(rng, l, np.float32) / 10).astype(np.complex64)
    xv, hv, out = DspVec(x), DspVec(h), DspVec.zeros(2 * n * rows, is_complex=True)
    plan = L.bdsp_conv_plan_create_c32(dptr(hv), l)
    assert plan
    assert L.bdsp_convolve_signal_rows_c32(dptr(xv), dptr(out), n, rows, plan) == 0
    got = out.to_numpy().reshape(rows, n)
    xr = x.reshape(rows, n)
    for r in range(rows):
        assert o.rel_l2(got[r], o.convolve_signal(xr[r], h)) <= tol(8192, np.float32), r
    L.bdsp_conv_plan_destroy(plan)


@pytest.mark.parametrize("dtype,n,rows,l", [(np.float32, 1 << 16, 3, 4095), (np.float32, 1 << 16, 2, 8191), (np.float32, 1 << 16, 2, 8192),
                                            (np.float32, 20000, 2, 4096), (np.float64, 1 << 15, 2, 4095), (np.float64, 1 << 15, 2, 4096),
                                            (np.float32, 20000, 3, 24), (np.float64, 20000, 2, 24), (np.float64, 20000, 3, 1023),
                                            (np.float64, 20000, 2, 2048), (np.float32, 3000, 4, 1000), (np.float64, 1500, 3, 700),
                                            (np.float32, 20001, 3, 1023)])
def test_convolve_signal_rows_tap_counts_at_the_block_limits(dtype, n, rows, l):
    """Impulse responses one short of / exactly at the longest block transform (regression: the 8192-point block step is 0
    for 8191 taps and must not be divided by), and at the other limits of the rows dispatch: <= 24 taps (direct FIR),
    c64 <= 2048 taps (fused 4096-point blocks), fewer than 4096 points (generic blocks whose loads wrap around the row)
    and odd row lengths (the unaligned fused 4096-point kernel)."""
    L = bd.lib()
    sfx = "c32" if dtype == np.float32 else "c64"
    rng = np.random.default_rng(n + l + rows)
    x = rand_c(rng, n * rows, dtype)
    h = (rand_c(rng, l, dtype) / 10).astype(x.dtype)
    xv, hv = DspVec(x), DspVec(h)
    out = DspVec.zeros(2 * n * rows, is_complex=True, dtype=dtype)
    plan = getattr(L, "bdsp_conv_plan_create_" + sfx)(dptr(hv), l)
    assert plan
    assert getattr(L, "bdsp_convolve_signal_rows_" + sfx)(dptr(xv), dptr(out), n, rows, plan) == 0
    got = out.to_numpy().reshape(rows, n)
    for r in range(rows):
        assert o.rel_l2(got[r], o.convolve_signal(x.reshape(rows, n)[r], h)) <= tol(n, dtype), r
    L.bdsp_conv_plan_destroy(plan)
    got1 = DspVec(x[:n]).convolve_signal(hv).to_numpy()
    assert o.rel_l2(got1, o.convolve_signal(x[:n], h)) <= tol(n, dtype)


def test_real_taps_on_complex_signal_fused_blocks():
    rng = np.random.default_rng(77)
    for n, l in [(30000, 1023), (70000, 3001)]:
        x = rand_c(rng, n, np.float32)
        h = rng.uniform(-1, 1, l).astype(np.float32)
        got = DspVec(x).convolve_signal(DspVec(h.astype(np.complex64))).to_numpy()
        assert o.rel_l2(got, o.convolve_signal(x, h.astype(np.complex128))) <= tol(8192, np.float32)


# ---- full-length frequency-domain path: impulse responses too long for a block transform ---------------------------
@pytest.mark.parametrize("dtype,n,l", [(np.float32, 3 * 32768, 9001), (np.float32, 31 * 16384, 8500), (np.float32, 1 << 17, 20000),
                                       (np.float32, 40000, 9000), (np.float64, 3 * 32768, 4500), (np.float64, 31 * 16384, 5000),
                                       (np.float64, 20001, 4099)])
def test_convolve_signal_full_length_path(dtype, n, l):
    rng = np.random.default_rng(n + l)
    x = rand_c(rng, n, dtype)
    h = (rand_c(rng, l, dtype) / 10).astype(x.dtype)
    got = DspVec(x).convolve_signal(DspVec(h)).to_numpy()
    assert o.rel_l2(got, o.convolve_signal(x, h)) <= tol(n, dtype)


@pytest.mark.parametrize("dtype,n,rows,l", [(np.float32, 3 * 32768, 3, 9001), (np.float64, 3 * 16384, 4, 4500), (np.float32, 31 * 4096, 5, 10000)])
def test_convolve_signal_rows_full_length_path(dtype, n, rows, l):
    L = bd.lib()
    sfx = "c32" if dtype == np.float32 else "c64"
    rng = np.random.default_rng(n + l + rows)
    x = rand_c(rng, n * rows, dtype)
    h = (rand_c(rng, l, dtype) / 10).astype(x.dtype)
    xv, hv = DspVec(x), DspVec(h)
    out = DspVec.zeros(2 * n * rows, is_complex=True, dtype=dtype)
    plan = getattr(L, "bdsp_conv_plan_create_" + sfx)(dptr(hv), l)
    assert plan
    for _ in range(2):   # the second call reuses (and must not have clobbered) every workspace
        assert getattr(L, "bdsp_convolve_signal_rows_" + sfx)(dptr(xv), dptr(out), n, rows, plan) == 0
        got = out.to_numpy().reshape(rows, n)
        for r in range(rows):
            assert o.rel_l2(got[r], o.convolve_signal(x.reshape(rows, n)[r], h)) <= tol(n, dtype), r
    L.bdsp_conv_plan_destroy(plan)


# ---- threads -----------------------------------------------------------------------------------------------------------
def test_two_threads_share_one_impulse_response():
    """`impulse_response` is a borrowed, read-only argument (facade32.rs:1171): two threads convolving different
    vectors with ONE shared response, each on its own stream, while the response's spectrum cache is cold."""
    L = bd.lib()
    rng = np.random.default_rng(5)
    n, l = 1 << 18, 1023
    h = (rand_c(rng, l, np.float32) / 10).astype(np.complex64)
    xs = [rand_c(rng, n, np.float32) for _ in range(2)]
    refs = [o.convolve_signal(x, h) for x in xs]
    errs = []

    for attempt in range(4):
        hv = DspVec(h)          # fresh response: the plan is built inside the racing calls
        start = threading.Barrier(2)

        def work(i):
            try:
                st = L.bdsp_stream_create()
                L.bdsp_set_stream(st)
                v = DspVec(xs[i])
                start.wait()
                for _ in range(3):
                    v.upload(xs[i].view(np.float32))
                    got = v.convolve_signal(hv).to_numpy()
                    e = o.rel_l2(got, refs[i])
                    if not e <= tol(4096, np.float32):
                        errs.append((attempt, i, e))
                del v
                L.bdsp_set_stream(None)
                L.bdsp_stream_destroy(st)
            except Exception as exc:  # noqa: BLE001
                errs.append((attempt, i, repr(exc)))

        ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
        [t.start() for t in ts]
        [t.join() for t in ts]
    assert not errs, errs


def test_threads_without_streams_do_not_share_workspaces():
    """Two threads on the default stream running multi-kernel transforms (three-pass, mixed radix, chirp-z) on their
    own vectors: scratch buffers are per thread (ADVICE r1)."""
    rng = np.random.default_rng(6)
    sizes = [3 * (1 << 16), 1 << 21, 10007 * 3, 1 << 17]
    data = {n: rand_c(rng, n, np.float32) for n in sizes}
    refs = {n: o.plain_fft(data[n]) for n in sizes}
    errs = []

    def work(order):
        try:
            for _ in range(3):
                for n in order:
                    got = DspVec(data[n]).plain_fft().to_numpy()
                    e = o.rel_l2(got, refs[n])
                    if not e <= tol(n, np.float32):
                        errs.append((n, e))
        except Exception as exc:  # noqa: BLE001
            errs.append(repr(exc))

    ts = [threading.Thread(target=work, args=(sizes,)), threading.Thread(target=work, args=(sizes[::-1],))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs


def test_chirp_filter_cache_is_bounded():
    """Many distinct non-smooth lengths: the chirp-z filter cache evicts instead of growing without bound
    (1 GiB cap; each of these lengths needs a 2^22-point c64 filter = 64 MiB)."""
    L = bd.lib()
    rng = np.random.default_rng(8)
    free0 = L.bdsp_mem_free() if hasattr(L, "bdsp_mem_free") else None
    primes = [1000003, 1000033, 1000037, 1000039, 1000081, 1000099, 1000117, 1000121, 1000133, 1000151, 1000159, 1000171,
              1000183, 1000187, 1000193, 1000199, 1000211, 1000213, 1000231, 1000249]
    for n in primes:
        x = rand_c(rng, n, np.float64)
        got = DspVec(x).plain_fft().to_numpy()
        if n in (primes[0], primes[-1]):
            assert o.rel_l2(got, o.plain_fft(x)) <= tol(n, np.float64)
    # the first length again (evicted by now: 20 x 64 MiB > 1 GiB) still gives the right answer
    x = rand_c(rng, primes[0], np.float64)
    assert o.rel_l2(DspVec(x).plain_fft().to_numpy(), o.plain_fft(x)) <= tol(primes[0], np.float64)
    if free0 is not None:
        assert free0 - L.bdsp_mem_free() < (3 << 30)


def test_device_ptr_access_invalidates_cached_spectrum():
    L = bd.lib()
    rng = np.random.default_rng(9)
    n, l = 20000, 500
    x = rand_c(rng, n, np.float32)
    h1 = (rand_c(rng, l, np.float32) / 10).astype(np.complex64)
    h2 = (rand_c(rng, l, np.float32) / 10).astype(np.complex64)
    hv = DspVec(h1)
    assert o.rel_l2(DspVec(x).convolve_signal(hv).to_numpy(), o.convolve_signal(x, h1)) <= tol(4096, np.float32)
    L.bdsp_memcpy_h2d(dptr(hv), h2.ctypes.data, l * 8)      # refresh the taps through the raw device pointer
    L.bdsp_sync()
    assert o.rel_l2(DspVec(x).convolve_signal(hv).to_numpy(), o.convolve_signal(x, h2)) <= tol(4096, np.float32)


# ---- batched (matrix-row) forms beyond fft / convolve_signal (matrix/src/time_freq.rs:52-74, matrix/src/complex.rs:18-26) ---------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_magnitude_phase_rows(dtype):
    L = bd.lib()
    sfx = "32" if dtype == np.float32 else "64"
    rng = np.random.default_rng(11)
    points, rows = 3001, 7
    x = rand_c(rng, points * rows, dtype)
    xv = DspVec(x)
    out = DspVec.zeros(points * rows, dtype=dtype)
    assert getattr(L, "bdsp_magnitude_rows_c" + sfx)(dptr(xv), dptr(out), points, rows) == 0
    assert o.ulp_diff(out.to_numpy(), o.magnitude(x, dtype), dtype).max() <= 4
    # (the C ABI's per-vector magnitude32 is the reference's magnitude_b = sqrt(re^2 + im^2), facade32.rs:559; the rows form is the
    # trait's magnitude = hypot, complex_to_real.rs:376: both within 4 ulp of the oracle, not bit-identical to each other)
    assert getattr(L, "bdsp_phase_rows_c" + sfx)(dptr(xv), dptr(out), points, rows) == 0
    assert o.ulp_diff(out.to_numpy(), o.phase(x, dtype), dtype).max() <= 4
    assert getattr(L, "bdsp_magnitude_squared_rows_c" + sfx)(dptr(xv), dptr(out), points, rows) == 0
    assert o.ulp_diff(out.to_numpy(), o.magnitude_squared(x, dtype), dtype).max() <= 4


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_fused_chain_rows(dtype):
    L = bd.lib()
    sfx = "32" if dtype == np.float32 else "64"
    rng = np.random.default_rng(12)
    points, rows = 5000, 5
    x, w = rand_c(rng, points * rows, dtype), rand_c(rng, points * rows, dtype)
    c = complex(0.75, -1.5)
    xv, wv = DspVec(x), DspVec(w)
    mag, ph = DspVec.zeros(points * rows, dtype=dtype), DspVec.zeros(points * rows, dtype=dtype)
    assert getattr(L, "bdsp_scale_mul_mag_phase_rows_c" + sfx)(dptr(xv), dptr(wv), dptr(mag), dptr(ph), points, rows, c.real, c.imag, 0) == 0
    ref = o.mul(o.complex_scale(x, c, dtype), w, dtype)
    assert o.ulp_diff(mag.to_numpy(), o.magnitude(ref, dtype), dtype).max() <= 4
    assert o.ulp_diff(ph.to_numpy(), o.phase(ref, dtype), dtype).max() <= 4
    # bit-identical to the per-vector fused call
    m1, p1 = DspVec.zeros(0, dtype=dtype), DspVec.zeros(0, dtype=dtype)
    DspVec(x[:points]).scale_mul_mag_phase(c, DspVec(w[:points]), m1, p1)
    assert np.array_equal(m1.to_numpy(), mag.to_numpy()[:points]) and np.array_equal(p1.to_numpy(), ph.to_numpy()[:points])


@pytest.mark.parametrize("dtype,cplx_", [(np.float32, False), (np.float32, True), (np.float64, False)])
def test_interpolatef_rows(dtype, cplx_):
    import ctypes
    L = bd.lib()
    sfx = "32" if dtype == np.float32 else "64"
    rng = np.random.default_rng(13)
    points, rows, F, conv_len = 3000, 4, 4, 12
    x = rand_c(rng, points * rows, dtype) if cplx_ else rng.uniform(-10, 10, points * rows).astype(dtype)
    xv = DspVec(x)
    out = DspVec.zeros((2 if cplx_ else 1) * points * rows * F, is_complex=cplx_, dtype=dtype)
    npts = ctypes.c_size_t(0)
    rc = getattr(L, "bdsp_interpolatef_rows" + sfx)(dptr(xv), dptr(out), points, rows, 1 if cplx_ else 0, bd.SINC, 0.0, float(F), 0.0, conv_len,
                                                    ctypes.byref(npts))
    assert rc == 0 and npts.value == points * F
    got = out.to_numpy().reshape(rows, points * F)
    xr = x.reshape(rows, points)
    for r in range(rows):
        ref = o.interpolatef(xr[r], lambda t: o.sinc_impulse(t, dtype), float(F), 0.0, conv_len, dtype)
        assert o.rel_l2(got[r], ref) <= tol(4096, dtype)
        # identical to the per-vector trait call
        assert np.array_equal(got[r], DspVec(xr[r].copy()).interpolatef(bd.SINC, 0.0, float(F), 0.0, conv_len).to_numpy())
    # both sides of every condition of the path rule (polyphase: conv_len <= 202, new_len >= 2000, integer factor)
    ulp = float(np.spacing(dtype(4)))
    near, off = (4 + ulp, 4 + 3 * ulp) if dtype == np.float32 else (4 + 5e-7, 4 + 2e-6)
    shapes = [(3000, 2.5, 12, False), (3000, 2.0, 202, True), (3000, 2.0, 203, False), (3000, near, 12, True), (3000, off, 12, False)]
    shapes += [(333, 3.0, 12, False), (500, 2.0, 12, True)] if cplx_ else [(999, 2.0, 12, False), (1000, 2.0, 12, True)]   # new_len 1998, 2000
    for points, factor, conv_len, poly in shapes:
        rows, scalars = 2, (2 if cplx_ else 1) * points
        new_len = o.interpolatef_new_len(scalars, factor, dtype)
        assert o.interpolatef_uses_fast_path(min(conv_len, points // 2), new_len, factor, dtype) == poly
        x = rand_c(rng, points * rows, dtype) if cplx_ else rng.uniform(-10, 10, points * rows).astype(dtype)
        xv, out = DspVec(x), DspVec.zeros(new_len * rows, is_complex=cplx_, dtype=dtype)
        rc = getattr(L, "bdsp_interpolatef_rows" + sfx)(dptr(xv), dptr(out), points, rows, 1 if cplx_ else 0, bd.SINC, 0.0, factor, 0.25,
                                                        conv_len, ctypes.byref(npts))
        assert rc == 0 and npts.value == new_len // (2 if cplx_ else 1), (points, factor, conv_len)
        got = out.to_numpy().reshape(rows, npts.value)
        for r, xr in enumerate(x.reshape(rows, points)):
            assert np.array_equal(got[r], DspVec(xr.copy()).interpolatef(bd.SINC, 0.0, factor, 0.25, conv_len).to_numpy()), (points, factor, conv_len)


def test_convolve_complex_callback_wraps_around_short_vectors():
    """2 len + 1 > points: the tap window wraps around the vector (ReverseWrappingIterator, time_freq/mod.rs:788-848;
    ADVICE r1: the complex-tap path used to return InvalidArgumentLength)."""
    rng = np.random.default_rng(78)
    for n, length in [(12, 10), (7, 7), (30, 20)]:
        x = rand_c(rng, n, np.float32)
        fn = lambda t: complex(o.sinc_impulse(t, np.float32), 0.5 * o.sinc_impulse(t * 0.5, np.float32))
        got = DspVec(x).convolve_complex(fn, 0.5, length).to_numpy()
        L_ = min(length, n)
        idx = np.arange(n)
        ref = np.zeros(n, dtype=np.complex128)
        for m in range(-L_, L_ + 1):
            ref += x[(idx + m) % n].astype(np.complex128) * fn(np.float32(-m * 0.5))
        assert o.rel_l2(got, ref) <= tol(4096, np.float32), (n, length)


# ---- multipliers fused into the first load of a transform (FftOpts::in_mul) --------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [16, 1000, 1001, 4096, 3 * 4096, 1 << 14, 1 << 15, 1 << 16, 3 * (1 << 15), 40000, 1 << 19, 1 << 21, 3 * (1 << 18), 5 * (1 << 17)])
def test_windowed_fft_every_transform_path(n, dtype):
    """windowed_fft = apply_window + fft (time_to_freq.rs:167-175) with the window carried by the transform's first load:
    single-CTA, two- and three-pass (generic, c64 tiles, packed c32 columns), mixed radix and chirp-z lengths; complex and
    real vectors."""
    rng = np.random.default_rng(n)
    x = rand_c(rng, n, dtype)
    for kind in (1, 2):
        X = DspVec(x).windowed_fft(kind).to_numpy()
        ref = o.windowed_fft(x, kind, dtype)
        assert o.rel_l2(X, ref) <= tol(n, dtype), kind
        # identical to the two separate calls up to summation order
        X2 = DspVec(x).apply_window(kind).fft().to_numpy()
        assert o.rel_l2(X, X2) <= tol(n, dtype), kind
    r = rng.uniform(-10, 10, n).astype(dtype)
    R = DspVec(r).windowed_fft(1).to_numpy()
    assert o.rel_l2(R, o.windowed_fft(r.astype(x.dtype), 1, dtype)) <= tol(n, dtype)


@pytest.mark.parametrize("dtype,n,l", [(np.float32, 1 << 15, 9000), (np.float32, 1 << 21, 8200), (np.float32, 5 * (1 << 13), 8500),
                                       (np.float64, 1 << 14, 4100), (np.float64, 1 << 16, 5000), (np.float64, 3 * (1 << 14), 4100),
                                       (np.float64, 30001, 4100)])
def test_convolve_signal_full_length_fused_spectrum_multiply(dtype, n, l):
    """Full-length frequency-domain convolution (impulse responses too long for a block transform): the spectrum multiply
    (convolution.rs:427-429) rides on the inverse transform's first load."""
    rng = np.random.default_rng(n + l)
    x = rand_c(rng, n, dtype)
    h = (rand_c(rng, l, dtype) / 10).astype(x.dtype)
    got = DspVec(x).convolve_signal(DspVec(h)).to_numpy()
    assert o.rel_l2(got, o.convolve_signal(x, h)) <= tol(n, dtype)
    xr = rng.uniform(-10, 10, n).astype(dtype)
    hr = (rng.uniform(-1, 1, l) / 10).astype(dtype)
    gr = DspVec(xr).convolve_signal(DspVec(hr)).to_numpy()
    assert o.rel_l2(gr, o.convolve_signal(xr.astype(x.dtype), hr.astype(x.dtype)).real) <= tol(n, dtype)


# ---- single-launch 2^16-point transform on a 16-CTA cluster (fftc.cu) ---------------------------------------------------
@pytest.mark.parametrize("rows", [1, 3, 8])
def test_cluster_fft_65536(rows):
    """Few 2^16-point c32 vectors take one launch on a thread-block cluster (transposition through distributed shared
    memory); every flag combination of the rows entry point and the vector methods against the oracle."""
    L = bd.lib()
    n = 1 << 16
    rng = np.random.default_rng(rows)
    x = rand_c(rng, n * rows, np.float32)
    xv = DspVec(x)
    out = DspVec.zeros(2 * n * rows, is_complex=True)
    xr = x.reshape(rows, n)
    for flags, ref in ((0, o.plain_fft), (bd.F_SHIFT, o.fft), (bd.F_INVERSE, lambda v: o.plain_ifft(v)),
                       (bd.F_INVERSE | bd.F_SHIFT, lambda v: o.ifft(v))):
        before = bd.kernel_launch_count()
        assert L.bdsp_fft_rows_c32(dptr(xv), dptr(out), n, rows, flags) == 0
        assert bd.kernel_launch_count() - before == 1
        got = out.to_numpy().reshape(rows, n)
        for r in range(rows):
            want = np.asarray(ref(xr[r]))
            assert o.rel_l2(got[r], want) <= tol(n, np.float32), (flags, r)
    v = DspVec(xr[0])
    assert o.rel_l2(v.fft().ifft().to_numpy(), xr[0]) <= 2 * tol(n, np.float32)


# ---- seeded sweep over lengths / rows / flags: every dispatch branch of the transforms ----------------------------------
def _sweep_lengths():
    rng = np.random.default_rng(20261017)
    out = []
    # powers of two, q * 2^k with odd q <= 31, and arbitrary lengths (chirp-z), small to multi-pass
    for k in rng.integers(1, 21, 10):
        out.append(1 << int(k))
    for _ in range(12):
        q = int(rng.choice([3, 5, 7, 9, 11, 13, 15, 17, 21, 25, 27, 31]))
        out.append(q << int(rng.integers(1, 16)))
    for _ in range(8):
        out.append(int(rng.integers(3, 200000)) | 1)
    return sorted(set(out))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", _sweep_lengths())
def test_fft_rows_sweep(n, dtype):
    """Rows entry point over a seeded sample of lengths with every flag combination, against pocketfft in c128."""
    L = bd.lib()
    sfx = "c32" if dtype == np.float32 else "c64"
    rng = np.random.default_rng(n)
    rows = int(max(1, min(5, (1 << 19) // n)))
    x = rand_c(rng, n * rows, dtype)
    xv = DspVec(x)
    out = DspVec.zeros(2 * n * rows, is_complex=True, dtype=dtype)
    xr = x.reshape(rows, n)
    fn = getattr(L, "bdsp_fft_rows_" + sfx)
    for flags, ref in ((0, o.plain_fft), (bd.F_SHIFT, o.fft), (bd.F_INVERSE, o.plain_ifft), (bd.F_INVERSE | bd.F_SHIFT, o.ifft)):
        assert fn(dptr(xv), dptr(out), n, rows, flags) == 0
        got = out.to_numpy().reshape(rows, n)
        for r in range(rows):
            assert o.rel_l2(got[r], np.asarray(ref(xr[r]))) <= 2 * tol(n, dtype), (flags, r)
    # magnitude epilogue and real input
    mag = DspVec.zeros(n * rows, is_complex=False, dtype=dtype)
    assert fn(dptr(xv), dptr(mag), n, rows, bd.F_SHIFT | bd.F_MAGNITUDE) == 0
    gm = mag.to_numpy().reshape(rows, n)
    for r in range(rows):
        assert o.rel_l2(gm[r], np.abs(o.fft(xr[r]))) <= 2 * tol(n, dtype), r
    xre = DspVec(np.ascontiguousarray(x.real))
    assert fn(dptr(xre), dptr(out), n, rows, bd.F_REAL_INPUT) == 0
    gr = out.to_numpy().reshape(rows, n)
    for r in range(rows):
        assert o.rel_l2(gr[r], o.plain_fft(xr[r].real)) <= 2 * tol(n, dtype), r


def _sweep_conv():
    rng = np.random.default_rng(20261018)
    out = []
    for _ in range(14):
        n = int(rng.integers(64, 300000))
        l = int(rng.integers(1, min(n, 9000)))
        out.append((n, l))
    return out


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,l", _sweep_conv())
def test_convolve_signal_sweep(n, l, dtype):
    rng = np.random.default_rng(n * 31 + l)
    x = rand_c(rng, n, dtype)
    h = (rand_c(rng, l, dtype) / 10).astype(x.dtype)
    got = DspVec(x).convolve_signal(DspVec(h)).to_numpy()
    ref = o.convolve_signal_direct(x, h) if n * l < 3e7 else o.convolve_signal(x, h)
    assert o.rel_l2(got, ref) <= tol(max(n, 4096), dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,rows", [(256, 512), (1024, 64), (4096, 32), (16384, 8), (1000, 70), (3 * 1024, 24), (1 << 15, 4), (1 << 17, 2), (64, 3)])
def test_windowed_fft_rows(n, rows, dtype):
    """BDSP_F_WINDOW: windowed_fft of every row (matrix/src/time_freq.rs:69-74) in one call; complex and real rows; equals the
    per-vector windowed_fft."""
    L = bd.lib()
    sfx = "c32" if dtype == np.float32 else "c64"
    fn = getattr(L, "bdsp_fft_rows_" + sfx)
    rng = np.random.default_rng(n + rows)
    x = rand_c(rng, n * rows, dtype)
    xv = DspVec(x)
    out = DspVec.zeros(2 * n * rows, is_complex=True, dtype=dtype)
    xr = x.reshape(rows, n)
    for kind in (bd.HAMMING, bd.BLACKMAN_HARRIS, bd.RECTANGULAR):
        assert fn(dptr(xv), dptr(out), n, rows, bd.F_SHIFT | bd.F_WINDOW(kind)) == 0
        got = out.to_numpy().reshape(rows, n)
        for r in (0, rows // 2, rows - 1):
            assert o.rel_l2(got[r], o.windowed_fft(xr[r], kind, dtype)) <= tol(n, dtype), (kind, r)
    one = DspVec(xr[rows - 1]).windowed_fft(bd.BLACKMAN_HARRIS).to_numpy()
    assert fn(dptr(xv), dptr(out), n, rows, bd.F_SHIFT | bd.F_WINDOW(bd.BLACKMAN_HARRIS)) == 0
    assert o.rel_l2(out.to_numpy().reshape(rows, n)[rows - 1], one) <= tol(n, dtype)
    xre = DspVec(np.ascontiguousarray(x.real))
    assert fn(dptr(xre), dptr(out), n, rows, bd.F_REAL_INPUT | bd.F_SHIFT | bd.F_WINDOW(bd.HAMMING)) == 0
    gr = out.to_numpy().reshape(rows, n)
    for r in (0, rows - 1):
        assert o.rel_l2(gr[r], o.windowed_fft(xr[r].real.astype(x.dtype), bd.HAMMING, dtype)) <= tol(n, dtype), r
    assert fn(dptr(xv), dptr(out), n, rows, bd.F_INVERSE | bd.F_WINDOW(bd.HAMMING)) != 0   # forward transforms only


def test_two_devices_in_one_process():
    """One process driving two devices (bdsp_set_device): kernels that need more than 48 KB of dynamic shared memory are
    configured per device, plans / tables / staging buffers / workspaces are per device."""
    if bd.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = bd.lib()
    rng = np.random.default_rng(2)
    try:
        for dev in (0, 1, 0):
            assert L.bdsp_set_device(dev) == 0
            n, rows = 16384, 3
            x = rand_c(rng, n * rows, np.float32)
            xv = DspVec(x)
            out = DspVec.zeros(2 * n * rows, is_complex=True)
            assert L.bdsp_fft_rows_c32(dptr(xv), dptr(out), n, rows, 0) == 0
            got = out.to_numpy().reshape(rows, n)
            assert o.rel_l2(got[1], o.plain_fft(x.reshape(rows, n)[1])) <= tol(n, np.float32)
            xs = rand_c(rng, 1 << 16, np.float32)
            h = (rand_c(rng, 1023, np.float32) / 10).astype(np.complex64)
            y = DspVec(xs).convolve_signal(DspVec(h)).to_numpy()
            assert o.rel_l2(y, o.convolve_signal(xs, h)) <= tol(1 << 16, np.float32)
            assert o.rel_l2(DspVec(xs).fft().ifft().to_numpy(), xs) <= 2 * tol(1 << 16, np.float32)
            xd = rand_c(rng, 3 * (1 << 14), np.float64)
            assert o.rel_l2(DspVec(xd).plain_fft().to_numpy(), o.plain_fft(xd)) <= tol(xd.size, np.float64)
            r = rng.uniform(-1, 1, 20001).astype(np.float32)
            DspVec(r).interpolatef(bd.SINC, 0.0, 4.0, 0.0, 12).to_numpy()
            # a callback window: its table is staged in this device's memory
            xw = rand_c(rng, 1001, np.float32)
            w = np.array([np.float32(1.0 + i / 1001) for i in range(1001)])
            got = DspVec(xw).custom_window("apply_custom_window", lambda i, p: 1.0 + i / p, is_symmetric=False).to_numpy()
            assert o.rel_l2(got, xw * w) < 1e-6
            assert abs(DspVec(r).sum() - float(np.sum(r.astype(np.float64)))) < 1e-2
    finally:
        L.bdsp_set_device(0)
