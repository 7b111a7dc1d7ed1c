"""bdsp_ifft_frames_*: a device signal from the spectra of its overlapping frames (inverse short-time transform).

The definition the tests hold the library to is test_ifft_frames_reference.synthesis: the inverse transform of every
frame scaled by 1/points, then the least-squares weighted overlap-add.  On top of accuracy against a higher-precision
reference: the round trip through bdsp_fft_frames_*, byte identity with bdsp_fft_rows_* where frames do not overlap, the
number of kernel launches, bit-reproducible results, that a frame only reaches the samples it covers, that nothing
outside the output is written, and the error contract."""
import itertools

import numpy as np
import pytest

import basic_dsp_b200 as bd
from oracle import accuracy as acc
from oracle.accuracy import F_INVERSE as INV, F_MAGNITUDE as MAG, F_REAL_INPUT as REAL, F_SHIFT as SH
from test_gpu_accuracy import F32, F64, Buf, check_rows, rand_c
from test_ifft_frames_reference import analysis, synthesis

pytestmark = pytest.mark.gpu

RO = bd.F_REAL_OUTPUT
PAD = 64   # sentinel points before and after every output


def fn(name, dtype):
    return getattr(bd.lib(), "%s_%s" % (name, "c32" if dtype == F32 else "c64"))


def run_ifft(X, hop, flags, dtype):
    """bdsp_ifft_frames_* over the spectra X (frames x points) -> (output, kernel launches); checks that the PAD points
    on either side of the output keep their sentinel."""
    frames, points = X.shape
    length = (frames - 1) * hop + points
    xin = Buf(X, 0, dtype)
    sentinel = np.full(length + 2 * PAD, 1234.5, dtype=dtype if flags & RO else acc.ctype(dtype))
    out = Buf(sentinel, 0, dtype)
    before = bd.kernel_launch_count()
    rc = fn("bdsp_ifft_frames", dtype)(xin.ptr, out.ptr + PAD * out.esize, points, hop, frames, flags)
    launches = bd.kernel_launch_count() - before
    assert rc == 0, bd.lib().bdsp_last_error()
    got = out.get(sentinel.shape)
    assert np.array_equal(got[:PAD], sentinel[:PAD]) and np.array_equal(got[-PAD:], sentinel[-PAD:]), "write outside the output"
    return got[PAD:-PAD], launches


def run_rows(X, flags, dtype):
    """bdsp_fft_rows_* over the rows of X -> (result rows, kernel launches)"""
    frames, points = X.shape
    xin = Buf(X, 0, dtype)
    out = Buf.empty(frames * points, not flags & MAG, 0, dtype)
    before = bd.kernel_launch_count()
    rc = fn("bdsp_fft_rows", dtype)(xin.ptr, out.ptr, points, frames, flags)
    launches = bd.kernel_launch_count() - before
    assert rc == 0, bd.lib().bdsp_last_error()
    return out.get((frames, points)), launches


def run_frames(x, points, hop, flags, dtype):
    """bdsp_fft_frames_* over the device copy of x -> spectra (frames x points)"""
    frames = 1 + (x.size - points) // hop
    xin = Buf(x, 0, dtype)
    out = Buf.empty(frames * points, True, 0, dtype)
    rc = fn("bdsp_fft_frames", dtype)(xin.ptr, out.ptr, points, hop, frames, flags)
    assert rc == 0, bd.lib().bdsp_last_error()
    return out.get((frames, points))


def same_bytes(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def kind_of(flags):
    wk = (flags >> 8) & 15
    return wk - 1 if wk else None


def library_window(kind, points, dtype):
    """The built-in window as the library evaluates it in `dtype` (apply_window on ones: the same window_value_dev and
    mirrored index as the synthesis table), or None without a window."""
    if kind not in (bd.TRIANGULAR, bd.HAMMING, bd.BLACKMAN_HARRIS):
        return None
    return bd.DspVec(np.ones(points, dtype=dtype), is_complex=False, dtype=dtype).apply_window(kind).to_numpy()


# ---- 1. accuracy against a higher-precision reference ------------------------------------------------------------------
# The reference and the peer take the library's window table.  In float32 the Blackman-Harris end value (6e-5) is the sum of
# four terms near 0.1 ... 0.5 and carries a relative error of 5e-4 ... 9e-4; a sample that one frame covers is w y / w^2 = y / w,
# so a window evaluated apart from the library's would put that error into the comparison, in the reference and the peer
# alike.  The round trip below holds the window's own rounding to account: analysis and synthesis share the table.
POINTS = (64, 1024, 4096, 8192, 16384, 1000, 3072)
FLAGS = [0, SH, RO] + [SH | bd.F_WINDOW(k) for k in range(4)]


def _grid():
    """A seeded subset of precision x points x hop x flags; about 2^17 spectrum points per case."""
    cases = []
    for dtype, points in itertools.product((F32, F64), POINTS):
        hops = sorted({points // 4, points // 2 - 1, points} | ({1} if points <= 1024 else set()))
        for hop in hops:
            frames = 9 if hop == 1 else max(4, (1 << 17) // points)
            cases.extend((dtype, points, hop, frames, flags) for flags in FLAGS)
    rng = np.random.default_rng(2025)
    pick = [cases[i] for i in rng.choice(len(cases), 72, replace=False)]
    return sorted(pick, key=lambda c: (c[0] == F64, c[1], c[2], c[4]))


ACCURACY = _grid()


@pytest.mark.parametrize("dtype,points,hop,frames,flags", ACCURACY,
                         ids=["%s-%d-h%d-x%d-f%d" % ("c32" if c[0] == F32 else "c64", *c[1:]) for c in ACCURACY])
def test_synthesis_accuracy(dtype, points, hop, frames, flags):
    X = rand_c(np.random.default_rng(points * 7919 + hop * 31 + flags), (frames, points), dtype)
    got, _ = run_ifft(X, hop, flags, dtype)
    w = library_window(kind_of(flags), points, dtype)
    ref = synthesis(X, hop, kind_of(flags), flags, acc.ref_ctype(dtype), w)
    peer = synthesis(X, hop, kind_of(flags), flags, acc.ctype(dtype), w)
    check_rows(got, ref, peer, dtype, "ifft frames %d h%d f%d" % (points, hop, flags), tol_n=points)


# ---- 2. round trip through bdsp_fft_frames_* ---------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,real,length,points,hop,kind,shift", [
    (F32, True, 1 << 20, 1024, 256, bd.HAMMING, 0),
    (F32, False, 1 << 22, 4096, 1024, bd.BLACKMAN_HARRIS, SH),
    (F64, False, 1 << 20, 2048, 512, bd.TRIANGULAR, SH),
], ids=["real-2^20-hamming-1024-h256", "c32-2^22-blackman-harris-4096-h1024-shift", "c64-2^20-triangular-2048-h512-shift"])
def test_round_trip(dtype, real, length, points, hop, kind, shift):
    rng = np.random.default_rng(length + points)
    x = rand_c(rng, length, dtype)
    if real:
        x = np.ascontiguousarray(x.real)
    fwd = shift | bd.F_WINDOW(kind) | (REAL if real else 0)
    inv = shift | bd.F_WINDOW(kind) | (RO if real else 0)
    got, _ = run_ifft(run_frames(x, points, hop, fwd, dtype), hop, inv, dtype)
    want = x[:got.size]
    assert got.size == (1 + (length - points) // hop - 1) * hop + points
    peer = synthesis(analysis(x, points, hop, kind, shift, acc.ctype(dtype)), hop, kind, shift | (RO if real else 0), acc.ctype(dtype))
    check_rows(got, want, peer, dtype, "fft frames > ifft frames %d h%d" % (points, hop), tol_n=points)


# ---- 3. frames that do not overlap are the inverse rows ----------------------------------------------------------------
@pytest.mark.parametrize("dtype,points,frames", [
    (F32, 1024, 64), (F32, 4096, 16), (F32, 16384, 4), (F32, 65536, 2), (F32, 3072, 128), (F32, 1000, 8), (F64, 1024, 16),
    (F64, 8192, 4), (F64, 1000, 4),
])
@pytest.mark.parametrize("real_out", [False, True])
def test_hop_equal_to_points_is_the_inverse_row_transform(dtype, points, frames, real_out):
    X = rand_c(np.random.default_rng(points + frames), (frames, points), dtype)
    flags = SH | (RO if real_out else 0)
    run_ifft(X, points, flags, dtype)   # cached chirp-z filters and kernel attributes are set up once
    run_rows(X, INV | SH, dtype)
    got, n_got = run_ifft(X, points, flags, dtype)
    want, n_want = run_rows(X, INV | SH, dtype)
    want = want.ravel()
    assert same_bytes(got, np.ascontiguousarray(want.real) if real_out else want)
    assert n_got == n_want + 1


# ---- 4. launches: the inverse rows, the window table, one overlap-add ----------------------------------------------------
@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F32, 1024, 256, 64, 0),
    (F32, 1024, 256, 64, SH | bd.F_WINDOW(1)),
    (F32, 4096, 1024, 16, RO | bd.F_WINDOW(2)),
    (F32, 16384, 4096, 4, SH | bd.F_WINDOW(0)),
    (F32, 1000, 250, 16, bd.F_WINDOW(1)),
    (F32, 256, 64, 64, bd.F_WINDOW(3)),   # rectangular: no table
    (F64, 2048, 512, 8, SH | RO | bd.F_WINDOW(1)),
])
def test_launch_count(dtype, points, hop, frames, flags):
    X = rand_c(np.random.default_rng(points + hop), (frames, points), dtype)
    rows_flags = INV | (flags & SH)
    run_ifft(X, hop, flags, dtype)
    run_rows(X, rows_flags, dtype)
    _, n_got = run_ifft(X, hop, flags, dtype)
    _, n_want = run_rows(X, rows_flags, dtype)
    table = 1 if kind_of(flags) in (0, 1, 2) else 0
    assert n_got == n_want + 1 + table


# ---- 5. bit-reproducible ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,flags", [(F32, SH | bd.F_WINDOW(1)), (F32, RO), (F64, bd.F_WINDOW(2))])
def test_repeated_calls_give_the_same_bytes(dtype, flags):
    points, hop = 1024, 128
    frames = 1 + ((1 << 22) - points) // hop
    X = rand_c(np.random.default_rng(11), (frames, points), dtype)
    first, _ = run_ifft(X, hop, flags, dtype)
    assert first.size >= 1 << 22
    for _ in range(2):
        again, _ = run_ifft(X, hop, flags, dtype)
        assert same_bytes(first, again)


# ---- 6. locality -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F32, 1024, 256, 64, SH | bd.F_WINDOW(1)),
    (F32, 1000, 333, 16, RO),
    (F64, 512, 512, 8, 0),
])
def test_a_frame_reaches_only_the_samples_it_covers(dtype, points, hop, frames, flags):
    X = rand_c(np.random.default_rng(points + frames), (frames, points), dtype)
    f = frames // 2
    X[f, points // 3] = np.nan
    got, _ = run_ifft(X, hop, flags, dtype)
    inside = np.zeros(got.size, dtype=bool)
    inside[f * hop:f * hop + points] = True
    assert np.all(np.isfinite(got[~inside]))
    assert np.all(np.isnan(got[inside]))


# ---- 7. contract -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, F64])
def test_bad_arguments_and_overlap_are_rejected(dtype):
    L = bd.lib()
    f = fn("bdsp_ifft_frames", dtype)
    esz = np.dtype(dtype).itemsize * 2
    x = Buf(rand_c(np.random.default_rng(1), 8192, dtype), 0, dtype)
    base = x.ptr
    out = base + 4096 * esz
    before = bd.kernel_launch_count()
    for flag, name in ((INV, b"BDSP_F_INVERSE"), (MAG, b"BDSP_F_MAGNITUDE"), (REAL, b"BDSP_F_REAL_INPUT"), (32, b"0x20"),
                       (1 << 12, b"0x1000")):
        assert f(base, out, 1024, 512, 4, SH | flag) == -2
        assert name in L.bdsp_last_error()
    assert f(base, out, 1024, 0, 4, 0) == -2
    assert b"hop" in L.bdsp_last_error()
    assert f(base, out, 1024, 1025, 4, 0) == -2
    assert b"no frame covers" in L.bdsp_last_error()
    assert f(base, out, 1 << 40, 1 << 40, 1 << 30, 0) == -2                          # frames * points overflows
    assert b"overflow" in L.bdsp_last_error()
    # input [0, 4096) points, output (3 * 512 + 1024 = 2560 points) starting inside, at or one point before its end
    assert f(base, base + 4095 * esz, 1024, 512, 4, 0) == -3
    assert f(base, base, 1024, 512, 4, 0) == -3
    assert f(base + 2559 * esz, base, 1024, 512, 4, 0) == -3                        # output [0, 2560) ends one point in
    assert f(base + 1279 * esz, base, 1024, 512, 4, RO) == -3                       # 2560 real scalars = 1280 points
    assert b"overlap" in L.bdsp_last_error()
    assert bd.kernel_launch_count() == before
    # adjacent ranges are fine
    assert f(base, base + 4096 * esz, 1024, 512, 4, 0) == 0
    assert f(base + 2560 * esz, base, 1024, 512, 4, 0) == 0
    assert f(base + 1280 * esz, base, 1024, 512, 4, RO) == 0
    bd.synchronize()


@pytest.mark.parametrize("dtype", [F32, F64])
def test_empty_calls_launch_nothing(dtype):
    f = fn("bdsp_ifft_frames", dtype)
    x = Buf(rand_c(np.random.default_rng(2), 1024, dtype), 0, dtype)
    out = Buf.empty(1024, True, 0, dtype)
    before = bd.kernel_launch_count()
    assert f(x.ptr, out.ptr, 1024, 256, 0, bd.F_WINDOW(1)) == 0
    assert f(x.ptr, out.ptr, 0, 256, 4, 0) == 0
    assert bd.kernel_launch_count() == before
