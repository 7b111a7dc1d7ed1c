"""bdsp_fft_frames_*: transforms of overlapping (or spaced) frames of one device signal.

The definition the tests hold the library to: row f of the result is byte for byte what bdsp_fft_rows_* writes for the
same points, frames and flags when the frames lie back to back (built here on the host with sliding_window_view).  On
top of that: accuracy of two realistic short-time transforms against a higher-precision reference, the number of kernel
launches (the fused path is one kernel, plus the window table), the error contract, and that no point outside the frames
is read."""
import itertools

import numpy as np
import pytest
from numpy.lib.stride_tricks import sliding_window_view

import basic_dsp_b200 as bd
from oracle import accuracy as acc
from oracle.accuracy import F_MAGNITUDE as MAG, F_REAL_INPUT as REAL, F_SHIFT as SH
from test_gpu_accuracy import F32, F64, Buf, check_rows, rand_c

pytestmark = pytest.mark.gpu


def fn(name, dtype):
    return getattr(bd.lib(), "%s_%s" % (name, "c32" if dtype == F32 else "c64"))


def signal(rng, length, dtype, real):
    x = rand_c(rng, length, dtype)
    return np.ascontiguousarray(x.real) if real else x


def n_frames(length, points, hop):
    return 1 + (length - points) // hop


def frames_of(x, points, hop, frames):
    return np.ascontiguousarray(sliding_window_view(x, points)[::hop][:frames])


def run_frames(x, points, hop, frames, flags, dtype, off=0):
    """bdsp_fft_frames_* over the device copy of x -> (result rows, kernel launches)"""
    xin = Buf(x, off, dtype)
    out = Buf.empty(frames * points, not flags & MAG, 0, dtype)
    before = bd.kernel_launch_count()
    rc = fn("bdsp_fft_frames", dtype)(xin.ptr, out.ptr, points, hop, frames, flags)
    launches = bd.kernel_launch_count() - before
    assert rc == 0, bd.lib().bdsp_last_error()
    return out.get((frames, points)), launches


def run_rows(rows, flags, dtype):
    """bdsp_fft_rows_* over the frames laid back to back -> (result rows, kernel launches)"""
    frames, points = rows.shape
    xin = Buf(rows, 0, dtype)
    out = Buf.empty(frames * points, not flags & MAG, 0, dtype)
    before = bd.kernel_launch_count()
    rc = fn("bdsp_fft_rows", dtype)(xin.ptr, out.ptr, points, frames, flags)
    launches = bd.kernel_launch_count() - before
    assert rc == 0, bd.lib().bdsp_last_error()
    return out.get((frames, points)), launches


def same_bytes(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def fused_frame_counts(points):
    """Frame counts inside the fused conditions (n * frames >= 2^16, whole groups of 4096 / n frames) and outside them."""
    inside = max(65536 // points, 1)
    return (inside, inside + 1, 3)


# ---- 1. byte identity with bdsp_fft_rows_* on the frames laid back to back ----------------------------------------------
POINTS = (64, 128, 512, 1024, 4096, 8192, 16384, 1000, 3072)
FLAGS = [s | r | w for s in (0, SH, MAG, SH | MAG) for r in (0, REAL) for w in [0] + [bd.F_WINDOW(k) for k in range(4)]]


def _grid():
    """A seeded subset: 64 cases of the fused route (c32, 64 .. 8192 points, the even hop points / 4, whole groups of
    frames) and 96 of everything else."""
    fused, other = [], []
    for dtype, points in itertools.product((F32, F64), POINTS):
        for hop in sorted({1, points // 4, points // 2 - 1, points - 1, points, points + 3}):
            for i, frames in enumerate(fused_frame_counts(points)):
                if hop == 1 and frames > 64:
                    continue   # a signal barely longer than one frame: kept to the small counts
                eligible = dtype == F32 and points & (points - 1) == 0 and points <= 8192 and hop == points // 4 and i == 0
                (fused if eligible else other).extend((dtype, points, hop, frames, flags) for flags in FLAGS)
    rng = np.random.default_rng(2024)
    pick = [fused[i] for i in rng.choice(len(fused), 64, replace=False)] + [other[i] for i in rng.choice(len(other), 96, replace=False)]
    return sorted(pick, key=lambda c: (c[0] == F64, c[1], c[2], c[3], c[4]))


IDENTITY = _grid()


@pytest.mark.parametrize("dtype,points,hop,frames,flags", IDENTITY,
                         ids=["%s-%d-h%d-x%d-f%d" % ("c32" if c[0] == F32 else "c64", *c[1:]) for c in IDENTITY])
def test_frames_match_rows_byte_for_byte(dtype, points, hop, frames, flags):
    rng = np.random.default_rng(points * 7919 + hop * 31 + frames * 3 + flags)
    x = signal(rng, (frames - 1) * hop + points, dtype, flags & REAL)
    got, _ = run_frames(x, points, hop, frames, flags, dtype)
    want, _ = run_rows(frames_of(x, points, hop, frames), flags, dtype)
    assert same_bytes(got, want)


# shapes of the frame pass whose gathered rows take each multi-kernel route (test_fft_frames_route.py NESTED), and fused
# shapes at every packed length: (dtype, points, hop, frames, flags, launches beyond the rows' own)
NESTED = [
    (F32, 16384, 4096, 4, bd.F_WINDOW(1), 1),              # frame pass > mul-pass > packed-16k
    (F32, 16384, 4096, 4, REAL | MAG | bd.F_WINDOW(2), 1),  # frame pass > mul-pass > real-rows
    (F32, 3072, 1536, 128, SH, 1),                         # frame pass > q-rows-interleave > packed
    (F32, 3072, 1536, 4, MAG, 1),                          # frame pass > q-rows
    (F32, 1000, 250, 16, bd.F_WINDOW(0), 1),                # frame pass > bluestein
    (F64, 1000, 250, 16, SH | REAL, 1),                    # frame pass > bluestein
    (F64, 1024, 255, 16, bd.F_WINDOW(1), 1),                # frame pass > c64-rows
    (F32, 1024, 511, 64, bd.F_WINDOW(1), 1),                # frame pass > mul-pass > packed
    (F32, 1024, 512, 65, 0, 1),                            # frame pass > block
    (F32, 64, 32, 1024, SH | MAG, 0),                      # packed frames
    (F32, 8192, 2050, 8, REAL | bd.F_WINDOW(2), -1),        # packed frames: window on the first load, no multiplier pass
]


@pytest.mark.parametrize("dtype,points,hop,frames,flags,extra", NESTED, ids=["%d-%d-h%d-x%d" % (i, c[1], c[2], c[3]) for i, c in enumerate(NESTED)])
def test_nested_routes_match_rows(dtype, points, hop, frames, flags, extra):
    rng = np.random.default_rng(points + hop + frames)
    x = signal(rng, (frames - 1) * hop + points, dtype, flags & REAL)
    rows = frames_of(x, points, hop, frames)
    run_frames(x, points, hop, frames, flags, dtype)   # cached chirp-z filters and kernel attributes are set up once
    run_rows(rows, flags, dtype)
    got, n_got = run_frames(x, points, hop, frames, flags, dtype)
    want, n_want = run_rows(rows, flags, dtype)
    assert same_bytes(got, want)
    assert n_got == n_want + extra, (n_got, n_want)


# ---- 2. accuracy against a higher-precision reference ------------------------------------------------------------------
def windowed_frames_transform(rows, kind, flags, ct):
    rt = np.finfo(ct).dtype.type
    w = acc.window(kind, rows.shape[-1], rt)
    xw = rows.astype(rt) * w if flags & REAL else rows.astype(ct) * w
    return acc.transform(xw, flags, ct)


@pytest.mark.parametrize("real,length,points,hop,kind,flags", [
    (True, 1 << 20, 1024, 256, bd.HAMMING, REAL | MAG),
    (False, 1 << 22, 4096, 1024, bd.BLACKMAN_HARRIS, SH),
], ids=["real-2^20-hamming-1024-h256-mag", "c32-2^22-blackman-harris-4096-h1024-shift"])
def test_stft_accuracy(real, length, points, hop, kind, flags):
    rng = np.random.default_rng(length + points)
    x = signal(rng, length, F32, real)
    frames = n_frames(length, points, hop)
    got, _ = run_frames(x, points, hop, frames, flags | bd.F_WINDOW(kind), F32)
    rows = frames_of(x, points, hop, frames)
    ref = windowed_frames_transform(rows, kind, flags, acc.ref_ctype(F32))
    peer = windowed_frames_transform(rows, kind, flags, acc.ctype(F32))
    check_rows(got, ref, peer, F32, "fft frames %d h%d f%d" % (points, hop, flags))


# ---- 3. the fused path is taken ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("points,hop,frames,flags,launches", [
    (1024, 256, 64, 0, 1),
    (1024, 256, 64, REAL | MAG, 1),
    (1024, 256, 64, REAL | MAG | bd.F_WINDOW(1), 2),
    (4096, 2048, 16, SH | MAG | bd.F_WINDOW(2), 2),
    (8192, 4096, 8, bd.F_WINDOW(0), 2),
    (256, 130, 256, SH, 1),
])
def test_eligible_shape_is_one_kernel(points, hop, frames, flags, launches):
    rng = np.random.default_rng(points + hop)
    x = signal(rng, (frames - 1) * hop + points, F32, flags & REAL)
    run_frames(x, points, hop, frames, flags, F32)
    _, n = run_frames(x, points, hop, frames, flags, F32)
    assert n == launches


@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F32, 1024, 255, 64, 0),
    (F32, 1024, 256, 63, REAL | bd.F_WINDOW(1)),
    (F32, 16384, 8192, 4, SH),
    (F64, 1024, 256, 64, MAG),
    (F32, 1000, 500, 80, bd.F_WINDOW(2)),
])
def test_frame_pass_is_one_kernel_more(dtype, points, hop, frames, flags):
    rng = np.random.default_rng(points + hop + 1)
    x = signal(rng, (frames - 1) * hop + points, dtype, flags & REAL)
    rows = frames_of(x, points, hop, frames)
    run_frames(x, points, hop, frames, flags, dtype)
    run_rows(rows, flags, dtype)
    got, n_got = run_frames(x, points, hop, frames, flags, dtype)
    want, n_want = run_rows(rows, flags, dtype)
    assert same_bytes(got, want)
    assert n_got == n_want + 1


# ---- 4. contract -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, F64])
def test_inverse_hop_zero_and_overlap_are_rejected(dtype):
    L = bd.lib()
    f = fn("bdsp_fft_frames", dtype)
    x = Buf(rand_c(np.random.default_rng(1), 4096, dtype), 0, dtype)
    out = Buf.empty(4096, True, 0, dtype)
    before = bd.kernel_launch_count()
    assert f(x.ptr, out.ptr, 1024, 512, 4, bd.F_INVERSE) == -2
    assert b"INVERSE" in L.bdsp_last_error()
    assert f(x.ptr, out.ptr, 1024, 0, 4, 0) == -2
    assert b"hop" in L.bdsp_last_error()
    assert f(x.ptr, out.ptr, 1 << 40, 1 << 40, 1 << 30, 0) == -2                   # (frames - 1) * hop overflows
    esz = np.dtype(dtype).itemsize * 2
    # the input range is (4 - 1) * 512 + 1024 = 2560 points: outputs that start inside it, at it, or end one point into it
    assert f(x.ptr, x.ptr + 2559 * esz, 1024, 512, 4, 0) == -3
    assert f(x.ptr, x.ptr, 1024, 512, 4, 0) == -3
    assert f(x.ptr + 1023 * esz, x.ptr, 256, 512, 4, 0) == -3                       # output [0, 1024), input from 1023
    assert b"overlap" in L.bdsp_last_error()
    assert bd.kernel_launch_count() == before
    # adjacent ranges are fine: the output ends where the input starts, or starts where the input range [0, 1792) ends
    assert f(x.ptr + 1024 * esz, x.ptr, 256, 512, 4, 0) == 0
    assert f(x.ptr, x.ptr + 1792 * esz, 256, 512, 4, 0) == 0
    bd.synchronize()


@pytest.mark.parametrize("dtype", [F32, F64])
def test_empty_calls_launch_nothing(dtype):
    f = fn("bdsp_fft_frames", dtype)
    x = Buf(rand_c(np.random.default_rng(2), 1024, dtype), 0, dtype)
    out = Buf.empty(1024, True, 0, dtype)
    before = bd.kernel_launch_count()
    assert f(x.ptr, out.ptr, 1024, 256, 0, bd.F_WINDOW(1)) == 0
    assert f(x.ptr, out.ptr, 0, 256, 4, 0) == 0
    assert bd.kernel_launch_count() == before


@pytest.mark.parametrize("dtype,points,frames,flags", [
    (F32, 1024, 64, 0), (F32, 1024, 64, REAL | MAG | bd.F_WINDOW(1)), (F32, 4096, 16, SH | bd.F_WINDOW(2)),
    (F32, 16384, 4, SH), (F32, 3072, 128, 0), (F64, 1024, 16, SH | MAG), (F32, 1000, 8, bd.F_WINDOW(0)),
])
def test_hop_equal_to_points_is_the_row_transform(dtype, points, frames, flags):
    rng = np.random.default_rng(points + frames)
    x = signal(rng, points * frames, dtype, flags & REAL)
    run_frames(x, points, points, frames, flags, dtype)
    run_rows(x.reshape(frames, points), flags, dtype)
    got, n_got = run_frames(x, points, points, frames, flags, dtype)
    want, n_want = run_rows(x.reshape(frames, points), flags, dtype)
    assert same_bytes(got, want)
    assert n_got == n_want


@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F32, 1024, 256, 64, REAL | MAG | bd.F_WINDOW(1)),     # packed frames
    (F32, 1024, 1030, 64, SH | bd.F_WINDOW(2)),            # packed frames, gaps between the frames
    (F32, 1024, 1027, 64, SH),                             # frame pass, gaps between the frames
    (F32, 16384, 16387, 4, MAG),                           # frame pass > packed-16k
    (F64, 512, 515, 8, REAL),                              # frame pass, c64
])
def test_no_point_outside_the_frames_is_read(dtype, points, hop, frames, flags):
    """NaN in every skipped sample and right after the last frame: the result stays finite and equals the plain rows'."""
    rng = np.random.default_rng(points + hop + frames + 7)
    length = (frames - 1) * hop + points
    x = signal(rng, length + 64, dtype, flags & REAL)
    inside = np.zeros(x.size, dtype=bool)
    for f in range(frames):
        inside[f * hop:f * hop + points] = True
    x[~inside] = np.nan
    got, _ = run_frames(x, points, hop, frames, flags, dtype)
    want, _ = run_rows(frames_of(x, points, hop, frames), flags, dtype)
    assert np.all(np.isfinite(got))
    assert same_bytes(got, want)
