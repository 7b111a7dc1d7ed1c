"""bdsp_welch_*: Welch's averaged periodogram of a device signal.

The definition the tests hold the library to is test_welch_reference.closed_form (pinned to scipy.signal.welch without a
GPU), with the library's own window table.  On top of accuracy against a higher-precision reference: the route taken
(counted in kernel launches: the fused kernel covers incomplete groups of frames, the general path runs per chunk of
frames), exact scaling, bit-reproducible results, that nothing outside the output is written, the error contract, and a
workspace that stays bounded whatever the frame count."""
import itertools

import numpy as np
import pytest

import basic_dsp_b200 as bd
from oracle import accuracy as acc
from oracle.accuracy import F_REAL_INPUT as REAL, F_SHIFT as SH
from test_gpu_accuracy import F32, F64, Buf, check_rows, rand_c
from test_welch_reference import closed_form

pytestmark = pytest.mark.gpu

ONE, PSD = bd.F_ONESIDED, bd.F_POWER_SPECTRUM
PAD = 64                  # sentinel values before and after every output
CHUNK_POINTS = 1 << 24    # spectrum points per chunk of the general path (fft.cu welch_exec)
FS = 48000.0


def fn(name, dtype):
    return getattr(bd.lib(), "%s_%s" % (name, "c32" if dtype == F32 else "c64"))


def signal(rng, length, dtype, real):
    x = rand_c(rng, length, dtype)
    return np.ascontiguousarray(x.real) if real else x


def n_out(points, flags):
    return points // 2 + 1 if flags & ONE else points


def run_welch(x, points, hop, frames, flags, dtype, fs=FS, off=0):
    """bdsp_welch_* over the device copy of x (`off` elements past an aligned start) -> (output, kernel launches); checks
    that the PAD values on either side of the output keep their sentinel."""
    xin = Buf(x, off, dtype)
    sentinel = np.full(n_out(points, flags) + 2 * PAD, 1234.5, dtype=dtype)
    out = Buf(sentinel, 0, dtype)
    before = bd.kernel_launch_count()
    rc = fn("bdsp_welch", dtype)(xin.ptr, out.ptr + PAD * out.esize, points, hop, frames, flags, fs)
    launches = bd.kernel_launch_count() - before
    assert rc == 0, bd.lib().bdsp_last_error()
    got = out.get(sentinel.shape)
    assert np.array_equal(got[:PAD], sentinel[:PAD]) and np.array_equal(got[-PAD:], sentinel[-PAD:]), "write outside the output"
    return got[PAD:-PAD], launches


def kind_of(flags):
    wk = (flags >> 8) & 15
    return wk - 1 if wk else None


def library_window(kind, points, dtype):
    """The built-in window as the library evaluates it in `dtype` (the table of window_table_kernel), None without one."""
    if kind not in (bd.TRIANGULAR, bd.HAMMING, bd.BLACKMAN_HARRIS):
        return None
    return bd.DspVec(np.ones(points, dtype=dtype), is_complex=False, dtype=dtype).apply_window(kind).to_numpy()


def per_group(points):
    return 4096 // points if points < 4096 and points & (points - 1) == 0 else 1


def same_bytes(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


# ---- 1. accuracy against a higher-precision reference ------------------------------------------------------------------
POINTS = (64, 256, 1024, 4096, 8192, 16384, 1000, 3072)
FLAGS = [0, REAL, REAL | ONE, SH, PSD, REAL | PSD | ONE] + [REAL | bd.F_WINDOW(k) for k in range(4)] + [SH | bd.F_WINDOW(1)]


def _grid():
    """A seeded subset of precision x points x hop x flags x frame count (whole groups of 4096 / points frames, and one
    frame more or fewer); about 2^17 spectrum points per case."""
    cases = []
    for dtype, points in itertools.product((F32, F64), POINTS):
        per = per_group(points)
        whole = max(per, (1 << 17) // points // per * per)
        for hop in sorted({points // 4, points // 2 - 1, points, points + 2}):
            for frames in (whole, whole + 1, whole - 1):
                cases.extend((dtype, points, hop, frames, flags) for flags in FLAGS)
    rng = np.random.default_rng(2026)
    pick = [cases[i] for i in rng.choice(len(cases), 96, replace=False)]
    return sorted(pick, key=lambda c: (c[0] == F64, c[1], c[2], c[3], c[4]))


ACCURACY = _grid()


@pytest.mark.parametrize("dtype,points,hop,frames,flags", ACCURACY,
                         ids=["%s-%d-h%d-x%d-f%d" % ("c32" if c[0] == F32 else "c64", *c[1:]) for c in ACCURACY])
def test_welch_accuracy(dtype, points, hop, frames, flags):
    rng = np.random.default_rng(points * 7919 + hop * 31 + frames * 3 + flags)
    x = signal(rng, (frames - 1) * hop + points, dtype, flags & REAL)
    got, _ = run_welch(x, points, hop, frames, flags, dtype)
    w = library_window(kind_of(flags), points, dtype)
    ref = closed_form(x, points, hop, w, flags, FS, acc.ref_ctype(dtype))
    peer = closed_form(x, points, hop, w, flags, FS, acc.ctype(dtype))
    check_rows(got, ref, peer, dtype, "welch %d h%d x%d f%d" % (points, hop, frames, flags), tol_n=points)


def test_misaligned_input_takes_the_general_path_and_agrees():
    """c32 frames one point past an aligned start: the general path (the same closed form, other kernels)."""
    rng = np.random.default_rng(9)
    points, hop, frames = 1024, 256, 61
    x = signal(rng, (frames - 1) * hop + points, F32, True)
    got, _ = run_welch(x, points, hop, frames, REAL | ONE | bd.F_WINDOW(1), F32, off=1)
    w = library_window(1, points, F32)
    ref = closed_form(x, points, hop, w, REAL | ONE, FS, acc.ref_ctype(F32))
    peer = closed_form(x, points, hop, w, REAL | ONE, FS, acc.ctype(F32))
    check_rows(got, ref, peer, F32, "welch misaligned", tol_n=points)


# Groups of 4096 / points frames several times the fused grid (592 CTAs, 296 for 8192 points): every CTA adds later rows
# into its partial row, and the float32 partials are summed over several rows each; some with an incomplete last group.
MANY_ROWS = [
    (64, 16, 1 << 17, REAL | ONE),                                # 2048 groups: 3-4 rows per CTA
    (64, 34, (1 << 17) + 5, SH | bd.F_WINDOW(2)),                 # complex; the last group holds 5 of 64 frames
    (1024, 256, 4 * 592 * 4 + 1, REAL | ONE | bd.F_WINDOW(1)),    # 2369 groups, the last one with one frame
    (1024, 512, 4 * 592 * 4 + 3, PSD),                            # complex
    (8192, 4096, 296 * 3 + 1, REAL | bd.F_WINDOW(0)),             # 889 rows over 296 CTAs
]


@pytest.mark.parametrize("points,hop,frames,flags", MANY_ROWS, ids=["%d-h%d-x%d-f%d" % c for c in MANY_ROWS])
def test_fused_accuracy_with_many_rows_per_cta(points, hop, frames, flags):
    rng = np.random.default_rng(points + hop + frames)
    x = signal(rng, (frames - 1) * hop + points, F32, flags & REAL)
    got, launches = run_welch(x, points, hop, frames, flags, F32)
    assert launches == 2 + (2 if kind_of(flags) in (0, 1, 2) else 0)   # the fused route
    w = library_window(kind_of(flags), points, F32)
    ref = closed_form(x, points, hop, w, flags, FS, acc.ref_ctype(F32))
    peer = closed_form(x, points, hop, w, flags, FS, acc.ctype(F32))
    check_rows(got, ref, peer, F32, "welch fused %d h%d x%d f%d" % (points, hop, frames, flags), tol_n=points)


# ---- 2. the route taken, by kernel launches ----------------------------------------------------------------------------
@pytest.mark.parametrize("points,hop,frames,flags,launches", [
    (1024, 256, 64, REAL | bd.F_WINDOW(1), 4),      # window table + window sums + fused + final
    (1024, 256, 65, REAL | ONE, 2),                 # incomplete last group: still fused + final
    (1024, 256, 1 + ((1 << 22) - 1024) // 256, REAL | ONE | bd.F_WINDOW(1), 4),
    (64, 34, 1000, SH | bd.F_WINDOW(2), 4),
    (8192, 4096, 3, PSD, 2),
    (256, 130, 4097, bd.F_WINDOW(3), 2),            # rectangular: no table
])
def test_fused_call_is_table_kernel_and_final(points, hop, frames, flags, launches):
    x = signal(np.random.default_rng(points + hop), (frames - 1) * hop + points, F32, flags & REAL)
    run_welch(x, points, hop, frames, flags, F32)
    _, n = run_welch(x, points, hop, frames, flags, F32)
    assert n == launches


def frames_launches(x, points, hop, frames, flags, dtype):
    """Kernel launches of bdsp_fft_frames_* over the same frames, with the window table the general path builds once."""
    xin = Buf(x, 0, dtype)
    out = Buf.empty(frames * points, True, 0, dtype)
    f = fn("bdsp_fft_frames", dtype)
    assert f(xin.ptr, out.ptr, points, hop, frames, flags) == 0, bd.lib().bdsp_last_error()
    before = bd.kernel_launch_count()
    assert f(xin.ptr, out.ptr, points, hop, frames, flags) == 0, bd.lib().bdsp_last_error()
    return bd.kernel_launch_count() - before - (1 if kind_of(flags) in (0, 1, 2) else 0)


@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F64, 1024, 256, 64, REAL | bd.F_WINDOW(1)),
    (F64, 4096, 1024, 20, SH),
    (F32, 1024, 255, 64, REAL | ONE | bd.F_WINDOW(2)),   # odd hop
    (F32, 1000, 250, 40, bd.F_WINDOW(0)),
    (F32, 32, 8, 100, REAL),
    (F32, 16384, 4096, 2100, REAL | bd.F_WINDOW(1)),     # three chunks of 1024, 1024 and 52 frames
])
def test_general_path_runs_per_chunk(dtype, points, hop, frames, flags):
    x = signal(np.random.default_rng(points + hop + 1), (frames - 1) * hop + points, dtype, flags & REAL)
    chunk = max(1, min(CHUNK_POINTS // points, frames))
    sizes = [min(chunk, frames - f0) for f0 in range(0, frames, chunk)]
    rows_flags = flags & (REAL | 0xf00)
    per_chunk = sum(frames_launches(x, points, hop, cf, rows_flags, dtype) for cf in sizes)
    table = 2 if kind_of(flags) in (0, 1, 2) else 0      # window table + window sums
    run_welch(x, points, hop, frames, flags, dtype)
    _, n = run_welch(x, points, hop, frames, flags, dtype)
    assert n == table + per_chunk + len(sizes) + 1       # + one accumulate kernel per chunk, + the final kernel


# ---- 3. exact scaling, reproducibility ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F32, 1024, 256, 1021, REAL | ONE | bd.F_WINDOW(1)),   # fused, incomplete last group
    (F32, 512, 127, 300, SH | bd.F_WINDOW(2)),            # general
    (F64, 2048, 512, 100, REAL | PSD),                    # general
])
def test_scaling_by_a_power_of_two_is_exact(dtype, points, hop, frames, flags):
    x = signal(np.random.default_rng(points + frames), (frames - 1) * hop + points, dtype, flags & REAL)
    base, _ = run_welch(x, points, hop, frames, flags, dtype)
    for k in ((10, -10) if dtype == F32 else (100, -100)):
        got, _ = run_welch((x * dtype(2.0) ** k).astype(x.dtype), points, hop, frames, flags, dtype)
        want = base * dtype(4.0) ** k
        assert same_bytes(got, want), k


@pytest.mark.parametrize("dtype,flags", [(F32, REAL | ONE | bd.F_WINDOW(1)), (F32, SH), (F64, REAL | bd.F_WINDOW(2))])
def test_repeated_calls_give_the_same_bytes(dtype, flags):
    points, hop = 1024, 256
    frames = 1 + ((1 << 22) - points) // hop
    x = signal(np.random.default_rng(11), (frames - 1) * hop + points, dtype, flags & REAL)
    first, _ = run_welch(x, points, hop, frames, flags, dtype)
    for _ in range(2):
        again, _ = run_welch(x, points, hop, frames, flags, dtype)
        assert same_bytes(first, again)


# ---- 4. contract -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, F64])
def test_bad_arguments_and_overlap_are_rejected(dtype):
    L = bd.lib()
    f = fn("bdsp_welch", dtype)
    esz = np.dtype(dtype).itemsize
    x = Buf(rand_c(np.random.default_rng(1), 8192, dtype), 0, dtype)
    base = x.ptr
    out = base + 2 * 4096 * esz
    before = bd.kernel_launch_count()
    for flag, name in ((bd.F_INVERSE, b"BDSP_F_INVERSE"), (bd.F_MAGNITUDE, b"BDSP_F_MAGNITUDE"), (bd.F_REAL_OUTPUT, b"BDSP_F_REAL_OUTPUT"),
                       (128, b"0x80"), (1 << 12, b"0x1000")):
        assert f(base, out, 1024, 512, 4, REAL | flag, FS) == -2
        assert name in L.bdsp_last_error()
    assert f(base, out, 1024, 512, 4, ONE, FS) == -2                        # one-sided needs real input
    assert b"ONESIDED" in L.bdsp_last_error()
    assert f(base, out, 1024, 512, 4, REAL | ONE | SH, FS) == -2
    assert b"ONESIDED" in L.bdsp_last_error()
    assert f(base, out, 1024, 0, 4, 0, FS) == -2
    assert b"hop" in L.bdsp_last_error()
    for fs in (0.0, -1.0, float("nan"), float("inf")):
        assert f(base, out, 1024, 512, 4, REAL, fs) == -2
        assert b"fs" in L.bdsp_last_error()
    assert f(base, out, 1 << 40, 1 << 40, 1 << 30, 0, FS) == -2            # (frames - 1) * hop overflows
    assert b"overflow" in L.bdsp_last_error()
    # complex input [0, 2560) points = 5120 scalars; real input [0, 2560) scalars; outputs of 1024 or 513 scalars
    assert f(base, base + 5119 * esz, 1024, 512, 4, 0, FS) == -3
    assert f(base, base, 1024, 512, 4, 0, FS) == -3
    assert f(base + 1023 * esz, base, 1024, 512, 4, 0, FS) == -3           # output [0, 1024) scalars ends one into the input
    assert f(base + 512 * esz, base, 1024, 512, 4, REAL | ONE, FS) == -3   # 513 scalars
    assert b"overlap" in L.bdsp_last_error()
    assert bd.kernel_launch_count() == before
    # adjacent ranges are fine; fs is ignored for a power spectrum
    assert f(base, base + 5120 * esz, 1024, 512, 4, 0, FS) == 0
    assert f(base + 1024 * esz, base, 1024, 512, 4, 0, FS) == 0
    assert f(base + 513 * esz, base, 1024, 512, 4, REAL | ONE, FS) == 0
    assert f(base, out, 1024, 512, 4, REAL | PSD, float("nan")) == 0
    bd.synchronize()


@pytest.mark.parametrize("dtype", [F32, F64])
def test_empty_calls_launch_nothing_and_leave_the_output(dtype):
    f = fn("bdsp_welch", dtype)
    x = Buf(rand_c(np.random.default_rng(2), 1024, dtype), 0, dtype)
    sentinel = np.full(1024, 7.5, dtype=dtype)
    out = Buf(sentinel, 0, dtype)
    before = bd.kernel_launch_count()
    assert f(x.ptr, out.ptr, 1024, 256, 0, bd.F_WINDOW(1), FS) == 0
    assert f(x.ptr, out.ptr, 0, 256, 4, 0, FS) == 0
    assert bd.kernel_launch_count() == before
    assert np.array_equal(out.get(sentinel.shape), sentinel)


# ---- 5. bounded workspace ----------------------------------------------------------------------------------------------
def test_workspace_stays_bounded_past_16_gib_of_spectra():
    """c64, 2^18 + 1 frames of 4096 points 64 apart: the frame spectra would take 16 GiB + 64 KiB.  The call runs in chunks
    of 2^24 spectrum points (256 MiB); its workspace grows by less than 2 GiB."""
    torch = pytest.importorskip("torch")
    points, hop, frames = 4096, 64, (1 << 18) + 1
    assert frames * points * 16 > 16 << 30
    flags = REAL | ONE | bd.F_WINDOW(1)
    x = np.random.default_rng(12).uniform(-1, 1, (frames - 1) * hop + points)
    xin = Buf(x, 0, F64)
    out = Buf.empty(points // 2 + 1, False, 0, F64)
    bd.synchronize()
    free_before = bd.lib().bdsp_mem_free()
    assert fn("bdsp_welch", F64)(xin.ptr, out.ptr, points, hop, frames, flags, FS) == 0, bd.lib().bdsp_last_error()
    bd.synchronize()
    assert free_before - bd.lib().bdsp_mem_free() < 2 << 30
    got = out.get(points // 2 + 1)
    # reference: the same closed form on the GPU with torch, in float64, the library's window table
    w = torch.from_numpy(library_window(1, points, F64)).cuda()
    xt = torch.from_numpy(x).cuda()
    acc_p = torch.zeros(points // 2 + 1, dtype=torch.float64, device="cuda")
    for f0 in range(0, frames, 1 << 15):
        seg = xt[f0 * hop:].unfold(0, points, hop)[:min(1 << 15, frames - f0)]
        acc_p += (torch.fft.rfft(seg * w).abs() ** 2).sum(0)
    want = (acc_p / (frames * FS * (w * w).sum())).cpu().numpy()
    want[1:points // 2] *= 2
    assert np.max(np.abs(got - want)) <= 1e-11 * np.max(np.abs(want))
