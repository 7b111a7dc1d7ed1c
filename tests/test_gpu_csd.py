"""bdsp_csd_* and bdsp_coherence_*: cross-spectral density and coherence of two device signals.

The definition the tests hold the library to is test_csd_reference.closed_form (pinned to scipy.signal.csd and
scipy.signal.coherence without a GPU), with the library's own window table.  On top of accuracy against a higher-precision
reference: exact identities that follow from every cross product being rounded on its own, agreement with bdsp_welch_*,
zero power, the route taken (counted in kernel launches, per chunk of frames), bit-reproducible results, that nothing
outside the output is written, the error contract, and a workspace that stays bounded whatever the frame count."""
import itertools

import numpy as np
import pytest

import basic_dsp_b200 as bd
from oracle import accuracy as acc
from oracle.accuracy import F_REAL_INPUT as REAL, F_SHIFT as SH
from test_csd_reference import closed_form
from test_gpu_accuracy import F32, F64, Buf, check_rows, rand_c
from test_gpu_welch import fn, kind_of, library_window, per_group, run_welch, same_bytes
from test_welch_reference import closed_form as welch_closed_form

pytestmark = pytest.mark.gpu

ONE, PSD = bd.F_ONESIDED, bd.F_POWER_SPECTRUM
PAD = 64                  # sentinel values before and after every output
CHUNK_POINTS = 1 << 24    # spectrum points per signal and chunk (fft_route.h CSD_CHUNK_POINTS)
FS = 48000.0


def pair(rng, length, dtype, real):
    """x and y = x through a short filter plus independent noise: coherence spread over (0, 1)"""
    x, e = rand_c(rng, length, dtype), rand_c(rng, length, dtype)
    if real:
        x, e = np.ascontiguousarray(x.real), np.ascontiguousarray(e.real)
    y = (np.convolve(x, [0.5, 1.0, -0.25, 0.125], mode="same") + 0.7 * e).astype(x.dtype)
    return x, y


def n_out(points, flags):
    return points // 2 + 1 if flags & ONE else points


def run_csd(x, y, points, hop, frames, flags, dtype, coherence=False, fs=FS, same=False):
    """bdsp_csd_* or bdsp_coherence_* over device copies of x and y (same: y is x's buffer) -> (output, kernel launches);
    checks that the PAD values on either side of the output keep their sentinel."""
    xin = Buf(x, 0, dtype)
    yin = xin if same else Buf(y, 0, dtype)
    cplx = not coherence
    count = n_out(points, flags) + 2 * PAD
    sentinel = np.full(count, 1234.5 + 17j if cplx else 1234.5, dtype=acc.ctype(dtype) if cplx else dtype)
    out = Buf(sentinel, 0, dtype)
    before = bd.kernel_launch_count()
    if coherence:
        rc = fn("bdsp_coherence", dtype)(xin.ptr, yin.ptr, out.ptr + PAD * out.esize, points, hop, frames, flags)
    else:
        rc = fn("bdsp_csd", dtype)(xin.ptr, yin.ptr, out.ptr + PAD * out.esize, points, hop, frames, flags, fs)
    launches = bd.kernel_launch_count() - before
    assert rc == 0, bd.lib().bdsp_last_error()
    got = out.get(sentinel.shape)
    assert same_bytes(got[:PAD], sentinel[:PAD]) and same_bytes(got[-PAD:], sentinel[-PAD:]), "write outside the output"
    return got[PAD:-PAD], launches


# ---- 1. accuracy against a higher-precision reference ------------------------------------------------------------------
POINTS = (64, 256, 1024, 4096, 8192, 16384, 1000, 3072)
FLAGS = [0, REAL, REAL | ONE, SH, PSD, REAL | PSD | ONE] + [REAL | bd.F_WINDOW(k) for k in range(4)] + [SH | bd.F_WINDOW(1),
                                                                                                        REAL | ONE | bd.F_WINDOW(1)]


def _grid(seed, coherence):
    """A seeded subset of precision x points x hop x flags x frame count (whole groups of 4096 / points frames, and one
    frame more or fewer); about 2^17 spectrum points per case."""
    cases = []
    flags_set = sorted({f & ~PSD for f in FLAGS}) if coherence else FLAGS
    for dtype, points in itertools.product((F32, F64), POINTS):
        per = per_group(points)
        whole = max(per, (1 << 17) // points // per * per)
        for hop in sorted({points // 4, points // 2 - 1, points, points + 2}):
            for frames in (whole, whole + 1, whole - 1):
                cases.extend((dtype, points, hop, frames, flags) for flags in flags_set)
    rng = np.random.default_rng(seed)
    pick = [cases[i] for i in rng.choice(len(cases), 64, replace=False)]
    return sorted(pick, key=lambda c: (c[0] == F64, c[1], c[2], c[3], c[4]))


def _ids(cases):
    return ["%s-%d-h%d-x%d-f%d" % ("c32" if c[0] == F32 else "c64", *c[1:]) for c in cases]


CSD_ACCURACY, COH_ACCURACY = _grid(2027, False), _grid(2028, True)


def check_against_reference(dtype, points, hop, frames, flags, coherence):
    rng = np.random.default_rng(points * 7919 + hop * 31 + frames * 3 + flags + coherence)
    x, y = pair(rng, (frames - 1) * hop + points, dtype, flags & REAL)
    got, _ = run_csd(x, y, points, hop, frames, flags, dtype, coherence)
    w = library_window(kind_of(flags), points, dtype)
    ref = closed_form(x, y, points, hop, w, flags, FS, acc.ref_ctype(dtype), coherence)
    peer = closed_form(x, y, points, hop, w, flags, FS, acc.ctype(dtype), coherence)
    check_rows(got, ref, peer, dtype, "%s %d h%d x%d f%d" % ("coherence" if coherence else "csd", points, hop, frames, flags), tol_n=points)
    return got


@pytest.mark.parametrize("dtype,points,hop,frames,flags", CSD_ACCURACY, ids=_ids(CSD_ACCURACY))
def test_csd_accuracy(dtype, points, hop, frames, flags):
    check_against_reference(dtype, points, hop, frames, flags, False)


@pytest.mark.parametrize("dtype,points,hop,frames,flags", COH_ACCURACY, ids=_ids(COH_ACCURACY))
def test_coherence_accuracy(dtype, points, hop, frames, flags):
    got = check_against_reference(dtype, points, hop, frames, flags, True)
    assert np.all((got >= 0) & (got <= 1 + 1e-5))


@pytest.mark.parametrize("coherence", [False, True])
@pytest.mark.parametrize("dtype,points,hop,flags", [(F32, 1024, 256, REAL | ONE | bd.F_WINDOW(1)), (F64, 4096, 1024, SH | bd.F_WINDOW(0))])
def test_accuracy_over_several_chunks(dtype, points, hop, flags, coherence):
    """frame counts past two whole chunks: the partial rows carry the sums of earlier chunks"""
    per = per_group(points) if dtype == F32 else 1
    frames = 2 * (CHUNK_POINTS // points // per * per) + 3
    check_against_reference(dtype, points, hop, frames, flags, coherence)


# ---- 2. exact identities -----------------------------------------------------------------------------------------------
IDENTITY = [
    (F32, 1024, 256, 1021, REAL | ONE | bd.F_WINDOW(1)),   # packed frames route, incomplete last group
    (F32, 512, 127, 300, SH | bd.F_WINDOW(2)),            # odd hop: frame pass
    (F32, 1000, 250, 200, REAL),                          # not a power of two
    (F64, 2048, 512, 100, REAL | PSD),
    (F64, 256, 64, 70000, bd.F_WINDOW(0)),                # two chunks, of 65536 and 4464 frames
]


@pytest.mark.parametrize("dtype,points,hop,frames,flags", IDENTITY, ids=_ids(IDENTITY))
def test_cross_spectrum_identities_are_exact(dtype, points, hop, frames, flags):
    rng = np.random.default_rng(points + frames)
    x, y = pair(rng, (frames - 1) * hop + points, dtype, flags & REAL)
    cflags = flags & ~PSD
    # csd(x, x) is real, coherence(x, x) is 1 in every bin (all have power here)
    sxx, _ = run_csd(x, None, points, hop, frames, flags, dtype, same=True)
    assert np.all(sxx.imag == 0)
    cxx, _ = run_csd(x, None, points, hop, frames, cflags, dtype, coherence=True, same=True)
    assert np.all(cxx == 1.0)
    # swapping x and y conjugates csd and keeps coherence (both buffers aligned alike: the same transform routes)
    sxy, _ = run_csd(x, y, points, hop, frames, flags, dtype)
    syx, _ = run_csd(y, x, points, hop, frames, flags, dtype)
    assert same_bytes(syx.real, sxy.real) and same_bytes(syx.imag, -sxy.imag + 0.0)   # a zero imaginary part is +0 both ways
    cxy, _ = run_csd(x, y, points, hop, frames, cflags, dtype, coherence=True)
    cyx, _ = run_csd(y, x, points, hop, frames, cflags, dtype, coherence=True)
    assert same_bytes(cxy, cyx)
    # scaling x by 2^a and y by 2^b scales csd by exactly 2^(a + b) and leaves coherence's bytes as they are
    for a, b in ((5, -3), (-7, 11)) if dtype == F32 else ((60, -40), (-90, 100)):
        xs, ys = (x * dtype(2.0) ** a).astype(x.dtype), (y * dtype(2.0) ** b).astype(y.dtype)
        got, _ = run_csd(xs, ys, points, hop, frames, flags, dtype)
        assert same_bytes(got, (sxy * dtype(2.0) ** (a + b)).astype(sxy.dtype)), (a, b)
        got, _ = run_csd(xs, ys, points, hop, frames, cflags, dtype, coherence=True)
        assert same_bytes(got, cxy), (a, b)
    # csd(x, x) is welch(x) up to the order of the sums: both within the bounds of the same reference
    pw, _ = run_welch(x, points, hop, frames, flags, dtype)
    w = library_window(kind_of(flags), points, dtype)
    ref = welch_closed_form(x, points, hop, w, flags, FS, acc.ref_ctype(dtype))
    peer = welch_closed_form(x, points, hop, w, flags, FS, acc.ctype(dtype))
    check_rows(sxx.real, ref, peer, dtype, "csd(x, x) %d h%d x%d f%d" % (points, hop, frames, flags), tol_n=points)
    check_rows(pw, ref, peer, dtype, "welch(x) %d h%d x%d f%d" % (points, hop, frames, flags), tol_n=points)


@pytest.mark.parametrize("dtype", [F32, F64])
def test_a_silent_signal_gives_nan_coherence_and_zero_csd(dtype):
    points, hop, frames = 256, 64, 100
    x, _ = pair(np.random.default_rng(5), (frames - 1) * hop + points, dtype, True)
    y = np.zeros_like(x)
    coh, _ = run_csd(x, y, points, hop, frames, REAL | ONE | bd.F_WINDOW(1), dtype, coherence=True)
    assert np.all(np.isnan(coh))
    s, _ = run_csd(x, y, points, hop, frames, REAL | ONE | bd.F_WINDOW(1), dtype)
    assert np.all(s == 0)


# ---- 3. the route taken, by kernel launches ----------------------------------------------------------------------------
def frames_launches(buf, start, points, hop, frames, flags, dtype):
    """Kernel launches of bdsp_fft_frames_* over `frames` frames from point `start` of buf, without the window table that
    the call builds once."""
    out = Buf.empty(frames * points, True, 0, dtype)
    f = fn("bdsp_fft_frames", dtype)
    ptr = buf.ptr + start * buf.esize
    assert f(ptr, out.ptr, points, hop, frames, flags) == 0, bd.lib().bdsp_last_error()
    before = bd.kernel_launch_count()
    assert f(ptr, out.ptr, points, hop, frames, flags) == 0, bd.lib().bdsp_last_error()
    return bd.kernel_launch_count() - before - (1 if kind_of(flags) in (0, 1, 2) else 0)


def plan_chunks(dtype, points, frames):
    """fft_route.h csd_plan: frames per chunk"""
    per = per_group(points) if dtype == F32 else 1
    whole = 1 if points > CHUNK_POINTS else CHUNK_POINTS // points // per * per
    return min(whole, frames)


@pytest.mark.parametrize("coherence", [False, True])
@pytest.mark.parametrize("dtype,points,hop,frames,flags", [
    (F32, 1024, 256, 2 * 16384 + 5, REAL | ONE | bd.F_WINDOW(1)),  # packed frames, then a frame pass for the last 5
    (F32, 1024, 256, 64, REAL),                                    # one chunk, no window
    (F32, 64, 34, 3 * 262144, SH | bd.F_WINDOW(2)),                # three whole chunks
    (F32, 1024, 255, 64, REAL | ONE | bd.F_WINDOW(2)),             # odd hop
    (F32, 1000, 250, 40, bd.F_WINDOW(0)),
    (F32, 32, 8, 100, REAL),
    (F32, 16384, 4096, 2100, REAL | bd.F_WINDOW(1)),               # chunks of 1024, 1024 and 52 frames
    (F64, 1024, 256, 64, REAL | bd.F_WINDOW(1)),
    (F64, 4096, 1024, 4102, SH),                                   # chunks of 4096 and 6 frames
])
def test_call_runs_two_transforms_and_one_sum_per_chunk(dtype, points, hop, frames, flags, coherence):
    x, y = pair(np.random.default_rng(points + hop + 1), (frames - 1) * hop + points, dtype, flags & REAL)
    xb, yb = Buf(x, 0, dtype), Buf(y, 0, dtype)
    chunk = plan_chunks(dtype, points, frames)
    rows_flags = flags & (REAL | 0xf00)
    per_chunk = sum(frames_launches(b, f0 * hop, points, hop, min(chunk, frames - f0), rows_flags, dtype)
                    for f0 in range(0, frames, chunk) for b in (xb, yb))
    chunks = -(-frames // chunk)
    table = (1 if coherence else 2) if kind_of(flags) in (0, 1, 2) else 0   # window table (+ window sums for csd)
    run_csd(x, y, points, hop, frames, flags, dtype, coherence)
    _, n = run_csd(x, y, points, hop, frames, flags, dtype, coherence)
    assert n == table + per_chunk + chunks + 1       # + one accumulate kernel per chunk, + the final kernel


# ---- 4. reproducibility ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("coherence", [False, True])
@pytest.mark.parametrize("dtype,flags", [(F32, REAL | ONE | bd.F_WINDOW(1)), (F32, SH), (F64, REAL | bd.F_WINDOW(2))])
def test_repeated_calls_give_the_same_bytes(dtype, flags, coherence):
    points, hop = 1024, 256
    frames = 1 + ((1 << 23) - points) // hop   # two chunks
    x, y = pair(np.random.default_rng(11), (frames - 1) * hop + points, dtype, flags & REAL)
    first, _ = run_csd(x, y, points, hop, frames, flags, dtype, coherence)
    for _ in range(2):
        again, _ = run_csd(x, y, points, hop, frames, flags, dtype, coherence)
        assert same_bytes(first, again)


# ---- 5. contract -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("coherence", [False, True])
@pytest.mark.parametrize("dtype", [F32, F64])
def test_bad_arguments_and_overlap_are_rejected(dtype, coherence):
    L = bd.lib()
    g = fn("bdsp_coherence" if coherence else "bdsp_csd", dtype)

    def f(x, y, out, points, hop, frames, flags, fs=FS):
        return g(x, y, out, points, hop, frames, flags) if coherence else g(x, y, out, points, hop, frames, flags, fs)

    esz = np.dtype(dtype).itemsize
    oesz = esz if coherence else 2 * esz          # bytes per output value
    buf = Buf(rand_c(np.random.default_rng(1), 16384, dtype), 0, dtype)
    base = buf.ptr
    x, y, out = base, base + 8192 * esz, base + 24000 * esz   # complex x and y: 2560 points = 5120 scalars each
    before = bd.kernel_launch_count()
    bad = [(bd.F_INVERSE, b"BDSP_F_INVERSE"), (bd.F_MAGNITUDE, b"BDSP_F_MAGNITUDE"), (bd.F_REAL_OUTPUT, b"BDSP_F_REAL_OUTPUT"),
           (128, b"0x80"), (1 << 12, b"0x1000")] + ([(PSD, b"BDSP_F_POWER_SPECTRUM")] if coherence else [])
    for flag, name in bad:
        assert f(x, y, out, 1024, 512, 4, REAL | flag) == -2
        assert name in L.bdsp_last_error()
    assert f(x, y, out, 1024, 512, 4, ONE) == -2                        # one-sided needs real input
    assert b"ONESIDED" in L.bdsp_last_error()
    assert f(x, y, out, 1024, 512, 4, REAL | ONE | SH) == -2
    assert b"ONESIDED" in L.bdsp_last_error()
    assert f(x, y, out, 1024, 0, 4, 0) == -2
    assert b"hop" in L.bdsp_last_error()
    if not coherence:
        for fs in (0.0, -1.0, float("nan"), float("inf")):
            assert f(x, y, out, 1024, 512, 4, REAL, fs) == -2
            assert b"fs" in L.bdsp_last_error()
    assert f(x, y, out, 1 << 40, 1 << 40, 1 << 30, 0) == -2            # (frames - 1) * hop overflows
    assert b"overflow" in L.bdsp_last_error()
    # outputs of 1024 values (or 513 one-sided) overlapping x, or y only
    assert f(x, y, x + 5119 * esz, 1024, 512, 4, 0) == -3
    assert b"overlaps x" in L.bdsp_last_error()
    assert f(x, y, y + 5119 * esz, 1024, 512, 4, 0) == -3
    assert b"overlaps y" in L.bdsp_last_error()
    assert f(x, y, y - 1023 * oesz + esz, 1024, 512, 4, 0) == -3       # ends one scalar into y
    assert f(x, y, y, 1024, 512, 4, REAL | ONE) == -3
    assert f(x + 1024 * oesz - esz, y, x, 1024, 512, 4, 0) == -3       # the output ends one scalar into x
    assert bd.kernel_launch_count() == before
    # adjacent ranges are fine, x and y may be the same buffer or overlap, fs is ignored for a power spectrum
    assert f(x, y, y - 1024 * oesz, 1024, 512, 4, 0) == 0
    assert f(x, x, out, 1024, 512, 4, 0) == 0
    assert f(x, x + 100 * esz, out, 1024, 512, 4, 0) == 0
    assert f(x, y, y + 5120 * esz, 1024, 512, 4, 0) == 0
    if not coherence:
        assert f(x, y, out, 1024, 512, 4, REAL | PSD, float("nan")) == 0
    bd.synchronize()


@pytest.mark.parametrize("coherence", [False, True])
@pytest.mark.parametrize("dtype", [F32, F64])
def test_empty_calls_launch_nothing_and_leave_the_output(dtype, coherence):
    x = Buf(rand_c(np.random.default_rng(2), 1024, dtype), 0, dtype)
    sentinel = np.full(2048, 7.5, dtype=dtype)
    out = Buf(sentinel, 0, dtype)
    g = fn("bdsp_coherence" if coherence else "bdsp_csd", dtype)
    extra = () if coherence else (FS,)
    before = bd.kernel_launch_count()
    assert g(x.ptr, x.ptr, out.ptr, 1024, 256, 0, bd.F_WINDOW(1), *extra) == 0
    assert g(x.ptr, x.ptr, out.ptr, 0, 256, 4, 0, *extra) == 0
    assert bd.kernel_launch_count() == before
    assert np.array_equal(out.get(sentinel.shape), sentinel)


# ---- 6. bounded workspace ----------------------------------------------------------------------------------------------
def test_workspace_stays_bounded_past_32_gib_of_spectra():
    """c64, 2^18 + 1 frames of 4096 points 64 apart: the frame spectra of x and y would take 32 GiB + 128 KiB.  The call runs
    in chunks of CHUNK_POINTS spectrum points per signal; its workspace grows by less than 2 GiB."""
    torch = pytest.importorskip("torch")
    points, hop, frames = 4096, 64, (1 << 18) + 1
    assert 2 * frames * points * 16 > 32 << 30
    flags = REAL | ONE | bd.F_WINDOW(1)
    rng = np.random.default_rng(12)
    x = rng.uniform(-1, 1, (frames - 1) * hop + points)
    y = np.convolve(x, [0.5, 1.0, -0.25], mode="same") + 0.5 * rng.uniform(-1, 1, x.size)
    xin, yin = Buf(x, 0, F64), Buf(y, 0, F64)
    out = Buf.empty(points // 2 + 1, True, 0, F64)
    bd.synchronize()
    free_before = bd.lib().bdsp_mem_free()
    assert fn("bdsp_csd", F64)(xin.ptr, yin.ptr, out.ptr, points, hop, frames, flags, FS) == 0, bd.lib().bdsp_last_error()
    bd.synchronize()
    assert free_before - bd.lib().bdsp_mem_free() < 2 << 30
    got = out.get(points // 2 + 1)
    # reference: the same closed form on the GPU with torch, in float64, the library's window table
    w = torch.from_numpy(library_window(1, points, F64)).cuda()
    xt, yt = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    acc_p = torch.zeros(points // 2 + 1, dtype=torch.complex128, device="cuda")
    for f0 in range(0, frames, 1 << 14):
        cnt = min(1 << 14, frames - f0)
        X = torch.fft.rfft(xt[f0 * hop:].unfold(0, points, hop)[:cnt] * w)
        Y = torch.fft.rfft(yt[f0 * hop:].unfold(0, points, hop)[:cnt] * w)
        acc_p += (X.conj() * Y).sum(0)
    want = (acc_p / (frames * FS * (w * w).sum())).cpu().numpy()
    want[1:points // 2] *= 2
    assert np.max(np.abs(got - want)) <= 1e-11 * np.max(np.abs(want))
