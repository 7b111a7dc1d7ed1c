"""Routes of strided input frames (FftRouteIn::in_stride, bdsp_fft_frames_*) without a GPU: a g++-built driver prints the
route fft_route picks.  With in_stride 0 or n every answer is the one of the row driver (tests/cpp/fft_route_driver.cpp);
otherwise the fused packed frames route is taken exactly where the frames, laid back to back, would reach the packed or
real-row single pass, and the gathering frame pass everywhere else."""
import itertools
import os
import subprocess

import pytest

from test_fft_route import BOUNDARIES, IN, OUT, WORK, WS1, WS2, chain, route, rows_api  # noqa: F401  (route: fixture)
from test_gpu_accuracy import F32, F64, FFT_CASES, WINDOWED_CASES, SH

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WS6 = 0x7f6000000000   # workspace slot 6: the gathered frames
GRID_MAX = 0x7FFFFFFF


@pytest.fixture(scope="module")
def frames_route(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("fft_frames_route") / "fft_frames_route_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "basic_dsp_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cpp", "fft_frames_route_driver.cpp"), "-o", exe])
    proc = subprocess.Popen([exe], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)

    def run(dtype, n, rows, inverse=False, real=False, mag=False, in_mul=0, in_rot=0, out_rot=0, src=IN, dst=OUT, work=0,
            cluster=True, generic=False, stride=0):
        """-> (route name, groups, n1, log2n2, log2n3, q, P)"""
        proc.stdin.write("%d %d %d %d %d %d %d %d %d %x %x %x %d %d %d\n" % (dtype == F64, n, rows, inverse, real, mag, in_mul, in_rot,
                                                                             out_rot, src, dst, work, cluster, generic, stride))
        proc.stdin.flush()
        f = proc.stdout.readline().split()
        return (f[0],) + tuple(int(v) for v in f[1:])

    yield run
    proc.stdin.close()
    proc.wait()


def test_contiguous_strides_route_as_rows(route, frames_route):
    """in_stride 0 and in_stride n answer exactly as the row driver, at every level of every case of test_fft_route.py."""
    calls = []

    def both(*args, **kw):
        want = route(*args, **kw)
        n = kw["n"] if "n" in kw else args[1]
        for stride in (0, n):
            assert frames_route(*args, stride=stride, **kw) == want, (args, kw, stride)
        calls.append(want[0])
        return want

    for case in FFT_CASES:
        dtype, n, rows, flags, variant = case.values[:5]
        rows_api(both, dtype, n, rows, flags, variant)
    for dtype, n, rows, _, _ in WINDOWED_CASES:
        rows_api(both, dtype, n, rows, SH, window=True)
    for args, _ in BOUNDARIES:
        both(**args)
    assert len(calls) > len(FFT_CASES) + len(BOUNDARIES)


def fused_by_rule(dtype, n, frames, hop, real, mag, in_mul, out_rot, src, dst):
    """The fused frames route as specified: c32, forward, n = 2^k in [64, 8192], multiplier kind 0 or 1, fft_shift or none
    on the store, n * frames >= 2^16, whole groups of 4096 / n frames below 4096 points, the grid limit, the alignment of
    the packed (complex: in 16 B) and real-row (in 8 B) single passes with out 8 B, an even hop, out != in."""
    per = 4096 // n if n < 4096 else 1
    grid = frames // per * 2 if real else (frames // per if n < 4096 else frames * 2)
    return (dtype == F32 and n & (n - 1) == 0 and 64 <= n <= 8192 and in_mul in (0, 1) and out_rot in (0, n // 2) and
            n * frames >= 1 << 16 and frames % per == 0 and grid <= GRID_MAX and src % (8 if real else 16) == 0 and dst % 8 == 0 and
            hop % 2 == 0 and src != dst)


def test_fused_route_exactly_where_specified(frames_route):
    grid = itertools.product(
        (F32, F64), (32, 64, 128, 1000, 1024, 4096, 8192, 16384), (1, 15, 16, 63, 64, 65, 1023, 1024),
        ("even", "odd", "over"), (False, True), (False, True), (0, 1, 2), ("none", "half", "one"),
        ((IN, OUT), (IN + 4, OUT), (IN + 8, OUT), (IN + 16, OUT), (IN, OUT + 4), (IN, OUT + 8), (IN, IN)))
    seen = set()
    for dtype, n, frames, hopk, real, mag, in_mul, rot, (src, dst) in grid:
        hop = {"even": n // 2, "odd": n // 2 - 1, "over": n + 2}[hopk]
        out_rot = {"none": 0, "half": n // 2, "one": 1}[rot]
        r = frames_route(dtype, n, frames, real=real, mag=mag, in_mul=in_mul, out_rot=out_rot, src=src, dst=dst, stride=hop)
        want = fused_by_rule(dtype, n, frames, hop, real, mag, in_mul, out_rot, src, dst)
        assert r[0] == ("packed-frames" if want else "frame-pass"), (dtype, n, frames, hop, real, mag, in_mul, out_rot, src, dst)
        if want:
            assert r[1] == frames // (4096 // n if n < 4096 else 1)
        seen.add(r[0])
    assert seen == {"packed-frames", "frame-pass"}


# (arguments of the driver call, expected route): the boundaries of the fused frames route
FRAME_BOUNDARIES = [
    # n of 32, 64, 8192 and 16384
    (dict(dtype=F32, n=32, rows=4096, stride=16), "frame-pass"),
    (dict(dtype=F32, n=64, rows=1024, stride=32), "packed-frames"),
    (dict(dtype=F32, n=8192, rows=8, stride=4096), "packed-frames"),
    (dict(dtype=F32, n=8192, rows=8, stride=4096, real=True, mag=True), "packed-frames"),
    (dict(dtype=F32, n=16384, rows=4, stride=8192), "frame-pass"),
    # n * frames just below and at 2^16 (and 2^16 - 1 exactly, at a length that is not a power of two)
    (dict(dtype=F32, n=4096, rows=15, stride=2048), "frame-pass"),
    (dict(dtype=F32, n=4096, rows=16, stride=2048), "packed-frames"),
    (dict(dtype=F32, n=17 * 257, rows=15, stride=2048), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=63, stride=256, real=True), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=256, real=True), "packed-frames"),
    # frames not a multiple of 4096 / n
    (dict(dtype=F32, n=1024, rows=65, stride=256), "frame-pass"),
    (dict(dtype=F32, n=256, rows=4097, stride=128), "frame-pass"),
    (dict(dtype=F32, n=256, rows=4096, stride=128), "packed-frames"),
    # odd hop, hop > n
    (dict(dtype=F32, n=1024, rows=64, stride=511), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=1027), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=1030), "packed-frames"),
    # hop == n is the row layout
    (dict(dtype=F32, n=1024, rows=64, stride=1024), "packed"),
    (dict(dtype=F32, n=1024, rows=64, stride=1024, real=True), "real-rows"),
    # 8- versus 16-byte misalignment of in and out
    (dict(dtype=F32, n=1024, rows=64, stride=512, src=IN + 8), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, src=IN + 16), "packed-frames"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, src=IN + 4, real=True), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, src=IN + 8, real=True), "packed-frames"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, dst=OUT + 4), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, dst=OUT + 8), "packed-frames"),
    # c64, in == out, inverse, ifft_shift, a fft_shift other than n / 2, a complex multiplier table, the grid limit
    (dict(dtype=F64, n=1024, rows=64, stride=512), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, dst=IN), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, inverse=True), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, in_rot=512), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, out_rot=512, mag=True, in_mul=1), "packed-frames"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, out_rot=1), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=64, stride=512, in_mul=2), "frame-pass"),
    (dict(dtype=F32, n=4096, rows=GRID_MAX // 2, stride=2048), "packed-frames"),
    (dict(dtype=F32, n=4096, rows=GRID_MAX // 2 + 1, stride=2048), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=4 * GRID_MAX, stride=512), "packed-frames"),
    (dict(dtype=F32, n=1024, rows=4 * (GRID_MAX + 1), stride=512), "frame-pass"),
    (dict(dtype=F32, n=1024, rows=4 * (GRID_MAX // 2), stride=512, real=True), "packed-frames"),
    (dict(dtype=F32, n=1024, rows=4 * (GRID_MAX // 2 + 1), stride=512, real=True), "frame-pass"),
]


@pytest.mark.parametrize("args,expected", FRAME_BOUNDARIES, ids=["%d-%s" % (i, e) for i, (_, e) in enumerate(FRAME_BOUNDARIES)])
def test_frame_route_boundaries(frames_route, args, expected):
    assert frames_route(**args)[0] == expected


def frames_chain(run, dtype, n, rows, hop, real=False, mag=False, in_mul=0, out_rot=0, src=IN, dst=OUT):
    """The routes fft_any takes for strided frames: the frame pass gathers into workspace slot 6 and routes the rows again
    with in_stride = n, as the row driver's chain does from there on."""
    r = run(dtype, n, rows, real=real, mag=mag, in_mul=in_mul, out_rot=out_rot, src=src, dst=dst, stride=hop)
    if r[0] != "frame-pass":
        return r[0]

    def rows_run(*args, **kw):   # chain() passes n positionally: every level routes contiguous rows of its own length
        return run(*args, stride=args[1], **kw)

    return "frame-pass > " + chain(rows_run, dtype, n, rows, False, real, mag, in_mul, 0, out_rot, WS6, dst)


# the nested cases of the frame pass: what the gathered rows are routed to (the GPU tests run each of them)
NESTED = [
    (dict(dtype=F32, n=16384, rows=4, hop=4096, in_mul=1), "frame-pass > mul-pass > packed-16k"),
    (dict(dtype=F32, n=16384, rows=4, hop=4096, real=True, in_mul=1), "frame-pass > mul-pass > real-rows"),
    (dict(dtype=F32, n=3072, rows=128, hop=1536), "frame-pass > q-rows-interleave > packed"),
    (dict(dtype=F32, n=3072, rows=4, hop=1536), "frame-pass > q-rows"),
    (dict(dtype=F32, n=1000, rows=16, hop=250, in_mul=1), "frame-pass > bluestein"),
    (dict(dtype=F64, n=1000, rows=16, hop=250), "frame-pass > bluestein"),
    (dict(dtype=F64, n=1024, rows=16, hop=255), "frame-pass > c64-rows"),
    (dict(dtype=F32, n=1024, rows=64, hop=511, in_mul=1), "frame-pass > mul-pass > packed"),
    (dict(dtype=F32, n=1024, rows=65, hop=512), "frame-pass > block"),
]


@pytest.mark.parametrize("args,expected", NESTED, ids=["%d-%s" % (i, e) for i, (_, e) in enumerate(NESTED)])
def test_frame_pass_nested_routes(frames_route, args, expected):
    assert frames_chain(frames_route, **args) == expected


def test_frames_never_reenter_the_gather_slot(frames_route):
    """The rows gathered by the frame pass are routed with in_stride = n: never a frame route again."""
    for n in (32, 1000, 3072, 16384, 1 << 16):
        got = frames_chain(frames_route, F32, n, 8, n // 2 + 1, src=IN, dst=OUT)
        assert got.startswith("frame-pass > ") and "frame" not in got[len("frame-pass > "):], got
