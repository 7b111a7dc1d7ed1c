"""The FFT routing table (basic_dsp_b200/csrc/fft_route.h) without a GPU: a g++-built driver prints the route fft_route
picks, for every case of the GPU accuracy tests and for the boundaries between routes."""
import os
import subprocess

import numpy as np
import pytest

from test_gpu_accuracy import F32, F64, FFT_CASES, INV, MAG, REAL, SH, WINDOWED_CASES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK_MAX = {F32: 16384, F64: 8192}
# device addresses: the caller's buffers, the pass workspace and workspace slots 1 / 2 (256-byte aligned allocations)
IN, OUT, WORK, WS1, WS2 = 0x7f0000000000, 0x7f1000000000, 0x7f2000000000, 0x7f3000000000, 0x7f4000000000


@pytest.fixture(scope="module")
def route(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("fft_route") / "fft_route_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "basic_dsp_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cpp", "fft_route_driver.cpp"), "-o", exe])
    proc = subprocess.Popen([exe], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)

    def run(dtype, n, rows, inverse=False, real=False, mag=False, in_mul=0, in_rot=0, out_rot=0, src=IN, dst=OUT, work=0,
            cluster=True, generic=False):
        """-> (route name, groups, n1, log2n2, log2n3, q, P)"""
        proc.stdin.write("%d %d %d %d %d %d %d %d %d %x %x %x %d %d\n" % (dtype == F64, n, rows, inverse, real, mag, in_mul, in_rot,
                                                                          out_rot, src, dst, work, cluster, generic))
        proc.stdin.flush()
        f = proc.stdout.readline().split()
        return (f[0],) + tuple(int(v) for v in f[1:])

    yield run
    proc.stdin.close()
    proc.wait()


def chain(run, dtype, n, rows, inverse, real, mag, in_mul, in_rot, out_rot, src, dst, work=0):
    """The routes fft_any takes level by level ("mul-pass > packed"): the multiplier and complexifying passes route their
    product again, a q * 2^k transform routes its rows of P points."""
    if n & (n - 1) == 0 and n > BLOCK_MAX[dtype]:
        work = work or WORK
    r = run(dtype, n, rows, inverse, real, mag, in_mul, in_rot, out_rot, src, dst, work)
    if r[0] == "mul-pass":
        return r[0] + " > " + chain(run, dtype, n, rows, inverse, real, mag, 0, in_rot, out_rot, WS2, dst, work)
    if r[0] == "complexify":
        return r[0] + " > " + chain(run, dtype, n, rows, inverse, False, mag, in_mul, in_rot, out_rot, WS1, dst, work)
    if r[0] == "q-rows-interleave":
        q, P = r[5], r[6]
        return r[0] + " > " + chain(run, dtype, P, rows * q, inverse, False, False, 0, 0, 0, WS1, WS2, WORK if P > BLOCK_MAX[dtype] else 0)
    return r[0]


def rows_api(run, dtype, n, rows, flags, variant="", window=False):
    """Routes of bdsp_fft_rows_* (capi.cu fft_rows) on buffers laid out as test_gpu_accuracy.Buf does."""
    inverse, real, mag = bool(flags & INV), bool(flags & REAL), bool(flags & MAG)
    esize = np.dtype(dtype).itemsize
    off = 1 if variant == "offset" else 0
    src = IN + off * esize * (1 if real else 2)
    dst = src if variant == "inplace" else OUT + off * esize * (1 if mag else 2)
    half = n // 2 if flags & SH else 0
    return chain(run, dtype, n, rows, inverse, real, mag, 1 if window else 0, half if inverse else 0, 0 if inverse else half, src, dst)


@pytest.mark.parametrize("case", [c.values for c in FFT_CASES], ids=[c.id for c in FFT_CASES])
def test_accuracy_case_route(route, case):
    dtype, n, rows, flags, variant, branch, cond, expected = case
    got = rows_api(route, dtype, n, rows, flags, variant)
    want = expected.get(flags, expected[None]) if isinstance(expected, dict) else expected
    assert got == want, (branch, cond)


@pytest.mark.parametrize("dtype,n,rows,branch,expected", WINDOWED_CASES)
def test_windowed_case_route(route, dtype, n, rows, branch, expected):
    assert rows_api(route, dtype, n, rows, SH, window=True) == expected, branch


# (arguments of the driver call, expected route): the boundaries between routes
BOUNDARIES = [
    # n * batch just below and at 2^16: separate multiplier pass, packed real rows
    (dict(dtype=F32, n=4096, rows=15, in_mul=1), "block"),
    (dict(dtype=F32, n=4096, rows=16, in_mul=1), "mul-pass"),
    (dict(dtype=F32, n=4096, rows=15, real=True), "block"),
    (dict(dtype=F32, n=4096, rows=16, real=True), "real-rows"),
    # n * batch just below and at 2^18: complexifying pass, packed rows of a q * 2^k transform
    (dict(dtype=F32, n=4096, rows=63, real=True, inverse=True), "block"),
    (dict(dtype=F32, n=4096, rows=64, real=True, inverse=True), "complexify"),
    (dict(dtype=F32, n=3 * 4096, rows=21), "q-rows"),
    (dict(dtype=F32, n=3 * 4096, rows=22), "q-rows-interleave"),
    # whole groups of 4096 points: rows % (4096 / n)
    (dict(dtype=F32, n=1024, rows=8), "packed"),
    (dict(dtype=F32, n=1024, rows=9), "block"),
    (dict(dtype=F32, n=1024, rows=64, real=True), "real-rows"),
    (dict(dtype=F32, n=1024, rows=65, real=True), "block"),
    (dict(dtype=F32, n=1024, rows=256, real=True, inverse=True), "complexify"),
    (dict(dtype=F32, n=1024, rows=257, real=True, inverse=True), "block"),
    (dict(dtype=F32, n=768, rows=352), "q-rows-interleave"),
    (dict(dtype=F32, n=768, rows=353), "q-rows"),
    # 16384 points: the persistent kernel from two rows on
    (dict(dtype=F32, n=16384, rows=1), "packed"),
    (dict(dtype=F32, n=16384, rows=2), "packed-16k"),
    # 8 vs 9 rows at 2^16, cluster not usable
    (dict(dtype=F32, n=65536, rows=8), "cluster"),
    (dict(dtype=F32, n=65536, rows=9, work=WORK), "two-pass"),
    (dict(dtype=F32, n=65536, rows=1, work=WORK, cluster=False), "two-pass"),
    # 8- vs 16-byte misalignment
    (dict(dtype=F32, n=4096, rows=1, src=IN + 8), "block"),
    (dict(dtype=F32, n=4096, rows=1, src=IN + 16), "packed"),
    (dict(dtype=F32, n=4096, rows=16, real=True, src=IN + 4), "block"),
    (dict(dtype=F32, n=4096, rows=16, real=True, src=IN + 8), "real-rows"),
    (dict(dtype=F32, n=65536, rows=1, src=IN + 8), "cluster"),
    (dict(dtype=F32, n=65536, rows=1, src=IN + 4, work=WORK), "hybrid"),
    (dict(dtype=F32, n=1 << 20, rows=1, src=IN + 8, dst=OUT + 8, work=WORK), "hybrid"),
    (dict(dtype=F32, n=1 << 20, rows=1, src=IN + 16, dst=OUT + 8, work=WORK), "two-pass"),
    (dict(dtype=F32, n=1 << 20, rows=1, src=IN + 8, dst=OUT + 4, work=WORK), "tiles"),
    (dict(dtype=F32, n=1 << 20, rows=1, work=WORK + 8), "tiles"),
    (dict(dtype=F32, n=1 << 21, rows=1, src=IN + 8, work=WORK), "tiles"),
    # in == out, work == in
    (dict(dtype=F32, n=4096, rows=1, dst=IN), "block"),
    (dict(dtype=F32, n=65536, rows=1, dst=IN, work=WORK), "two-pass"),
    (dict(dtype=F32, n=1 << 18, rows=1, work=IN), "tiles"),
    (dict(dtype=F32, n=1 << 22, rows=1, work=OUT), "tiles"),
    (dict(dtype=F64, n=1024, rows=4, dst=IN), "c64-rows"),
    (dict(dtype=F64, n=1024, rows=4, dst=IN, mag=True), "block"),
    (dict(dtype=F64, n=1024, rows=4, dst=IN, real=True), "block"),
    (dict(dtype=F64, n=1024, rows=1 << 31), "block"),
    # inverse with magnitude or fft_shift on the store
    (dict(dtype=F32, n=4096, rows=1, inverse=True, mag=True), "block"),
    (dict(dtype=F32, n=4096, rows=1, inverse=True, out_rot=2048), "block"),
    (dict(dtype=F32, n=4096, rows=1, inverse=True, in_rot=2048), "packed"),
    (dict(dtype=F32, n=65536, rows=1, inverse=True, out_rot=32768), "cluster"),
    (dict(dtype=F32, n=65536, rows=9, inverse=True, out_rot=32768, work=WORK), "tiles"),
    (dict(dtype=F32, n=65536, rows=9, inverse=True, mag=True, work=WORK), "tiles"),
    (dict(dtype=F32, n=1 << 21, rows=1, inverse=True, mag=True, work=WORK), "tiles"),
    # real input with inverse or ifft_shift
    (dict(dtype=F32, n=4096, rows=64, real=True, in_rot=2048), "complexify"),
    (dict(dtype=F32, n=1 << 15, rows=1, real=True, inverse=True, work=WORK), "complexify"),
    (dict(dtype=F32, n=1 << 15, rows=1, real=True, work=WORK), "two-pass"),
    # forward with ifft_shift: the packed single-pass kernels have no such variant, the column passes do
    (dict(dtype=F32, n=4096, rows=1, in_rot=2048), "block"),
    (dict(dtype=F32, n=16384, rows=2, in_rot=8192), "block"),
    (dict(dtype=F32, n=65536, rows=9, in_rot=32768, work=WORK), "two-pass"),
    (dict(dtype=F32, n=4096, rows=1, in_rot=1), "block"),
    # the generic kernels only: the rows of a q * 2^k transform and the Bluestein sub-transforms
    (dict(dtype=F32, n=4096, rows=16, generic=True), "block"),
    (dict(dtype=F32, n=1 << 16, rows=1, dst=IN, work=WORK, generic=True), "hybrid"),
    # q * 2^k: the f64 folded radix-q first pass and its limits, Bluestein
    (dict(dtype=F64, n=3 << 14, rows=1), "q-three-pass"),
    (dict(dtype=F64, n=3 << 14, rows=1, mag=True), "q-rows-interleave"),
    (dict(dtype=F64, n=3 << 27, rows=1), "q-rows-interleave"),
    (dict(dtype=F64, n=3 << 13, rows=1), "q-rows"),
    (dict(dtype=F32, n=33 * 64, rows=1), "bluestein"),
    (dict(dtype=F32, n=31 * 64, rows=1), "q-rows"),
    (dict(dtype=F32, n=31, rows=1), "bluestein"),
]


@pytest.mark.parametrize("args,expected", BOUNDARIES, ids=["%d-%s" % (i, e) for i, (_, e) in enumerate(BOUNDARIES)])
def test_route_boundaries(route, args, expected):
    assert route(**args)[0] == expected


def test_packed_geometry(route):
    """Launch geometry handed to the packed launchers."""
    assert route(F32, 1024, 8)[1] == 2                                 # CTAs of four 1024-point rows
    assert route(F32, 1 << 20, 64, work=WORK)[1:4] == (64 * 64, 256, 12)
    assert route(F32, 1 << 16, 9, work=WORK)[1:4] == (9 * 16, 256, 8)
    assert route(F32, 1 << 24, 1, work=WORK)[1:5] == (16 * 256, 256, 0, 8)
    assert route(F32, 1 << 20, 1, src=IN + 8, work=WORK)[1:3] == (256, 1024)
    assert route(F64, 3 << 26, 1)[2:7] == (768, 9, 9, 3, 1 << 26)
