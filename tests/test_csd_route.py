"""Chunk plan of bdsp_csd_* / bdsp_coherence_* (fft_route.h csd_plan) composed with fft_route, without a GPU: a g++-built
driver prints the frames per chunk, the partial rows, and the route of each chunk's frame transforms of x and of y as
csd_exec calls them.  Checked: the chunks cover every frame once; two chunk spectra hold at most 2 * CSD_CHUNK_POINTS
points (one frame per chunk when a frame is longer); for c32 below 4096 points a chunk holds whole groups of 4096 / n
frames, so that with a power-of-two n in [64, 8192], an even hop and aligned input every chunk but the last takes the
packed frames route, and so does the last when the frames make whole groups."""
import itertools
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
X, Y, SPEC = 0x7f0000000000, 0x7f4000000000, 0x7e0000000000
ACC_THREADS = 1 << 18   # fft_route.h CSD_ACC_THREADS


def route_names():
    with open(os.path.join(ROOT, "basic_dsp_b200", "csrc", "fft_route.h")) as fh:
        body = re.search(r"enum class FftRoute \{(.*?)\};", fh.read(), re.S).group(1)
    return [m for m in re.findall(r"^\s*(\w+),", body, re.M)]


@pytest.fixture(scope="module")
def csd_plan(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("csd_route") / "csd_route_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "basic_dsp_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cpp", "csd_route_driver.cpp"), "-o", exe])
    proc = subprocess.Popen([exe], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
    chunk_points = int(proc.stdout.readline())
    names = route_names()

    def run(f64, n, hop, frames, real=False, window=True, x=X, y=Y):
        """-> (chunk, slabs, [(frames of the chunk, route of x, route of y)])"""
        proc.stdin.write("%d %d %d %d %d %d %x %x %x\n" % (f64, n, hop, frames, real, window, x, y, SPEC))
        proc.stdin.flush()
        f = [int(v) for v in proc.stdout.readline().split()]
        chunks = [(f[i], names[f[i + 1]], names[f[i + 2]]) for i in range(3, len(f), 3)]
        assert len(chunks) == f[2]
        return f[0], f[1], chunks

    run.chunk_points = chunk_points
    yield run
    proc.stdin.close()
    proc.wait()


def per_group(f64, n):
    return 4096 // n if not f64 and 64 <= n < 4096 else 1


GRID = list(itertools.product((False, True), (64, 128, 256, 1000, 1024, 3072, 4096, 8192, 16384, 1 << 20, 1 << 23),
                              ("quarter", "odd", "equal", "over"), (False, True)))


@pytest.mark.parametrize("f64,n,hopk,real", GRID, ids=["%s-%d-%s-%s" % ("c64" if c[0] else "c32", c[1], c[2], "real" if c[3] else "cpx")
                                                       for c in GRID])
def test_chunks_cover_the_frames_within_the_bound(csd_plan, f64, n, hopk, real):
    hop = {"quarter": n // 4, "odd": n // 2 - 1, "equal": n, "over": n + 2}[hopk]
    per = per_group(f64, n)
    for frames in sorted({1, 3, per, per + 1, 4 * csd_plan.chunk_points // n + 1, 4 * csd_plan.chunk_points // n // per * per,
                          (1 << 16) + 5}):
        chunk, slabs, chunks = csd_plan(f64, n, hop, frames, real)
        assert sum(cf for cf, _, _ in chunks) == frames
        assert all(cf == chunk for cf, _, _ in chunks[:-1]) and 0 < chunks[-1][0] <= chunk
        if n <= csd_plan.chunk_points:
            assert 2 * chunk * n <= 2 * csd_plan.chunk_points
        else:
            assert chunk == 1
        if chunk < frames:
            assert chunk % per == 0
        assert slabs == min(-(-ACC_THREADS // n), chunk)


PACKED = list(itertools.product((64, 128, 256, 512, 1024, 2048, 4096, 8192), ("quarter", "half", "over"), (False, True), (False, True)))


@pytest.mark.parametrize("n,hopk,real,window", PACKED, ids=["%d-%s-%s-%s" % (n, h, "real" if r else "cpx", "win" if w else "rect")
                                                           for n, h, r, w in PACKED])
def test_whole_chunks_keep_the_packed_frames_route(csd_plan, n, hopk, real, window):
    """c32, n = 2^k in [64, 8192], an even hop other than n (hop == n: the frames are plain rows), aligned x and y."""
    hop = {"quarter": n // 4, "half": n // 2, "over": n + 2}[hopk]
    per = per_group(False, n)
    whole = csd_plan.chunk_points // n
    for frames in (3 * whole, 3 * whole + per, 3 * whole + 1, 3 * whole - per, 2 * whole + (1 << 16) // n // per * per + per):
        chunk, _, chunks = csd_plan(False, n, hop, frames, real, window)
        assert chunk == whole and len(chunks) > 1
        for cf, rx, ry in chunks[:-1]:
            assert rx == ry == "PackedFrames", (frames, cf)
        cf, rx, ry = chunks[-1]
        if frames % per == 0 and cf * n >= 1 << 16:   # fft_route's whole-group and size rules for the last chunk
            assert rx == ry == "PackedFrames", (frames, cf)
        else:
            assert rx == ry == "FramePass", (frames, cf)


def test_misaligned_y_leaves_x_on_the_packed_route(csd_plan):
    n, hop = 1024, 256
    frames = 2 * csd_plan.chunk_points // n
    _, _, chunks = csd_plan(False, n, hop, frames, True, True, y=Y + 4)
    assert all(rx == "PackedFrames" and ry == "FramePass" for _, rx, ry in chunks)
