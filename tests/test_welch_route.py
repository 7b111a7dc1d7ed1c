"""Route of bdsp_welch_* (fft_route.h welch_route) without a GPU: a g++-built driver prints whether the power sum is fused
into the packed frames kernel, over how many groups of 4096 / n frames (n >= 4096: one frame per group), and how many
CTAs loop over them.  The fused rule: c32, n = 2^k in [64, 8192], an even hop, the input aligned like the packed frames
route (16 B complex, 8 B real), the grid limit.  Unlike bdsp_fft_frames_* an incomplete last group stays fused."""
import itertools
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IN = 0x7f0000000000
GRID_MAX = 0x7FFFFFFF
CTAS = {8192: 296}   # WELCH_CTAS_8192; every other fused length: WELCH_CTAS
CTAS_DEFAULT = 592


@pytest.fixture(scope="module")
def welch_route(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("welch_route") / "welch_route_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "basic_dsp_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cpp", "welch_route_driver.cpp"), "-o", exe])
    proc = subprocess.Popen([exe], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)

    def run(f64, n, hop, frames, real=False, src=IN):
        """-> (fused, groups, ctas)"""
        proc.stdin.write("%d %d %d %d %d %x\n" % (f64, n, hop, frames, real, src))
        proc.stdin.flush()
        f = proc.stdout.readline().split()
        return bool(int(f[0])), int(f[1]), int(f[2])

    yield run
    proc.stdin.close()
    proc.wait()


def per_group(n):
    return 4096 // n if n < 4096 else 1


def fused_by_rule(f64, n, hop, frames, real, src):
    groups = -(-frames // per_group(n))
    return (not f64 and n & (n - 1) == 0 and 64 <= n <= 8192 and hop % 2 == 0 and src % (8 if real else 16) == 0 and
            groups <= GRID_MAX)


def test_fused_exactly_where_specified(welch_route):
    seen = set()
    grid = itertools.product((False, True), (32, 64, 128, 256, 1000, 1024, 3072, 4096, 8192, 16384), (1, 3, 15, 16, 17, 63, 64, 65, 1023, 1048573),
                             ("quarter", "odd", "equal", "over"), (False, True), (IN, IN + 4, IN + 8, IN + 16))
    for f64, n, frames, hopk, real, src in grid:
        hop = {"quarter": n // 4, "odd": n // 2 - 1, "equal": n, "over": n + 2}[hopk]
        fused, groups, ctas = welch_route(f64, n, hop, frames, real, src)
        want = fused_by_rule(f64, n, hop, frames, real, src)
        assert fused == want, (f64, n, hop, frames, real, hex(src))
        if want:
            assert groups == -(-frames // per_group(n))
            assert ctas == min(groups, CTAS.get(n, CTAS_DEFAULT))
        seen.add(fused)
    assert seen == {False, True}


# (arguments, fused): the boundaries of the rule
BOUNDARIES = [
    # lengths: 32, 64, 8192, 16384, and lengths that are not powers of two
    (dict(f64=False, n=32, hop=8, frames=4096), False),
    (dict(f64=False, n=64, hop=16, frames=4096), True),
    (dict(f64=False, n=8192, hop=2048, frames=8), True),
    (dict(f64=False, n=16384, hop=4096, frames=8), False),
    (dict(f64=False, n=1000, hop=250, frames=64), False),
    (dict(f64=False, n=3072, hop=768, frames=64), False),
    # c64
    (dict(f64=True, n=1024, hop=256, frames=64), False),
    # hop parity, hop above n
    (dict(f64=False, n=1024, hop=255, frames=64), False),
    (dict(f64=False, n=1024, hop=1026, frames=64), True),
    (dict(f64=False, n=1024, hop=1027, frames=64), False),
    # alignment: 16 B for complex points, 8 B for real scalars
    (dict(f64=False, n=1024, hop=256, frames=64, src=IN + 8), False),
    (dict(f64=False, n=1024, hop=256, frames=64, src=IN + 16), True),
    (dict(f64=False, n=1024, hop=256, frames=64, real=True, src=IN + 4), False),
    (dict(f64=False, n=1024, hop=256, frames=64, real=True, src=IN + 8), True),
    # the grid limit
    (dict(f64=False, n=4096, hop=2048, frames=GRID_MAX), True),
    (dict(f64=False, n=4096, hop=2048, frames=GRID_MAX + 1), False),
    (dict(f64=False, n=1024, hop=512, frames=4 * GRID_MAX), True),
    (dict(f64=False, n=1024, hop=512, frames=4 * GRID_MAX + 1), False),   # the last group holds one frame
]


@pytest.mark.parametrize("args,fused", BOUNDARIES, ids=["%d-%s" % (i, f) for i, (_, f) in enumerate(BOUNDARIES)])
def test_boundaries(welch_route, args, fused):
    assert welch_route(**args)[0] == fused


@pytest.mark.parametrize("n,frames,groups,ctas", [
    (1024, 1048573, 262144, 592),   # 2^28 real samples, hop 256: 1048573 = 4 * 262143 + 1 frames, the last group holds one
    (1024, 1048572, 262143, 592),
    (256, 524287, 32768, 592),      # 2^26 points, hop 128: 15 frames past whole groups of 16
    (4096, 32767, 32767, 592),
    (8192, 100, 100, 100),
    (8192, 1000, 1000, 296),
    (64, 1, 1, 1),                  # one frame: one CTA, 63 frames of zeros
    (64, 65, 2, 2),
])
def test_incomplete_groups_are_fused(welch_route, n, frames, groups, ctas):
    assert welch_route(False, n, 2, frames) == (True, groups, ctas)
    assert welch_route(False, n, 2, frames, real=True) == (True, groups, ctas)
