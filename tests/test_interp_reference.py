"""CPU checks of the interpolation reference and peer of oracle/accuracy.py, the interpolation lengths on ties, and the
impulse placement of the exact-tap tests (tests/test_gpu_interp_accuracy.py).  No GPU needed."""
import ctypes

import numpy as np
import pytest

from oracle import accuracy as acc
from oracle import dsp_oracle as o

F32, F64 = np.float32, np.float64


def _x(rng, n, cplx, dtype):
    x = rng.uniform(-10, 10, n) + (1j * rng.uniform(-10, 10, n) if cplx else 0)
    return x.astype(acc.ctype(dtype) if cplx else dtype)


@pytest.mark.parametrize("dtype", [F32, F64])
@pytest.mark.parametrize("n,factor,L,delay,kind,cplx", [(600, 4.0, 12, 0.0, 0, False), (700, 3.0, 7, 0.3, 1, True),
                                                       (404, 5.0, 202, 0.0, 1, False), (300, 2.5, 8, -0.2, 0, True),
                                                       (500, 0.5, 10, 0.0, 1, False), (250, 4.0, 125, 0.0, 0, True)])
def test_reference_and_peer_match_oracle(n, factor, L, delay, kind, cplx, dtype):
    """Both restate dsp_oracle.interpolatef (given the same tap function): they differ from it by rounding only."""
    rng = np.random.default_rng(n + L)
    x = _x(rng, n, cplx, dtype)
    ref, peer, poly = acc.interpf_pair(x, kind, 0.25, factor, delay, L, dtype)
    assert poly == (factor == int(factor) and n * factor * (2 if cplx else 1) >= 2000)
    want = o.interpolatef(x, acc.impulse(kind, 0.25, dtype), factor, delay, L, dtype)
    assert len(ref) == len(peer) == len(want)
    u = float(np.finfo(dtype).eps)
    assert o.rel_l2(np.asarray(ref, dtype=np.complex128), want) <= (4 * u if poly else 64 * u)
    assert o.rel_l2(np.asarray(peer, dtype=np.complex128), want) <= (64 * u)


@pytest.mark.parametrize("dtype", [F32, F64])
def test_impulse_matches_closed_form(dtype):
    """The tap function is the oracle's closed form up to the last bits of sin / cos (absolute: near the zeros of
    sin(pi x) the relative difference grows), and takes the special point |x| = 1 / (2 rolloff) of the raised cosine."""
    xs = np.linspace(-30, 30, 481).astype(dtype)
    for kind in (0, 1):
        f = acc.impulse(kind, 0.25, dtype)
        g = (lambda t: o.sinc_impulse(t, dtype)) if kind == 0 else (lambda t: o.raised_cosine_impulse(t, 0.25, dtype))
        got = np.array([f(t) for t in xs])
        assert np.max(np.abs(got - np.array([g(t) for t in xs], dtype=dtype))) <= 4 * np.finfo(dtype).eps
        assert np.array_equal(acc.impulse_vec(kind, 0.25, xs, np.float64 if dtype == F64 else F32)[xs == 0], [1])
    assert acc.impulse(1, 0.25, dtype)(2.0) == o.raised_cosine_impulse(2.0, 0.25, dtype)


def test_tie_lengths_round_half_away_from_zero():
    """C's round (the library) and Rust's round (the reference) take halves away from zero."""
    assert o.round_half_away(2502.5) == 2503 and o.round_half_away(-2.5) == -3 and o.round_half_away(2.4999) == 2
    assert o.interpolatef_new_len(1001, 2.5, F32) == 2504                 # real N = 1001, x2.5
    assert o.interpolatef_new_len(2 * 1001, 2.25, F32) == 4506            # complex N = 1001, x2.25
    assert o.interpolatef_new_len(1001, 2.5, F64) == 2504
    assert o.interpolate_lin_dest_len(998, 2.5, F32) == 2494
    assert o.interpolate_lin_dest_len(998, 2.5, F64) == 2494


@pytest.mark.parametrize("sfx,dtype", [("32", F32), ("64", F64)])
@pytest.mark.parametrize("points,cplx,factor", [(1001, 0, 2.5), (1001, 1, 2.25), (1000, 0, 4.0), (777, 1, 3.0)])
def test_tie_lengths_match_library(points, cplx, factor, sfx, dtype):
    """bdsp_interpolatef_rows* with rows = 0 reports new_points without touching a device."""
    import basic_dsp_b200 as bd
    n = ctypes.c_size_t(0)
    rc = getattr(bd.lib(), "bdsp_interpolatef_rows" + sfx)(None, None, points, 0, cplx, 0, 0.0, factor, 0.0, 12, ctypes.byref(n))
    assert rc == 0
    assert n.value == o.interpolatef_new_len((2 if cplx else 1) * points, factor, dtype) // (2 if cplx else 1)


@pytest.mark.parametrize("N,L,tile", [(512, 12, 512), (1537, 0, 512), (2049, 202, 512), (408, 202, 512), (1000, 3, 256),
                                      (5000, 101, 1024), (2000, 202, 256)])
def test_impulse_groups_one_per_window(N, L, tile):
    """No window of 2L + 3 consecutive input points (circular) holds two impulses of one group."""
    pos = [0, 1, L, 2 * L + 1, tile - 1, tile, tile + 1, N - L - 1, N - 2, N - 1]
    groups = acc.impulse_groups(N, L, pos)
    assert sorted(p for g in groups for p in g) == sorted(set(p for p in pos if 0 <= p < N))
    for g in groups:
        marks = np.zeros(N, dtype=np.int64)
        marks[g] = 1
        c = np.concatenate([marks, marks[:2 * L + 2]]).cumsum()
        window_counts = c[2 * L + 2:2 * L + 2 + N] - np.concatenate([[0], c[:N - 1]])
        assert window_counts.max() <= 1, (N, L, g)
    with pytest.raises(AssertionError):
        acc.impulse_groups(2 * L + 3, L, [0])
