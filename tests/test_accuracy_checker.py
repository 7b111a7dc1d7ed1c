"""The per-element, peer-relative checker (oracle/accuracy.py) passes correct same-precision results and catches faults
that BASELINE's relative-L2 tolerance lets through.  CPU only: the "GPU results" here are the peers' own outputs, with
and without injected faults."""
import numpy as np
import pytest

from oracle import accuracy as acc


def rand_c(rng, shape, dtype):
    ct = acc.ctype(dtype)
    return (rng.uniform(-10, 10, shape) + 1j * rng.uniform(-10, 10, shape)).astype(ct)


def baseline_passes(got, ref, n, dtype):
    """The assertion the GPU suite has used so far: relative L2 of the whole vector against BASELINE."""
    g = np.asarray(got).astype(np.complex128).ravel()
    r = np.asarray(ref).astype(np.complex128).ravel()
    return np.linalg.norm(g - r) / np.linalg.norm(r) <= acc.baseline_tol(n, dtype)


def fails(got, ref, peer, dtype, **kw):
    with pytest.raises(acc.AccuracyError):
        acc.check(got, ref, peer, dtype, **kw)
    return True


# ---- correct results pass ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("flags", [0, acc.F_SHIFT, acc.F_INVERSE, acc.F_INVERSE | acc.F_SHIFT, acc.F_SHIFT | acc.F_MAGNITUDE,
                                   acc.F_REAL_INPUT])
@pytest.mark.parametrize("n,rows", [(1024, 3), (3000, 2), (10007, 1)])
def test_peer_transform_passes(n, rows, flags, dtype):
    rng = np.random.default_rng(n + flags)
    x = rand_c(rng, (rows, n), dtype)
    if flags & acc.F_REAL_INPUT:
        x = np.ascontiguousarray(x.real)
    ref, peer = acc.fft_pair(x, flags, dtype)
    rec = acc.check(peer, ref, peer, dtype, path="peer")
    assert rec["rows"] == rows and rec["rel_ratio"] == 1.0 and rec["el_ratio"] == 1.0


def test_windowed_peer_passes():
    rng = np.random.default_rng(3)
    x = rand_c(rng, (2, 4096), np.float32)
    ref = acc.windowed_transform(x, 2, np.complex128)
    peer = acc.windowed_transform(x, 2, np.complex64)
    acc.check(peer, ref, peer, np.float32)
    assert acc.metrics(peer, ref)[0][0] < 1e-6


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,rows,L", [(5000, 2, 30), (20000, 1, 1023), (9000, 3, 2046), (40000, 1, 3000), (3000, 2, 100)])
def test_ols_peer_matches_reference(n, rows, L, dtype):
    """The block overlap-save peer computes the centred circular convolution, in both block geometries, with the error
    of a same-precision transform; the FIR peer too."""
    rng = np.random.default_rng(n + L)
    x = rand_c(rng, (rows, n), dtype)
    h = (rand_c(rng, L, dtype) / 10).astype(x.dtype)
    ref = acc.conv_ref(x, h, dtype)
    for M in (4096, 8192):
        if L > M // 2 - 2:
            continue
        for geo in ("generic", "olsi"):
            peer = acc.ols_peer(x, h, dtype, M, geo)
            rec = acc.check(peer, ref, peer, dtype)
            assert rec["rel_gpu"] < 50 * acc.unit_roundoff(dtype), (M, geo, rec)
    xr = np.ascontiguousarray(x.real)
    hr = np.ascontiguousarray(h.real)
    peer_r = acc.ols_peer(xr, hr, dtype, 4096 if L <= 1024 else 8192)
    assert peer_r.dtype == np.dtype(dtype)
    assert acc.metrics(peer_r, acc.conv_ref(xr, hr, dtype))[0][0] < 50 * acc.unit_roundoff(dtype)
    if L <= 30:
        fp = acc.fir_peer(x, h, dtype)
        assert fp.dtype == x.dtype
        assert max(r for r, _ in acc.metrics(fp, ref)) < 50 * acc.unit_roundoff(dtype)


def test_ols_block_choice_mirrors_conv_cu():
    f32, f64 = np.float32, np.float64
    assert acc.ols_block(f32, 1023, True, 1 << 20, 1) == (4096, "olsi")
    assert acc.ols_block(f32, 1450, True, 1 << 22, 1) == (8192, "olsi")        # >= 592 blocks of 8192 points
    assert acc.ols_block(f32, 1450, True, 100000, 1) == (4096, "olsi")         # fewer blocks: 4096-point blocks
    assert acc.ols_block(f32, 1449, True, 1 << 22, 1) == (4096, "olsi")
    assert acc.ols_block(f32, 3000, True, 20000, 1) == (8192, "olsi")
    assert acc.ols_block(f32, 3000, True, 6000, 1) == (8192, "generic")
    assert acc.ols_block(f32, 1000, True, 3000, 4) == (4096, "generic")
    assert acc.ols_block(f32, 1000, False, 30000, 1) == (4096, "generic")
    assert acc.ols_block(f32, 1100, False, 30000, 1) == (8192, "generic")
    assert acc.ols_block(f64, 2048, True, 5000, 1) == (4096, "generic")
    assert acc.ols_block(f64, 3000, True, 50000, 1) == (8192, "generic")
    assert acc.ols_block(f32, 5000, True, 50000, 1) == (16384, "generic")
    assert acc.olsi_geometry(4096, 1023) == (1, 1024, 3072)


# ---- the u_T floor -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [1, 2])
def test_tiny_transform_exact_peer(n, dtype):
    """Integer inputs of length 1 and 2: the peer is exact (error 0), so the bounds fall back to K * u_T."""
    x = np.array([[3 - 5j, -7 + 2j][:n]], dtype=acc.ctype(dtype))
    ref, peer = acc.fft_pair(x, 0, dtype)
    assert acc.metrics(peer, ref)[0] == (0.0, 0.0)
    acc.check(peer, ref, peer, dtype)
    u = acc.unit_roundoff(dtype)
    one_ulp = peer * (1 + 2 * u)
    acc.check(one_ulp, ref, peer, dtype)                      # one rounding step: within K * u_T
    fails(peer * (1 + 100 * u), ref, peer, dtype)             # 100 u_T: not


# ---- faults that pass BASELINE and fail the peer-relative check ------------------------------------------------------
def test_fault_two_wrong_bins():
    """DC and Nyquist bins of a 2^20-point f32 FFT 10 % off (a packing or shift bug of a real-input or F_SHIFT epilogue)."""
    n = 1 << 20
    x = rand_c(np.random.default_rng(1), (1, n), np.float32)
    ref, peer = acc.fft_pair(x, 0, np.float32)
    bad = peer.copy()
    bad[0, 0] *= np.float32(1.1)
    bad[0, n // 2] *= np.float32(1.1)
    assert baseline_passes(bad, ref, n, np.float32)
    assert fails(bad, ref, peer, np.float32)


def _fft_radix2(x, twiddle_err, rng):
    """Iterative radix-2 decimation-in-time FFT in complex64 whose twiddles carry a relative error of `twiddle_err`."""
    n = x.shape[-1]
    bits = n.bit_length() - 1
    rev = np.zeros(n, dtype=np.int64)
    for b in range(bits):
        rev |= ((np.arange(n) >> b) & 1) << (bits - 1 - b)
    a = x[..., rev].astype(np.complex64)
    half = 1
    while half < n:
        w = np.exp(-2j * np.pi * np.arange(half) / (2 * half))
        w = w * (1 + twiddle_err * np.exp(2j * np.pi * rng.uniform(0, 1, half)))
        w = w.astype(np.complex64)
        a = a.reshape(a.shape[:-1] + (n // (2 * half), 2, half))
        t = a[..., 1, :] * w
        a = np.concatenate([a[..., 0, :] + t, a[..., 0, :] - t], axis=-1).reshape(x.shape)
        half *= 2
    return a


def test_fault_imprecise_twiddles():
    """A 2^16-point f32 FFT whose twiddles each carry a 2e-5 relative error (~300 ulp: a degraded table or a product
    chain that is not re-anchored)."""
    n = 1 << 16
    rng = np.random.default_rng(2)
    x = rand_c(rng, (1, n), np.float32)
    ref, peer = acc.fft_pair(x, 0, np.float32)
    good = _fft_radix2(x, 0.0, rng)
    acc.check(good, ref, peer, np.float32)                     # exact twiddles (rounded to f32): a correct f32 FFT
    bad = _fft_radix2(x, 2e-5, rng)
    assert baseline_passes(bad, ref, n, np.float32)
    assert fails(bad, ref, peer, np.float32)


def _ols_case():
    rng = np.random.default_rng(4)
    n, L = 1 << 20, 1023
    x = rand_c(rng, (1, n), np.float32)
    h = (rand_c(rng, L, np.float32) / 10).astype(np.complex64)
    M, geo = acc.ols_block(np.float32, L, True, n, 1)
    return n, L, acc.conv_ref(x, h, np.float32), acc.ols_peer(x, h, np.float32, M, geo), acc.olsi_geometry(M, L)[2]


def test_fault_one_bad_output_per_block():
    """Overlap-save of 2^20 points with 1023 taps whose last output of every block is 1 % off (an off-by-one at the block
    boundary of the fused 4096-point kernel)."""
    n, L, ref, peer, step = _ols_case()
    acc.check(peer, ref, peer, np.float32)
    bad = peer.copy()
    bad[0, step - 1::step] *= np.float32(1.01)
    assert baseline_passes(bad, ref, n, np.float32)
    assert fails(bad, ref, peer, np.float32)


def test_fault_bad_tail_block():
    """The same convolution with the last 700 outputs (the partial tail block) 0.5 % off."""
    n, L, ref, peer, step = _ols_case()
    bad = peer.copy()
    bad[0, -700:] *= np.float32(1.005)
    assert baseline_passes(bad, ref, n, np.float32)
    assert fails(bad, ref, peer, np.float32)


def test_every_row_is_checked():
    """A fault in one row of a batch is not averaged away by the others."""
    rng = np.random.default_rng(5)
    x = rand_c(rng, (16, 4096), np.float32)
    ref, peer = acc.fft_pair(x, acc.F_SHIFT, np.float32)
    bad = peer.copy()
    bad[15, 100] += np.float32(20 * np.sqrt(np.mean(np.abs(ref[15]) ** 2)) * 1e-4)
    assert baseline_passes(bad, ref, 4096, np.float32)
    with pytest.raises(acc.AccuracyError, match="row 15"):
        acc.check(bad, ref, peer, np.float32)


def test_factor_cap():
    x = rand_c(np.random.default_rng(6), (1, 64), np.float32)
    ref, peer = acc.fft_pair(x, 0, np.float32)
    with pytest.raises(AssertionError, match="capped"):
        acc.check(peer, ref, peer, np.float32, k_el=32)
