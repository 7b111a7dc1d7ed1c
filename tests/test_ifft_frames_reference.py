"""The CPU reference of bdsp_ifft_frames_* (inverse short-time transform by least-squares weighted overlap-add), checked
without a GPU against torch.istft(center=False) and against a numpy analysis -> synthesis round trip.

synthesis() is the definition the GPU tests (test_gpu_ifft_frames.py) hold the library to, computed in a given complex
type: y_f = ifft(X_f) / points (F_SHIFT: X_f ifft-shifted first), then out[t] = sum_f w[p] y_f[p] / sum_f w[p]^2 with
p = t - f * hop, over the frames that cover t in ascending f."""
import numpy as np
import pytest
import scipy.fft as sfft
import torch

from oracle import accuracy as acc
from oracle.accuracy import F_SHIFT as SH

F_REAL_OUTPUT = 16   # include/basic_dsp_b200.h
KINDS = (0, 1, 2, 3)   # triangular, Hamming, Blackman-Harris, rectangular


def synthesis(X, hop, kind, flags, ct, w=None):
    """bdsp_ifft_frames_* over the frames x points spectra X, computed in complex type `ct` (kind None: no window).
    w: the window values to use instead of evaluating `kind` in `ct`'s precision, e.g. the library's own table."""
    X = np.asarray(X)
    frames, n = X.shape
    rt = np.finfo(ct).dtype.type
    xc = X.astype(ct)
    if flags & SH:
        xc = np.roll(xc, -(n // 2), axis=-1)
    y = sfft.ifft(xc * (rt(1) / rt(n)), axis=-1, norm="forward")
    w = acc.window(3 if kind is None else kind, n, rt) if w is None else np.asarray(w).astype(rt)
    length = (frames - 1) * hop + n
    num = np.zeros(length, dtype=ct)
    den = np.zeros(length, dtype=rt)
    for f in range(frames):
        num[f * hop:f * hop + n] += w * y[f]
        den[f * hop:f * hop + n] += w * w
    out = num / den
    return out.real if flags & F_REAL_OUTPUT else out


def analysis(x, points, hop, kind, flags, ct):
    """bdsp_fft_frames_* (complex spectra) of x in complex type `ct`."""
    rt = np.finfo(ct).dtype.type
    frames = 1 + (len(x) - points) // hop
    rows = np.lib.stride_tricks.sliding_window_view(np.asarray(x), points)[::hop][:frames]
    X = sfft.fft(rows.astype(ct) * acc.window(kind, points, rt), axis=-1)
    return np.roll(X, points // 2, axis=-1) if flags & SH else X


def spectra(rng, frames, points):
    return rng.standard_normal((frames, points)) + 1j * rng.standard_normal((frames, points))


SHAPES = [(64, h, 9) for h in (1, 16, 31, 64)] + [(1024, 256, 12), (15, 4, 7), (16, 8, 1), (1000, 1000, 3)]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("points,hop,frames", SHAPES, ids=["%d-h%d-x%d" % s for s in SHAPES])
def test_synthesis_matches_torch_istft(points, hop, frames, kind):
    X = spectra(np.random.default_rng(points * 31 + hop + frames), frames, points)
    got = synthesis(X, hop, kind, 0, np.complex128)
    w = torch.from_numpy(acc.window(kind, points, np.float64))
    want = torch.istft(torch.from_numpy(X.T.copy()), n_fft=points, hop_length=hop, win_length=points, window=w, center=False,
                       normalized=False, onesided=False, return_complex=True).numpy()
    assert got.shape == want.shape == ((frames - 1) * hop + points,)
    assert np.max(np.abs(got - want)) <= 1e-13 * np.max(np.abs(want))


def test_shift_and_real_output():
    X = spectra(np.random.default_rng(5), 6, 32)
    plain = synthesis(X, 8, 1, 0, np.complex128)
    assert np.allclose(synthesis(np.roll(X, 16, axis=-1), 8, 1, SH, np.complex128), plain, rtol=0, atol=1e-15)
    assert np.array_equal(synthesis(X, 8, 1, F_REAL_OUTPUT, np.complex128), plain.real)


def test_one_frame_without_a_window_is_the_inverse_transform():
    X = spectra(np.random.default_rng(6), 1, 48)
    assert np.array_equal(synthesis(X, 48, None, SH, np.complex64), acc.transform(X, acc.F_INVERSE | SH, np.complex64)[0])


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("flags", [0, SH])
@pytest.mark.parametrize("points,hop", [(256, 64), (256, 127), (256, 256), (63, 20)])
def test_analysis_synthesis_round_trip(points, hop, kind, flags):
    rng = np.random.default_rng(points + hop + kind)
    x = rng.standard_normal(points + 10 * hop) + 1j * rng.standard_normal(points + 10 * hop)
    X = analysis(x, points, hop, kind, flags, np.complex128)
    back = synthesis(X, hop, kind, flags, np.complex128)
    assert back.shape == x[:back.size].shape
    # a sample that one frame covers is w y / w^2: its rounding grows by 1 / w, up to 1.7e4 at the Blackman-Harris ends
    assert np.max(np.abs(back - x[:back.size])) <= 1e-10
    real = synthesis(analysis(x.real, points, hop, kind, flags, np.complex128), hop, kind, flags | F_REAL_OUTPUT, np.complex128)
    assert np.max(np.abs(real - x.real[:real.size])) <= 1e-10
