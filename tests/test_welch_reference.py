"""The CPU reference of bdsp_welch_* (Welch's averaged periodogram), pinned without a GPU to scipy.signal.welch.

closed_form() is the definition the GPU tests (test_gpu_welch.py) hold the library to, computed with the frame spectra in
a given complex type: X_f = DFT(w * frame f), frame f = x[f*hop : f*hop + points]; out[k] = scale / frames * sum_f |X_f[k]|^2
with scale = 1 / (fs sum w^2) (density) or 1 / (sum w)^2 (F_POWER_SPECTRUM); F_SHIFT: fftshift order; F_ONESIDED: bins
0 .. points/2, all but bin 0 and the Nyquist bin of an even `points` doubled.  |X|^2 is formed and summed over the frames
(in frame order) in the real type of `ct`; the scale is applied in float64 or wider."""
import numpy as np
import pytest
import scipy.fft as sfft
import scipy.signal

from oracle import accuracy as acc
from oracle.accuracy import F_REAL_INPUT as REAL, F_SHIFT as SH

F_ONESIDED, F_POWER_SPECTRUM = 32, 64   # include/basic_dsp_b200.h


def closed_form(x, points, hop, w, flags, fs, ct):
    """bdsp_welch_* over signal x (complex, or real with F_REAL_INPUT) with window values w (None: no window), the frame
    spectra computed in complex type `ct`."""
    rt = np.finfo(ct).dtype.type
    wide = np.longdouble if rt == np.longdouble else np.float64
    frames = 1 + (len(x) - points) // hop
    rows = np.lib.stride_tricks.sliding_window_view(np.asarray(x), points)[::hop][:frames]
    w = np.ones(points, dtype=rt) if w is None else np.asarray(w).astype(rt)
    xr = rows.astype(rt) if flags & REAL else rows.astype(ct)
    X = sfft.fft(xr * w, axis=-1)
    p = np.zeros(points, dtype=rt)
    for f in range(frames):   # in frame order, rounded in rt
        p += X[f].real * X[f].real + X[f].imag * X[f].imag
    ww = w.astype(wide)
    den = np.sum(ww) ** 2 if flags & F_POWER_SPECTRUM else wide(fs) * np.sum(ww * ww)
    out = p.astype(wide) / (wide(frames) * den)
    if flags & F_ONESIDED:
        out = out[:points // 2 + 1].copy()
        out[1:points // 2 + (points % 2)] *= 2
    elif flags & SH:
        out = np.roll(out, points // 2)
    return out


def scipy_welch(x, points, hop, w, flags, fs):
    _, p = scipy.signal.welch(x, fs=fs, window=w, nperseg=points, noverlap=points - hop, detrend=False,
                              return_onesided=bool(flags & F_ONESIDED), scaling="spectrum" if flags & F_POWER_SPECTRUM else "density",
                              average="mean")
    return np.fft.fftshift(p) if flags & SH else p


CASES = [(points, hop) for points in (64, 63, 1024, 1000, 15) for hop in (points // 4 or 1, points // 2 + 1, points)]


@pytest.mark.parametrize("points,hop", CASES, ids=["%d-h%d" % c for c in CASES])
@pytest.mark.parametrize("flags", [REAL, REAL | F_ONESIDED, REAL | F_POWER_SPECTRUM, REAL | F_ONESIDED | F_POWER_SPECTRUM, 0, SH,
                                   F_POWER_SPECTRUM | SH])
@pytest.mark.parametrize("kind", [0, 1, 2, None])
def test_closed_form_is_scipy_welch(points, hop, flags, kind):
    rng = np.random.default_rng(points * 131 + hop * 7 + flags + (kind or 5))
    length = points + 9 * hop + hop // 2
    x = rng.standard_normal(length)
    if not flags & REAL:
        x = x + 1j * rng.standard_normal(length)
    # scipy's named windows are periodic: the library's symmetric table goes in as an array
    w = acc.window(3 if kind is None else kind, points, np.float64)
    fs = 48000.0
    got = closed_form(x, points, hop, None if kind is None else w, flags, fs, np.complex128)
    want = scipy_welch(x, points, hop, w, flags, fs)
    assert got.shape == want.shape == ((points // 2 + 1,) if flags & F_ONESIDED else (points,))
    assert np.max(np.abs(got - want)) <= 1e-13 * np.max(np.abs(want))


def test_hop_above_points_skips_samples():
    """scipy.signal.welch takes no hop > nperseg: the closed form over spaced frames is the mean of the periodograms."""
    rng = np.random.default_rng(3)
    points, hop, frames = 32, 45, 7
    x = rng.standard_normal((frames - 1) * hop + points)
    got = closed_form(x, points, hop, None, REAL | F_POWER_SPECTRUM, 1.0, np.complex128)
    rows = [x[f * hop:f * hop + points] for f in range(frames)]
    want = np.mean([np.abs(np.fft.fft(r)) ** 2 for r in rows], axis=0) / points ** 2
    assert np.max(np.abs(got - want)) <= 1e-14 * np.max(want)

