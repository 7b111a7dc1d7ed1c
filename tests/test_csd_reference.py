"""The CPU reference of bdsp_csd_* and bdsp_coherence_*, pinned without a GPU to scipy.signal.csd and scipy.signal.coherence.

closed_form() is the definition the GPU tests (test_gpu_csd.py) hold the library to, computed with the frame spectra in a
given complex type: X_f = DFT(w * frame f of x), Y_f likewise for y, frames as in test_welch_reference.closed_form.  Per
frame, Re and Im of conj(X_f) Y_f (and for coherence |X_f|^2 and |Y_f|^2) are formed with every product and sum rounded in
the real type of `ct`, and summed over the frames in frame order in that type; the scale and the final quotient are
applied in float64 or wider.
  csd:       out[k] = scale / frames * sum_f conj(X_f[k]) Y_f[k], welch's scale, F_SHIFT order and F_ONESIDED fold;
  coherence: out[k] = |sum_f conj(X_f[k]) Y_f[k]|^2 / (sum_f |X_f[k]|^2 sum_f |Y_f[k]|^2), unscaled, not doubled."""
import numpy as np
import pytest
import scipy.fft as sfft
import scipy.signal

from oracle import accuracy as acc
from oracle.accuracy import F_REAL_INPUT as REAL, F_SHIFT as SH
from test_welch_reference import F_ONESIDED, F_POWER_SPECTRUM, closed_form as welch_closed_form


def frame_sums(x, y, points, hop, w, flags, ct, coherence):
    """(sum Re, sum Im of conj(X) Y[, sum |X|^2, sum |Y|^2]) over the frames, in the real type of ct, and the real type"""
    rt = np.finfo(ct).dtype.type
    frames = 1 + (len(x) - points) // hop
    w = np.ones(points, dtype=rt) if w is None else np.asarray(w).astype(rt)

    def spectra(s):
        rows = np.lib.stride_tricks.sliding_window_view(np.asarray(s), points)[::hop][:frames]
        return sfft.fft((rows.astype(rt) if flags & REAL else rows.astype(ct)) * w, axis=-1)

    X, Y = spectra(x), spectra(y)
    sums = [np.zeros(points, dtype=rt) for _ in range(4 if coherence else 2)]
    for f in range(frames):   # in frame order, every product and sum rounded in rt
        xr, xi, yr, yi = X[f].real, X[f].imag, Y[f].real, Y[f].imag
        sums[0] += xr * yr + xi * yi
        sums[1] += xr * yi - xi * yr
        if coherence:
            sums[2] += xr * xr + xi * xi
            sums[3] += yr * yr + yi * yi
    return sums, w, frames, rt


def closed_form(x, y, points, hop, w, flags, fs, ct, coherence=False):
    """bdsp_csd_* (complex) or bdsp_coherence_* (real) over signals x and y (complex, or real with F_REAL_INPUT) with
    window values w (None: no window), the frame spectra computed in complex type `ct`."""
    sums, w, frames, rt = frame_sums(x, y, points, hop, w, flags, ct, coherence)
    wide = np.longdouble if rt == np.longdouble else np.float64
    if coherence:
        re, im, sxx, syy = (s.astype(wide) for s in sums)
        with np.errstate(invalid="ignore", divide="ignore"):
            out = (re * re + im * im) / (sxx * syy)
        if flags & F_ONESIDED:
            out = out[:points // 2 + 1].copy()
    else:
        ww = w.astype(wide)
        den = np.sum(ww) ** 2 if flags & F_POWER_SPECTRUM else wide(fs) * np.sum(ww * ww)
        scale = wide(frames) * den
        out = sums[0].astype(wide) / scale + 1j * (sums[1].astype(wide) / scale)
        if flags & F_ONESIDED:
            out = out[:points // 2 + 1].copy()
            out[1:points // 2 + (points % 2)] *= 2
    if flags & SH:
        out = np.roll(out, points // 2)
    return out


def scipy_csd(x, y, points, hop, w, flags, fs):
    _, p = scipy.signal.csd(x, y, fs=fs, window=w, nperseg=points, noverlap=points - hop, detrend=False,
                            return_onesided=bool(flags & F_ONESIDED), scaling="spectrum" if flags & F_POWER_SPECTRUM else "density",
                            average="mean")
    return np.fft.fftshift(p) if flags & SH else p


def correlated(rng, length, real):
    """x and y = a filtered x plus independent noise: coherence spread over (0, 1)"""
    x = rng.standard_normal(length)
    e = rng.standard_normal(length)
    if not real:
        x = x + 1j * rng.standard_normal(length)
        e = e + 1j * rng.standard_normal(length)
    y = np.convolve(x, [0.5, 1.0, -0.25, 0.125], mode="same") + 0.7 * e
    return x, y


def window(kind, points):
    # scipy's named windows are periodic: the library's symmetric table goes in as an array
    return acc.window(3 if kind is None else kind, points, np.float64)


CASES = [(points, hop) for points in (64, 63, 1024, 1000, 15) for hop in (points // 4 or 1, points // 2 + 1, points)]
CSD_FLAGS = [REAL, REAL | F_ONESIDED, REAL | F_POWER_SPECTRUM, REAL | F_ONESIDED | F_POWER_SPECTRUM, 0, SH, F_POWER_SPECTRUM | SH,
             REAL | SH]


@pytest.mark.parametrize("points,hop", CASES, ids=["%d-h%d" % c for c in CASES])
@pytest.mark.parametrize("flags", CSD_FLAGS)
@pytest.mark.parametrize("kind", [0, 1, 2, None])
def test_csd_closed_form_is_scipy_csd(points, hop, flags, kind):
    rng = np.random.default_rng(points * 131 + hop * 7 + flags + (kind or 5))
    x, y = correlated(rng, points + 9 * hop + hop // 2, flags & REAL)
    w = window(kind, points)
    got = closed_form(x, y, points, hop, None if kind is None else w, flags, 48000.0, np.complex128)
    want = scipy_csd(x, y, points, hop, w, flags, 48000.0)
    assert got.shape == want.shape == ((points // 2 + 1,) if flags & F_ONESIDED else (points,))
    assert np.max(np.abs(got - want)) <= 1e-13 * np.max(np.abs(want))


@pytest.mark.parametrize("points,hop", CASES, ids=["%d-h%d" % c for c in CASES])
@pytest.mark.parametrize("flags", [REAL | F_ONESIDED, 0, SH, REAL, REAL | SH])
@pytest.mark.parametrize("kind", [0, 1, 2, None])
def test_coherence_closed_form_is_scipy_coherence(points, hop, flags, kind):
    rng = np.random.default_rng(points * 17 + hop * 5 + flags + (kind or 5))
    x, y = correlated(rng, points + 9 * hop + hop // 2, flags & REAL)
    w = window(kind, points)
    got = closed_form(x, y, points, hop, None if kind is None else w, flags, 1.0, np.complex128, coherence=True)
    if flags & REAL and not flags & F_ONESIDED:
        # scipy.signal.coherence of a real signal is one-sided: the two-sided form from its csd and welch
        kw = dict(fs=1.0, window=w, nperseg=points, noverlap=points - hop, detrend=False, return_onesided=False)
        _, pxy = scipy.signal.csd(x, y, **kw)
        _, pxx = scipy.signal.welch(x, **kw)
        _, pyy = scipy.signal.welch(y, **kw)
        want = np.abs(pxy) ** 2 / (pxx * pyy)
    else:
        _, want = scipy.signal.coherence(x, y, fs=1.0, window=w, nperseg=points, noverlap=points - hop, detrend=False)
    if flags & SH:
        want = np.fft.fftshift(want)
    assert got.shape == want.shape == ((points // 2 + 1,) if flags & F_ONESIDED else (points,))
    assert np.all((got >= 0) & (got <= 1 + 1e-12))
    assert np.max(np.abs(got - want)) <= 1e-12


@pytest.mark.parametrize("ct", [np.complex64, np.complex128])
@pytest.mark.parametrize("flags", [REAL | F_ONESIDED | F_POWER_SPECTRUM, SH, REAL])
def test_csd_of_x_with_itself_is_welch(ct, flags):
    """the same products and sums as test_welch_reference.closed_form, in the same type: equal, with no imaginary part"""
    rng = np.random.default_rng(7 + flags)
    points, hop = 256, 96
    x, _ = correlated(rng, points + 20 * hop, flags & REAL)
    w = window(1, points)
    got = closed_form(x, x, points, hop, w, flags, 48000.0, ct)
    want = welch_closed_form(x, points, hop, w, flags, 48000.0, ct)
    assert np.array_equal(got.real, want) and np.all(got.imag == 0)
    assert np.array_equal(closed_form(x, x, points, hop, w, flags & ~F_POWER_SPECTRUM, 1.0, ct, coherence=True), np.ones(want.shape))


def test_coherence_of_a_silent_signal_is_nan():
    rng = np.random.default_rng(4)
    x = rng.standard_normal(1024)
    got = closed_form(x, np.zeros_like(x), 64, 32, None, REAL | F_ONESIDED, 1.0, np.complex128, coherence=True)
    assert np.all(np.isnan(got))
    assert np.all(closed_form(x, np.zeros_like(x), 64, 32, None, REAL | F_ONESIDED, 1.0, np.complex128) == 0)
