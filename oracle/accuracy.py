"""Per-element accuracy checks of the FFT and convolution kernels against same-precision CPU peers (test-only code).

BASELINE's tolerance (relative L2 error <= 1e-5 log2 N for f32, 1e-12 log2 N for f64) is the contract with users, but it
leaves two to three orders of magnitude of room above what a correct transform in that precision achieves, so a kernel
that gets a few bins, a block boundary or its twiddles wrong can still pass it.  `check` therefore compares every row of
a GPU result with
  * a reference: the same operation in higher precision (complex128 for f32 results, the platform's long double through
    scipy.fft for f64 results; 80-bit extended on x86-64), and
  * a peer: the same operation computed on the CPU in the kernel's own precision (scipy.fft computes in its input's
    precision; the overlap-save peer uses the kernel's block length and block geometry),
and asserts that the GPU's error is within a small factor of the peer's error, both for the whole row (`rel`) and for its
worst element (`elmax`, relative to the row's RMS).
"""
import ctypes
import ctypes.util
import math

import numpy as np
import scipy.fft as sfft

F_INVERSE, F_SHIFT, F_MAGNITUDE, F_REAL_INPUT = 1, 2, 4, 8   # bdsp_fft_rows_* flags (include/basic_dsp_b200.h)

K_REL = 4.0
K_EL = 8.0
K_MAX = 16.0   # largest per-path factor a test may use, with the measured cause written next to it


def unit_roundoff(dtype):
    return float(np.finfo(dtype).eps) / 2


def baseline_tol(n, dtype):
    """BASELINE.md's relative L2 tolerance for a result of length n."""
    return (1e-5 if dtype == np.float32 else 1e-12) * max(1.0, math.log2(max(n, 2)))


def ctype(dtype):
    return np.complex64 if dtype == np.float32 else np.complex128


def ref_ctype(dtype):
    """Complex type of the reference computation for results in `dtype`."""
    return np.complex128 if dtype == np.float32 else np.clongdouble


def ref_rtype(dtype):
    return np.float64 if dtype == np.float32 else np.longdouble


# ---- metrics -------------------------------------------------------------------------------------------------------
def _rows(a):
    a = np.asarray(a)
    return a.reshape(1, -1) if a.ndim == 1 else a


def metrics(got, ref):
    """Per row: (rel, elmax) of `got` against `ref`, evaluated in the reference's precision."""
    g = _rows(got)
    r = _rows(ref)
    hi = np.clongdouble if r.dtype in (np.clongdouble, np.longdouble) else np.complex128
    out = []
    for gr, rr in zip(g, r):
        rr = rr.astype(hi)
        d = np.abs(gr.astype(hi) - rr)
        nref = np.sqrt(np.sum(np.abs(rr) ** 2))
        nd = np.sqrt(np.sum(d ** 2))
        rms = nref / np.sqrt(max(len(rr), 1))
        if nref > 0:
            out.append((float(nd / nref), float(np.max(d) / rms) if len(d) else 0.0))
        else:
            out.append((float(nd), float(np.max(d)) if len(d) else 0.0))
    return out


class AccuracyError(AssertionError):
    pass


def check(got, ref, peer, dtype, *, path="", k_rel=K_REL, k_el=K_EL, tol_n=None):
    """Asserts, for every row of `got` (1-D: one row; 2-D: rows x points):
         rel_gpu   <= k_rel * max(rel_peer, u_T)
         elmax_gpu <= k_el  * max(elmax_peer, u_T)
         rel_gpu   <= BASELINE tolerance (length `tol_n`, default the row length)
    and returns a record of the worst row for the report (path, n, rows, both metrics of GPU and peer, their ratios)."""
    assert k_rel <= K_MAX and k_el <= K_MAX, "per-path factors are capped at %g" % K_MAX
    g, r, p = _rows(got), _rows(ref), _rows(peer)
    assert g.shape == r.shape == p.shape, (g.shape, r.shape, p.shape)
    rows, n = g.shape
    u = unit_roundoff(dtype)
    tol = baseline_tol(tol_n if tol_n is not None else n, dtype)
    mg, mp = metrics(g, r), metrics(p, r)
    rec, worst = None, -1.0
    bad = []
    for i, ((rg, eg), (rp, ep)) in enumerate(zip(mg, mp)):
        rr, er = rg / max(rp, u), eg / max(ep, u)
        if max(rr / k_rel, er / k_el) > worst:   # the record shows the row closest to its bounds
            worst = max(rr / k_rel, er / k_el)
            rec = {"path": path, "n": n, "rows": rows, "row": i, "rel_gpu": rg, "rel_peer": rp, "elmax_gpu": eg,
                   "elmax_peer": ep, "rel_ratio": rr, "el_ratio": er}
        if not (rr <= k_rel and er <= k_el and rg <= tol):
            bad.append("row %d: rel %.3g (peer %.3g, x%.1f > %g?) elmax %.3g (peer %.3g, x%.1f > %g?) baseline %.3g"
                       % (i, rg, rp, rr, k_rel, eg, ep, er, k_el, tol))
    if bad:
        raise AccuracyError("%s n=%d rows=%d: %s" % (path, n, rows, "; ".join(bad[:4]) + (" ..." if len(bad) > 4 else "")))
    return rec


def format_record(rec):
    return ("%-44s n=%-9d rows=%-4d (worst row %d) rel gpu %.2e peer %.2e (x%5.2f)  elmax gpu %.2e peer %.2e (x%5.2f)"
            % (rec["path"], rec["n"], rec["rows"], rec["row"], rec["rel_gpu"], rec["rel_peer"], rec["rel_ratio"],
               rec["elmax_gpu"], rec["elmax_peer"], rec["el_ratio"]))


# ---- transforms ------------------------------------------------------------------------------------------------------
def transform(x, flags, ct):
    """bdsp_fft_rows semantics over the last axis, computed by scipy.fft in complex type `ct` (every operation, including
    the 1/n of the shifted inverse, is rounded to that precision).  x: complex rows, or real rows with F_REAL_INPUT."""
    x = np.asarray(x)
    rt = np.finfo(ct).dtype.type
    xc = x.astype(rt) if flags & F_REAL_INPUT else x.astype(ct)
    n = x.shape[-1]
    if flags & F_INVERSE:
        if flags & F_SHIFT:
            xc = np.roll(xc, -(n // 2), axis=-1) * (rt(1) / rt(n))
        y = sfft.ifft(xc, axis=-1, norm="forward")
    else:
        y = sfft.fft(xc, axis=-1)
        if flags & F_SHIFT:
            y = np.roll(y, n // 2, axis=-1)
    if flags & F_MAGNITUDE:
        y = np.abs(y)
    return y


def window(kind, n, rt):
    """Symmetric built-in window (window_functions.rs; mirror indices as multiply_window_priv), evaluated in `rt`."""
    i = np.arange(n)
    j = np.where(i < (n + 1) // 2, i, n - 1 - i).astype(rt)
    one, two, pi = rt(1), rt(2), rt(math.pi) if rt != np.longdouble else np.longdouble("3.14159265358979323846264338327950288")
    den = rt(n) - one
    if kind == 0:
        return one - np.abs((j - (rt(n) - one) / two) / (rt(n) / two))
    if kind == 1:
        return rt(0.54) - (one - rt(0.54)) * np.cos(two * pi * j / den)
    if kind == 2:
        return (rt(0.35875) - rt(0.48829) * np.cos(two * pi * j / den) + rt(0.14128) * np.cos(rt(4) * pi * j / den)
                - rt(0.01168) * np.cos(rt(6) * pi * j / den))
    return np.ones(n, dtype=rt)


def windowed_transform(x, kind, ct):
    """F_SHIFT | F_WINDOW(kind): the window applied and the transform computed in `ct`'s precision."""
    rt = np.finfo(ct).dtype.type
    w = window(kind, np.asarray(x).shape[-1], rt)
    return transform(np.asarray(x).astype(ct) * w, F_SHIFT, ct)


def fft_pair(x, flags, dtype):
    """(reference, peer) of bdsp_fft_rows for results in `dtype`."""
    return transform(x, flags, ref_ctype(dtype)), transform(x, flags, ctype(dtype))


# ---- convolution -----------------------------------------------------------------------------------------------------
def conv_full(x, h, ct):
    """Centred circular convolution y[i] = sum_k x[(i + cl - 1 - k) mod N] h[k] (cl = L - L/2) of every row through its
    FFT identity, computed in `ct`."""
    x = np.asarray(x)
    N, L = x.shape[-1], len(h)
    cl = L - L // 2
    hp = np.zeros(N, dtype=ct)
    hp[:L] = np.asarray(h).astype(ct)
    hp = np.roll(hp, -(cl - 1))
    y = sfft.ifft(sfft.fft(x.astype(ct), axis=-1) * sfft.fft(hp), axis=-1)
    return y if np.iscomplexobj(x) or np.iscomplexobj(h) else y.real


def conv_ref(x, h, dtype):
    return conv_full(x, h, ref_ctype(dtype))


def fir_peer(x, h, dtype):
    """Direct circular FIR accumulated in `dtype`, tap by tap."""
    x = np.asarray(x)
    cplx = np.iscomplexobj(x) or np.iscomplexobj(h)
    t = ctype(dtype) if cplx else dtype
    xt, ht = x.astype(t), np.asarray(h).astype(t)
    N, L = x.shape[-1], len(h)
    cl = L - L // 2
    idx = np.arange(N)
    y = np.zeros(x.shape, dtype=t)
    for k in range(L - 1, -1, -1):
        y += xt[..., (idx + cl - 1 - k) % N] * ht[k]
    return y


def olsi_geometry(M, L):
    """(d, m_first, step) of the fused c32 block kernels (olsi.cuh): a delay d folded into the spectrum makes the
    input-to-output distance even; block positions m_first .. m_first + step - 1 are valid outputs."""
    cl = L - L // 2
    d = (cl - 1) & 1
    mf = L - 1 + d
    mf += mf & 1
    return d, mf, (M - mf) & ~1


def ols_peer(x, h, dtype, M, geometry="generic"):
    """Block overlap-save in `dtype` with M-point blocks: block b covers outputs b*step .. b*step + step - 1, the
    spectrum of the (delayed) taps carries the 1/M of the inverse, as in the kernels.  geometry: "generic" (d = 0,
    step = M - L + 1; ols_conv_kernel, ols64) or "olsi" (ols4096i / ols8192i)."""
    x = np.asarray(x)
    real = not np.iscomplexobj(x)
    ct = ctype(dtype)
    rt = np.dtype(dtype).type
    N, L = x.shape[-1], len(h)
    cl = L - L // 2
    if geometry == "olsi":
        d, first, step = olsi_geometry(M, L)
    else:
        d, first, step = 0, L - 1, M - L + 1
    hp = np.zeros(M, dtype=ct)
    hp[d:d + L] = np.asarray(h).astype(ct)
    H = sfft.fft(hp) * rt(1.0 / M)
    nb = -(-N // step)
    i0 = np.arange(nb) * step
    p0 = i0 + cl - 1 + d - first
    idx = (p0[:, None] + np.arange(M)[None, :]) % N                    # blocks x M input indices
    seg = x.astype(rt if real else ct)[..., idx].astype(ct)
    y = sfft.ifft(sfft.fft(seg, axis=-1) * H, axis=-1, norm="forward")[..., first:first + step]
    y = y.reshape(x.shape[:-1] + (nb * step,))[..., :N]
    return y.real if real else y


def ols_block(dtype, L, complex_signal, N, rows):
    """(M, geometry) of the block overlap-save path conv.cu takes for these arguments (ols_block_len and the
    8192-point choice of convolve); None where a FIR or the full-length path runs instead."""
    c32 = dtype == np.float32 and complex_signal
    if c32 and 2 <= L <= 2046:
        blocks8 = -(-N // olsi_geometry(8192, L)[2]) if L <= 4094 else 0
        if N >= 8192 and L >= 1450 and blocks8 * rows >= 592:
            return 8192, "olsi"
        return (4096, "olsi") if N >= 4096 else (4096, "generic")
    if c32 and 2 <= L <= 4094:
        return (8192, "olsi") if N >= 8192 else (8192, "generic")
    if dtype == np.float64 and complex_signal and L <= 2048:
        return 4096, "generic"
    m = 1
    while m < 4 * max(L - 1, 1):
        m *= 2
    return min(max(m, 4096), 16384 if dtype == np.float32 else 8192), "generic"


# ---- interpolation ---------------------------------------------------------------------------------------------------
# interpolatef (dsp_oracle.interpolatef's formulas) with every output written as a sum over a window of 2L + 1 input
# points in ascending order, y[i] = sum_k x[(start_i + k) mod N] * taps_i[k]:
#   * polyphase path (integer factor F): the taps are the host-built tables in T, edge outputs (the first and last
#     (2L + 1) F) start at i // F - L + 1 with v_s, s = i % F; interior outputs at ceil(i / F) - L - 1 with v_s reversed,
#     s = (F - i % F) % F;
#   * per-output path: start floor(i / F) - L, taps f(j + k) with j = -L - frac + delay, all in T.
# The reference accumulates in float64 (f32 results) or long double (f64 results), the peer in T, tap by tap.
_LIBM = None


def _libm():
    global _LIBM
    if _LIBM is None:
        _LIBM = ctypes.CDLL(ctypes.util.find_library("m"))
        for name in ("sinf", "cosf"):
            getattr(_LIBM, name).restype = ctypes.c_float
            getattr(_LIBM, name).argtypes = [ctypes.c_float]
    return _LIBM


def impulse(kind, rolloff, dtype):
    """Built-in impulse response (0 Sinc, else RaisedCosine(rolloff)) as the library's host code evaluates it (capi.cu
    host_sinc / host_rc): every operation rounded to `dtype`, sin and cos from the C library.  numpy's float32 sin is not
    sinf: it differs in the last bit for about one argument in six, and the polyphase tables must match bit for bit."""
    T = np.dtype(dtype).type
    sin, cos = (_libm().sinf, _libm().cosf) if T == np.float32 else (math.sin, math.cos)
    one, two, pi, r = T(1), T(2), T(math.pi), T(rolloff)

    def f(x):
        x = T(x)
        if x == 0:
            return one
        if kind == 0:
            px = pi * x
            return T(sin(px)) / px
        if abs(x) == one / (two * r):
            arg = pi / two / r
            return T(sin(arg)) / arg * pi / (two * two)
        px = pi * x
        arg = two * r * x
        return T(sin(px)) * T(cos(px * r)) / px / (one - arg * arg)
    return f


def impulse_vec(kind, rolloff, x, dtype):
    """The same function over an array, in `dtype` with numpy's sin and cos (for the per-output path, whose kernel
    evaluates its taps on the device)."""
    T = np.dtype(dtype).type
    x = np.asarray(x, dtype=T)
    one, two, pi, r = T(1), T(2), T(math.pi), T(rolloff)
    with np.errstate(divide="ignore", invalid="ignore"):
        px = pi * x
        if kind == 0:
            y = np.sin(px) / px
        else:
            arg = two * r * x
            y = np.sin(px) * np.cos(px * r) / px / (one - arg * arg)
            a = pi / two / r
            y = np.where(np.abs(x) == one / (two * r), np.sin(a) / a * pi / (two * two), y)
        return np.where(x == 0, one, y).astype(T)


def interpf_windows(x_points, len_T, kind, rolloff, factor, delay, conv_len, dtype):
    """(new_points, poly, start, taps) of interpolatef on a vector of x_points points (len_T scalars): start[i] is the
    first input index of output i's window, taps[i] its 2L + 1 taps in ascending window order, in `dtype`."""
    from oracle import dsp_oracle as o
    T = np.dtype(dtype).type
    N = x_points
    L = min(conv_len, N // 2)
    new_len = o.interpolatef_new_len(len_T, factor, dtype)
    new_points = new_len // 2 if len_T == 2 * N else new_len
    i = np.arange(new_points)
    if o.interpolatef_uses_fast_path(L, new_len, factor, dtype):
        F = int(np.round(T(factor)))
        vs = o.interpolatef_tap_vectors(impulse(kind, rolloff, dtype), L, F, delay, dtype)
        scalar_len = (2 * L + 1) * F
        interior = (i >= scalar_len) & (i < new_points - scalar_len)
        start = np.where(interior, -(-i // F) - L - 1, i // F - L + 1)
        taps = np.where(interior[:, None], vs[(F - i % F) % F][:, ::-1], vs[i % F])
        return new_points, True, start, taps
    center = i.astype(T) / T(factor)
    rounded = np.floor(center)
    j = (-T(L) - (center - rounded)) + T(delay)
    taps = np.empty((new_points, 2 * L + 1), dtype=T)
    for k in range(2 * L + 1):
        taps[:, k] = impulse_vec(kind, rolloff, j, dtype)
        j = (j + T(1)).astype(T)
    return new_points, False, rounded.astype(np.int64) - L, taps


def interp_sum(x, start, taps, rt):
    """y[i] = sum_k x[(start[i] + k) mod N] * taps[i, k], accumulated in real type `rt` (complex x: its complex type),
    k ascending, every product and sum rounded to it."""
    x = np.asarray(x)
    ct = np.complex128 if rt == np.float64 else np.clongdouble if rt == np.longdouble else ctype(rt)
    xx = x.astype(ct if np.iscomplexobj(x) else rt)
    tt = np.asarray(taps).astype(rt)
    N = len(xx)
    acc = np.zeros(len(start), dtype=xx.dtype)
    for k in range(tt.shape[1]):
        acc += xx[(start + k) % N] * tt[:, k]
    return acc


def interpf_pair(x, kind, rolloff, factor, delay, conv_len, dtype):
    """(reference, peer) of interpolatef (delta 1) for results in `dtype`, and whether the polyphase path applies."""
    x = np.asarray(x)
    n, poly, start, taps = interpf_windows(len(x), (2 if np.iscomplexobj(x) else 1) * len(x), kind, rolloff, factor,
                                           delay, conv_len, dtype)
    return interp_sum(x, start, taps, ref_rtype(dtype)), interp_sum(x, start, taps, dtype), poly


def impulse_groups(N, L, positions):
    """Splits impulse positions into groups whose members are at least 2L + 4 apart circularly, so that no window of
    2L + 3 consecutive input points (the polyphase kernels' window superset [r - L - 1, r + L + 1]) holds two of them.
    Needs N >= 2L + 4: a shorter vector puts one impulse twice into a window."""
    assert N >= 2 * L + 4, (N, L)
    groups = []
    for p in sorted(set(q for q in positions if 0 <= q < N)):
        for g in groups:
            if all(min(abs(p - q), N - abs(p - q)) >= 2 * L + 4 for q in g):
                g.append(p)
                break
        else:
            groups.append([p])
    return groups
