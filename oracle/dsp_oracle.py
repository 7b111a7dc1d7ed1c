"""CPU oracle for the basic_dsp FFT-centred vector hot path.  TEST INFRASTRUCTURE ONLY.

This module restates, in NumPy, the *semantics* of the reference (liebharc/basic_dsp v0.10.0)
for the hot path named in BASELINE.json.  It is the checker for the CUDA kernels; it is never
imported by the product (`basic_dsp_b200/`).  Only `tests/`, `__graft_entry__.smoke()` and
`bench.py`'s cpu_baseline / `--impl reference` legs may import it.

Parity status: PINNED.  `tests/test_oracle_golden.py` checks every function below against the
known-answer vectors the reference's own tests hold (tests/golden/reference_kats.json, extracted by
tests/golden/extract_goldens.py from the reference sources).

The FFT arithmetic of the reference lives in the un-vendored third-party crate `rustfft ^6.0.0`
(vector/Cargo.toml:40; no Cargo.lock).  rustfft computes the plain unnormalised DFT
X[k] = sum_n x[n] exp(-+2 pi i n k / N); this oracle evaluates that definition with NumPy's
pocketfft in complex128, which is exact to ~1e-15 relative and therefore a valid stand-in at the
tolerances of BASELINE.json (rel-L2 <= 1e-5*log2 N for f32, 1e-12*log2 N for f64).

All file:line citations are relative to the reference tree (/root/reference in the build container).
Conventions: vectors are complex NumPy arrays (one element per point) or real arrays; `dtype`
(np.float32 / np.float64) is the precision `T` in which the reference evaluates taps and indices.
Accumulations are carried out in float64/complex128 so that the oracle is the mathematically exact
answer the reference approximates in precision T.
"""
from __future__ import annotations

import math

import numpy as np

# --------------------------------------------------------------------------------------------
# Error codes of the C ABI (interop/src/lib.rs:125-151)
# --------------------------------------------------------------------------------------------
ERR_OK = 0
ERR_VECTOR_INVALID = -1
ERR_SAME_SIZE = 1
ERR_META_DATA = 2
ERR_MUST_BE_COMPLEX = 3
ERR_MUST_BE_REAL = 4
ERR_MUST_BE_TIME = 5
ERR_MUST_BE_FREQ = 6
ERR_INVALID_ARG_LEN = 7
CONVERT_VOID_OK = 9  # interop/src/lib.rs:100-105 (quirk Q8)


# --------------------------------------------------------------------------------------------
# Impulse / frequency responses, evaluated in precision T  (conv_types.rs:391-518)
# --------------------------------------------------------------------------------------------
def _T(dtype):
    return np.dtype(dtype).type


def raised_cosine_impulse(x, rolloff, dtype=np.float64):
    """RaisedCosineFunction as RealImpulseResponse::calc, conv_types.rs:406-423."""
    T = _T(dtype)
    x = T(x)
    rolloff = T(rolloff)
    if x == T(0):
        return T(1)
    one, two = T(1), T(2)
    pi = T(math.pi)
    four = two * two
    if abs(x) == one / (two * rolloff):
        arg = pi / two / rolloff
        return T(np.sin(arg) / arg * pi / four)
    pi_x = pi * x
    arg = two * rolloff * x
    return T(np.sin(pi_x) * np.cos(pi_x * rolloff) / pi_x / (one - (arg * arg)))


def raised_cosine_freq(x, rolloff, dtype=np.float64):
    """RaisedCosineFunction as RealFrequencyResponse::calc, conv_types.rs:434-449."""
    T = _T(dtype)
    x = T(x)
    rolloff = T(rolloff)
    one, two = T(1), T(2)
    pi = T(math.pi)
    ax = abs(x)
    if ax <= (one - rolloff):
        return one
    if (one - rolloff) < ax <= (one + rolloff):
        return T(one / two * (one + np.cos(pi / rolloff * (ax - (one - rolloff)) / two)))
    return T(0)


def sinc_impulse(x, dtype=np.float64):
    """SincFunction as RealImpulseResponse::calc, conv_types.rs:479-487."""
    T = _T(dtype)
    x = T(x)
    if x == T(0):
        return T(1)
    pi_x = T(math.pi) * x
    return T(np.sin(pi_x) / pi_x)


def sinc_freq(x, dtype=np.float64):
    """SincFunction as RealFrequencyResponse::calc, conv_types.rs:498-505."""
    T = _T(dtype)
    return T(1) if abs(T(x)) <= T(1) else T(0)


def make_impulse_response(kind, rolloff, dtype):
    """interop translate_to_real_convolution_function (interop/src/lib.rs:166-178): 0 = Sinc, else RC."""
    if kind == 0:
        return lambda x: sinc_impulse(x, dtype)
    return lambda x: raised_cosine_impulse(x, rolloff, dtype)


def make_frequency_response(kind, rolloff, dtype):
    """interop translate_to_real_frequency_response (interop/src/lib.rs:180-192)."""
    if kind == 0:
        return lambda x: sinc_freq(x, dtype)
    return lambda x: raised_cosine_freq(x, rolloff, dtype)


# --------------------------------------------------------------------------------------------
# Half swaps  (vector_types/mod.rs:171-191, freq.rs:85-91)
# --------------------------------------------------------------------------------------------
def swap_array_halves_literal(data, forward):
    """Literal restatement of swap_array_halves (vector_types/mod.rs:171-191); small inputs only."""
    data = list(data)
    n = len(data)
    if n == 0:
        return data
    if n % 2 == 0:
        h = n // 2
        return data[h:] + data[:h]
    step = n // 2 if forward else n // 2 + 1
    temp = data[0]
    pos = step
    for _ in range(n):
        pos_new = (pos + step) % n
        temp, data[pos] = data[pos], temp
        pos = pos_new
    return data


def fft_shift(x):
    """FrequencyDomainOperations::fft_shift (freq.rs:85-87) == numpy.fft.fftshift."""
    x = np.asarray(x)
    return np.roll(x, len(x) // 2)


def ifft_shift(x):
    """FrequencyDomainOperations::ifft_shift (freq.rs:89-91) == numpy.fft.ifftshift."""
    x = np.asarray(x)
    return np.roll(x, -(len(x) // 2))


def swap_halves(x):
    """ReorganizeDataOps::swap_halves (data_reorganization.rs:247-252) -> swap_halves_priv(true)."""
    return fft_shift(x)


# --------------------------------------------------------------------------------------------
# Transforms  (time_freq/mod.rs:32-63, time_to_freq.rs:136-165, freq_to_time.rs:138-168)
# --------------------------------------------------------------------------------------------
def plain_fft(x):
    """Unnormalised forward DFT, DC at index 0.  Real input is first zero-interleaved to complex
    (time_to_freq.rs:147-150).  delta <- points*delta (time_freq/mod.rs:54-55) is handled by the
    caller (see `delta_after_fft`)."""
    return np.fft.fft(np.asarray(x).astype(np.complex128))


def fft(x):
    """plain_fft followed by fft_shift (time_to_freq.rs:158-165)."""
    return fft_shift(plain_fft(x))


def plain_ifft(X):
    """Unnormalised inverse DFT (rustfft Inverse direction, no 1/N)."""
    X = np.asarray(X).astype(np.complex128)
    return np.fft.ifft(X) * len(X)


def ifft(X):
    """scale(1/points) -> ifft_shift -> plain_ifft (freq_to_time.rs:160-168)."""
    X = np.asarray(X).astype(np.complex128)
    return plain_ifft(ifft_shift(X / len(X)))


def delta_after_fft(delta, points, dtype):
    """Q1: delta <- T(points)*delta for both directions (time_freq/mod.rs:54-55)."""
    T = _T(dtype)
    return T(T(points) * T(delta))


# --------------------------------------------------------------------------------------------
# convolve_signal: centred circular convolution
#   (convolution.rs:477-542, time_freq/mod.rs:275-361,456-473,788-848)
# --------------------------------------------------------------------------------------------
def conv_len_of(h_points):
    """conv_len = L - L/2 (time_freq/mod.rs:297-303); (L+1)/2 in overlap_discard (convolution.rs:381)."""
    return h_points - h_points // 2


def convolve_signal_direct(x, h):
    """Literal definition: y[i] = sum_k x[(i + cl - 1 - k) mod N] * h[k]
    (convolve_iteration + ReverseWrappingIterator, time_freq/mod.rs:456-473,788-848).
    O(N*L): small/medium inputs."""
    x = np.asarray(x)
    h = np.asarray(h)
    N, L = len(x), len(h)
    assert N >= L
    cl = conv_len_of(L)
    out_dtype = np.complex128 if (np.iscomplexobj(x) or np.iscomplexobj(h)) else np.float64
    xx = x.astype(out_dtype)
    y = np.zeros(N, dtype=out_dtype)
    idx = np.arange(N)
    for k in range(L):
        y += xx[(idx + cl - 1 - k) % N] * out_dtype(h[k])
    return y


def convolve_signal(x, h):
    """Same result via its FFT identity y = IFFT(FFT(x) * FFT(roll(pad(h, N), -(cl-1)))) in
    complex128 (error ~1e-15, far below the parity tolerance).  Use for large N."""
    x = np.asarray(x)
    h = np.asarray(h)
    N, L = len(x), len(h)
    assert N >= L
    cl = conv_len_of(L)
    hp = np.zeros(N, dtype=np.complex128)
    hp[:L] = h
    hp = np.roll(hp, -(cl - 1))
    y = np.fft.ifft(np.fft.fft(x.astype(np.complex128)) * np.fft.fft(hp))
    if not (np.iscomplexobj(x) or np.iscomplexobj(h)):
        return y.real.copy()
    return y


def check_convolve_signal_args(x_points, x_complex, x_domain, x_delta, h_points, h_complex, h_domain,
                               h_delta):
    """Error behaviour of convolve_signal (convolution.rs:485-492 + assert_meta_data! :257-268).
    Returns the C-ABI result code."""
    ratio = x_delta / h_delta
    if x_complex != h_complex or x_domain != h_domain or ratio > 1.1 or ratio < 0.9:
        return ERR_META_DATA
    if x_domain != 0:
        return ERR_MUST_BE_TIME
    if x_points < h_points:
        return ERR_INVALID_ARG_LEN
    return ERR_OK


# --------------------------------------------------------------------------------------------
# convolve with a function-defined impulse response
#   (convolution.rs:126-255, time_freq/mod.rs:174-213)
# --------------------------------------------------------------------------------------------
def would_benefit_from_simd(vec_len, imp_len, ratio, dtype):
    """convolution.rs:104-110."""
    T = _T(dtype)
    ratio = T(ratio)
    ratio_inv = T(1) / ratio
    return bool(imp_len <= 202 and vec_len > 2000
                and abs(np.round(ratio_inv) - ratio_inv) < T(1e-6) and ratio > T(0.5))


def function_taps(f, ratio, conv_len, dtype):
    """Tap table of convolve_function_priv (time_freq/mod.rs:199-209): for window offsets
    m = -L..L the tap is f(-j*ratio) with j = m counted up in precision T."""
    T = _T(dtype)
    ratio = T(ratio)
    taps = np.empty(2 * conv_len + 1, dtype=dtype)
    j = -T(conv_len)
    for q in range(2 * conv_len + 1):
        taps[q] = f(-j * ratio)
        j = j + T(1)
    return taps


def function_taps_simd_branch(f, ratio, conv_len, dtype):
    """Tap table of the `would_benefit_from_simd` branch (convolution.rs:151-167): f(j/ratio),
    j = -L..L, materialised and handed to convolve_signal."""
    T = _T(dtype)
    ratio_inv = T(1) / T(ratio)
    taps = np.empty(2 * conv_len + 1, dtype=dtype)
    j = -T(conv_len)
    for q in range(2 * conv_len + 1):
        taps[q] = f(j * ratio_inv)
        j = j + T(1)
    return taps


def convolve_function(x, f, ratio, conv_len, dtype, len_in_T=None):
    """Convolution::convolve for &dyn RealImpulseResponse (convolution.rs:136-192).

    Non-SIMD branch: y[i] = sum_{m=-L..L} x[(i+m) mod N] * f(-m*ratio), L = min(len, N)
    (time_freq/mod.rs:174-213; the WrappingIterator pre-increments, :745-763).
    SIMD branch (ratio == 1 in practice): the taps f(j/ratio) are materialised and routed through
    convolve_signal, i.e. y[i] = sum_k x[(i + cl - 1 - k) mod N] * t[k] with 2L+1 taps.

    Deliberate deviation (SURVEY Q4): for REAL vectors the reference's SIMD branch fills only every
    second tap (`i += 2`, convolution.rs:160-167); the oracle and the product implement the evident
    intent (all taps)."""
    x = np.asarray(x)
    N = len(x)
    if len_in_T is None:
        len_in_T = 2 * N if np.iscomplexobj(x) else N
    if would_benefit_from_simd(len_in_T, conv_len, ratio, dtype):
        taps = function_taps_simd_branch(f, ratio, conv_len, dtype)
        if len(taps) <= N:
            return convolve_signal_direct(x, taps.astype(np.float64)) if N * len(taps) < 5e7 else \
                convolve_signal(x, taps.astype(np.float64))
        # falls through in the reference to an InvalidArgumentLength panic (.expect); not reachable
        # for vec_len > 2000 and len <= 202.
    L = min(conv_len, N)
    taps = function_taps(f, ratio, L, dtype).astype(np.float64)
    out_dtype = np.complex128 if np.iscomplexobj(x) else np.float64
    xx = x.astype(out_dtype)
    y = np.zeros(N, dtype=out_dtype)
    idx = np.arange(N)
    for q in range(2 * L + 1):
        m = q - L
        y += xx[(idx + m) % N] * taps[q]
    return y


# --------------------------------------------------------------------------------------------
# multiply_frequency_response  (convolution.rs:545-610, time_freq/mod.rs:612-723)
# --------------------------------------------------------------------------------------------
def multiply_frequency_response(X, f, ratio, dtype):
    """X[i] <- X[i] * ratio * f(x_i * ratio), x_i = (i - c)/c with c = (points - points%2)/2
    (is_fft_shifted == false, time_freq/mod.rs:637-648 and fft_swap_x :67-78)."""
    T = _T(dtype)
    X = np.asarray(X)
    n = len(X)
    offset = n % 2
    mx = T(n - offset) / T(2)
    ratio = T(ratio)
    out = np.array(X, dtype=np.complex128 if np.iscomplexobj(X) else np.float64)
    j = -T(n - offset) / T(2)
    for i in range(n):
        out[i] = out[i] * float(ratio) * float(f(j / mx * ratio))
        j = j + T(1)
    return out


def fft_swap_x(is_fft_shifted, x_value, x_max):
    """time_freq/mod.rs:67-78."""
    if not is_fft_shifted:
        return x_value / x_max
    if x_value <= 0.0:
        return 1.0 + x_value / x_max
    return -(x_max - x_value + 1.0) / x_max


# --------------------------------------------------------------------------------------------
# interpolatef  (interpolation.rs:92-181,191-315,387-482)
# --------------------------------------------------------------------------------------------
def round_half_away(v):
    """Nearest integer, halves away from zero: Rust's f32/f64::round and C's round (np.round rounds halves to even)."""
    a = abs(float(v))
    r = math.floor(a)
    return int(math.copysign(r + 1 if a - r >= 0.5 else r, float(v)))


def interpolatef_new_len(len_T, factor, dtype):
    """new_len = round(len*F) rounded up to even (interpolation.rs:406-410), evaluated in T."""
    T = _T(dtype)
    n = round_half_away(T(len_T) * T(factor))
    return n + n % 2


def interpolatef_uses_fast_path(conv_len, new_len, factor, dtype):
    """interpolation.rs:411-414."""
    T = _T(dtype)
    factor = T(factor)
    return bool(conv_len <= 202 and new_len >= 2000 and abs(np.round(factor) - factor) < T(1e-6))


def interpolatef_tap_vectors(f, conv_len, factor_int, delay, dtype):
    """function_to_vectors (interpolation.rs:133-181): v_s[k] = f(j_k - s/F),
    j_0 = -(L-1) + delay, j_{k+1} = j_k + 1, all in precision T."""
    T = _T(dtype)
    vs = np.empty((factor_int, 2 * conv_len + 1), dtype=dtype)
    for s in range(factor_int):
        offset = T(s) / T(factor_int)
        j = -(T(conv_len) - T(1)) + T(delay)
        for k in range(2 * conv_len + 1):
            vs[s, k] = f(j - offset)
            j = j + T(1)
    return vs


def interpolatef(x, f, factor, delay, conv_len, dtype, delta=1.0, out_range=None):
    """InterpolationOps::interpolatef (interpolation.rs:387-482).

    out_range=(lo, hi): evaluate only output points lo <= i < hi of the result (same formulas; lets the
    tests walk BASELINE-sized vectors in bounded memory).

    * delay <- delay/delta (:397); L = min(conv_len, points/2) (:399-404).
    * integer-F fast path (interpolate_priv_simd :191-290): interior outputs use
      rc = ceil(i/F), s = (F - i%F)%F, y[i] = sum_q x[rc+L-1-q] * v_s[q]   (taps reversed, Q6);
      edge outputs (first/last (2L+1)*F) use interpolate_priv_simd_step :293-315:
      r = i//F, s = i%F, y[i] = sum_k x[(r-L+1+k) mod N] * v_s[k].
    * otherwise interpolate_priv_scalar :92-131: center = T(i)/F, r = floor(center),
      y[i] = sum_{k=0..2L} x[(r-L+k) mod N] * f(-L - (center-r) + delay + k).
    Output points: new_len (complex: new_len/2)."""
    T = _T(dtype)
    x = np.asarray(x)
    is_complex = np.iscomplexobj(x)
    N = len(x)
    len_T = 2 * N if is_complex else N
    delay = T(delay) / T(delta)
    L = min(conv_len, N // 2)
    new_len = interpolatef_new_len(len_T, factor, dtype)
    new_points = new_len // 2 if is_complex else new_len
    out_dtype = np.complex128 if is_complex else np.float64
    xx = x.astype(out_dtype) if out_range is None else x
    lo, hi = (0, new_points) if out_range is None else (max(0, int(out_range[0])), min(new_points, int(out_range[1])))
    y = np.zeros(hi - lo, dtype=out_dtype)
    if interpolatef_uses_fast_path(L, new_len, factor, dtype):
        F = int(np.round(T(factor)))
        vs = interpolatef_tap_vectors(f, L, F, delay, dtype).astype(np.float64)
        scalar_len = (2 * L + 1) * F
        i = np.arange(lo, hi)
        interior = (i >= scalar_len) & (i < new_points - scalar_len)
        # interior
        ii = i[interior]
        rc = (ii + F - 1) // F
        s = (F - ii % F) % F
        acc = np.zeros(len(ii), dtype=out_dtype)
        for q in range(2 * L + 1):
            acc += xx[rc + L - 1 - q] * vs[s, q]
        y[interior] = acc
        # edges
        ie = i[~interior]
        r = ie // F
        s = ie % F
        acc = np.zeros(len(ie), dtype=out_dtype)
        for k in range(2 * L + 1):
            acc += xx[(r - L + 1 + k) % N] * vs[s, k]
        y[~interior] = acc
        return y
    factor = T(factor)
    for i in range(lo, hi):
        center = T(i) / factor
        rounded = np.floor(center)
        r = int(rounded)
        j = -T(L) - (center - rounded) + delay
        acc = 0.0
        for k in range(2 * L + 1):
            acc = acc + xx[(r - L + k) % N] * float(f(j))
            j = j + T(1)
        y[i - lo] = acc
    return y


# --------------------------------------------------------------------------------------------
# interpolate_lin  (real_interpolation.rs:33-71)
# --------------------------------------------------------------------------------------------
def interpolate_lin_dest_len(data_len, factor, dtype):
    T = _T(dtype)
    return round_half_away(T(data_len - 1) * T(factor)) + 1


def interpolate_lin(x, factor, delay, dtype, replicate_counter_saturation=True):
    """dest_len = round((len-1)*F)+1; for i < dest_len-1: p = T(i)/F + delay (in T), b = floor(p),
    y[i] = x[b] + (x[b+1]-x[b])*(p-b) evaluated in T without FMA; last = x[len-1].

    The position p is computed in precision T exactly as the reference does, so the result is
    bit-reproducible.  Q7: the reference counts `i` in T by repeated `+ 1.0` (:53,65), which stops
    advancing at 2^24 in f32 (every later output is computed from the same position); the product
    replicates that saturation, and so does this oracle by default."""
    T = _T(dtype)
    x = np.asarray(x, dtype=dtype)
    n = len(x)
    dest_len = interpolate_lin_dest_len(n, factor, dtype)
    F = T(factor)
    d = T(delay)
    idx = np.arange(dest_len - 1, dtype=np.int64)
    i_T = idx.astype(dtype)
    if replicate_counter_saturation and dtype == np.float32:
        i_T = np.where(idx >= 2 ** 24, T(2 ** 24), i_T).astype(dtype)
    p = (i_T / F + d).astype(dtype)
    bf = np.floor(p)
    b = np.clip(bf.astype(np.int64), 0, n - 2)
    y0 = x[b]
    y1 = x[b + 1]
    out = np.empty(dest_len, dtype=dtype)
    out[:-1] = (y0 + ((y1 - y0).astype(dtype) * (p - bf).astype(dtype)).astype(dtype)).astype(dtype)
    out[-1] = x[n - 1]
    return out


# --------------------------------------------------------------------------------------------
# Elementwise chain  (elementary.rs:327-360,420-455,558-572; complex_to_real.rs:374-405,635-712;
#                     simd_extensions/fallback.rs:195-231)
# --------------------------------------------------------------------------------------------
def real_scale(x, c, dtype):
    """ScaleOps<T>::scale: every T scalar times c (elementary.rs:334-341)."""
    x = np.asarray(x)
    if np.iscomplexobj(x):
        ct = np.complex64 if dtype == np.float32 else np.complex128
        x = x.astype(ct)
        return (x.view(dtype) * _T(dtype)(c)).view(ct)
    return (x.astype(dtype) * _T(dtype)(c)).astype(dtype)


def _cmul_T(a_re, a_im, b_re, b_im, dtype):
    """(ac - bd, ad + bc) with every product and sum rounded to T, no FMA
    (num-complex Mul; simd_extensions/fallback.rs:195-203)."""
    a_re, a_im, b_re, b_im = (np.asarray(v, dtype=dtype) for v in (a_re, a_im, b_re, b_im))
    re = ((a_re * b_re).astype(dtype) - (a_im * b_im).astype(dtype)).astype(dtype)
    im = ((a_re * b_im).astype(dtype) + (a_im * b_re).astype(dtype)).astype(dtype)
    return re, im


def complex_scale(x, c, dtype):
    """ScaleOps<Complex<T>>::scale (elementary.rs:351-359)."""
    ct = np.complex64 if dtype == np.float32 else np.complex128
    x = np.asarray(x).astype(ct)
    re, im = _cmul_T(x.real, x.imag, np.real(c), np.imag(c), dtype)
    return (re + 1j * im).astype(ct)


def mul(x, w, dtype):
    """ElementaryOps::mul (elementary.rs:558-572): complex (ac-bd, ad+bc) or real product, in T."""
    x = np.asarray(x)
    w = np.asarray(w)
    if np.iscomplexobj(x):
        ct = np.complex64 if dtype == np.float32 else np.complex128
        x = x.astype(ct)
        w = w.astype(ct)
        re, im = _cmul_T(x.real, x.imag, w.real, w.imag, dtype)
        return (re + 1j * im).astype(ct)
    return (x.astype(dtype) * w.astype(dtype)).astype(dtype)


def add(x, w, dtype):
    ct = (np.complex64 if dtype == np.float32 else np.complex128) if np.iscomplexobj(x) else dtype
    return (np.asarray(x).astype(ct) + np.asarray(w).astype(ct)).astype(ct)


def sub(x, w, dtype):
    ct = (np.complex64 if dtype == np.float32 else np.complex128) if np.iscomplexobj(x) else dtype
    return (np.asarray(x).astype(ct) - np.asarray(w).astype(ct)).astype(ct)


def div(x, w, dtype):
    """ElementaryOps::div.  Complex: num-complex `Div` = (a*conj(b)) / |b|^2 component-wise, every
    operation rounded to T (elementary.rs:574-588 -> div_complex -> Complex::div)."""
    x = np.asarray(x)
    w = np.asarray(w)
    if np.iscomplexobj(x):
        ct = np.complex64 if dtype == np.float32 else np.complex128
        a, b = x.astype(ct), w.astype(ct)
        ar, ai, br, bi = (np.asarray(v, dtype=dtype) for v in (a.real, a.imag, b.real, b.imag))
        ns = ((br * br).astype(dtype) + (bi * bi).astype(dtype)).astype(dtype)
        re = ((ar * br).astype(dtype) + (ai * bi).astype(dtype)).astype(dtype)
        im = ((ai * br).astype(dtype) - (ar * bi).astype(dtype)).astype(dtype)
        return ((re / ns).astype(dtype) + 1j * (im / ns).astype(dtype)).astype(ct)
    return (x.astype(dtype) / w.astype(dtype)).astype(dtype)


def magnitude(x, dtype):
    """|x|: hypot (complex_to_real.rs:376) / sqrt(re^2+im^2) (fallback.rs:223-231); both are within
    1 ulp of the float64-evaluated value returned here."""
    x = np.asarray(x).astype(np.complex128)
    return np.hypot(x.real, x.imag).astype(dtype)


def magnitude_squared(x, dtype):
    x = np.asarray(x)
    re = x.real.astype(dtype)
    im = x.imag.astype(dtype)
    return ((re * re).astype(dtype) + (im * im).astype(dtype)).astype(dtype)


def phase(x, dtype):
    """atan2(im, re) (x.arg(), complex_to_real.rs:402)."""
    x = np.asarray(x).astype(np.complex128)
    return np.arctan2(x.imag, x.real).astype(dtype)


# --------------------------------------------------------------------------------------------
# SURVEY 8(f) rows: windows, correlation ("preparation" API), reverse, decimatei
# --------------------------------------------------------------------------------------------
def window_value(kind, n, length, dtype):
    """window_functions.rs:25-129; kind as in interop translate_to_window_function (lib.rs:153-164):
    0 Triangular, 1 Hamming(0.54), 2 BlackmanHarris, else Rectangular.  Evaluated in precision T."""
    T = _T(dtype)
    one, two = T(1), T(2)
    pi = T(math.pi)
    nn, ln = T(n), T(length)
    if kind == 0:
        return T(one - abs((nn - (ln - one) / two) / (ln / two)))
    if kind == 1:
        alpha = T(0.54)
        return T(alpha - (one - alpha) * np.cos(two * pi * nn / (ln - one)))
    if kind == 2:
        a0, a1, a2, a3 = T(0.35875), T(0.48829), T(0.14128), T(0.01168)
        return T(a0 - a1 * np.cos(two * pi * nn / (ln - one)) + a2 * np.cos(T(4) * pi * nn / (ln - one))
                 - a3 * np.cos(T(6) * pi * nn / (ln - one)))
    return one


def window_table(kind, points, dtype, unapply=False):
    """multiply_window_priv for symmetric windows (vector_types/mod.rs:528-598): element i of the second
    half is multiplied with the value computed for its mirror index points-1-i."""
    T = _T(dtype)
    tab = np.empty(points, dtype=dtype)
    for i in range(points):
        j = i if i < (points + 1) // 2 else points - 1 - i
        w = window_value(kind, j, points, dtype)
        tab[i] = T(1) / w if unapply else w
    return tab


def apply_window(x, kind, dtype, unapply=False):
    """TimeDomainOperations::apply_window / unapply_window (time.rs:33-66)."""
    x = np.asarray(x)
    tab = window_table(kind, len(x), dtype, unapply)
    if np.iscomplexobj(x):
        ct = np.complex64 if dtype == np.float32 else np.complex128
        xx = x.astype(ct)
        return ((xx.real.astype(dtype) * tab).astype(dtype) + 1j * (xx.imag.astype(dtype) * tab).astype(dtype)).astype(ct)
    return (x.astype(dtype) * tab).astype(dtype)


def windowed_fft(x, kind, dtype):
    """apply_window -> plain_fft -> fft_shift (time_to_freq.rs:167-175)."""
    return fft(apply_window(x, kind, dtype))


def windowed_ifft(X, kind, dtype):
    """ifft -> unapply_window (freq_to_time.rs:170-177)."""
    y = ifft(X)
    tab = window_table(kind, len(y), dtype, unapply=True).astype(np.float64)
    return y * tab


def zero_pad_surround(x, points):
    """zero_pad_b(.., PaddingOption::Surround) (data_reorganization.rs:426-439)."""
    x = np.asarray(x)
    diff = points - len(x)
    right = diff // 2
    left = diff - right
    return np.concatenate([np.zeros(left, dtype=x.dtype), x, np.zeros(right, dtype=x.dtype)])


def prepare_argument(b):
    """plain_fft then conj (correlation.rs:96-103)."""
    return np.conj(plain_fft(b))


def prepare_argument_padded(b):
    """zero_pad(2*points - 1, Surround) -> plain_fft -> conj (correlation.rs:105-117)."""
    b = np.asarray(b).astype(np.complex128)
    return np.conj(plain_fft(zero_pad_surround(b, 2 * len(b) - 1)))


def correlate(a, prepared):
    """CrossCorrelationOps::correlate (correlation.rs:131-163): zero_pad(other.points, Surround) ->
    plain_fft -> mul(other) -> plain_ifft -> scale(1/points) -> swap_halves."""
    a = np.asarray(a).astype(np.complex128)
    p = len(prepared)
    ap = zero_pad_surround(a, p)
    return swap_halves(plain_ifft(plain_fft(ap) * np.asarray(prepared)) / p)


def shifted_response_table(f, points, ratio, dtype, is_symmetric=True):
    """Multiplier table of multiply_function_priv with is_fft_shifted = true (time_freq/mod.rs:612-723,
    fft_swap_x :67-78) as used by interpolatei: X[i] *= ratio * f(swap(j_i) * ratio).
    Symmetric functions go through execute_sym_pairs_with_range (threading.rs:552-612): only the first
    half is evaluated (j <= 0: swap = 1 + j/max) and mirrored - element i pairs with points-i for an
    even and with points-1-i for an odd number of points."""
    T = _T(dtype)
    ratio = T(ratio)
    offset = points % 2
    mx = T(points - offset) / T(2)
    c = (points - offset) // 2
    tab = np.empty(points, dtype=dtype)

    def val(i):
        j = -mx + T(i)
        xv = (T(1) + j / mx) if j <= 0 else (-(mx - j + T(1)) / mx)
        return T(ratio * T(f(T(xv * ratio))))

    if not is_symmetric:
        for i in range(points):
            tab[i] = val(i)
        return tab
    for i in range(c + 1):
        tab[i] = val(i)
    if offset == 0:
        for i in range(1, c):
            tab[points - i] = tab[i]
    else:
        for i in range(c):
            tab[points - 1 - i] = tab[i]
    return tab


def interpolatei(x, f, factor, dtype):
    """InterpolationOps::interpolatei (interpolation.rs:484-538): zero_interleave -> plain_fft ->
    multiply with the (fft-shifted) frequency response * factor -> plain_ifft -> scale(1/points);
    real vectors are processed as complex and converted back with to_real."""
    x = np.asarray(x)
    if factor <= 1:
        return x.copy()
    is_complex = np.iscomplexobj(x)
    z = np.zeros(len(x) * factor, dtype=np.complex128)
    z[::factor] = x
    points = len(z)
    Z = plain_fft(z) * shifted_response_table(f, points, factor, dtype).astype(np.float64)
    y = plain_ifft(Z) / points
    return y if is_complex else y.real.copy()


ERR_CONJ_SYMMETRIC = 8
ERR_ODD_LENGTH = 9
ERR_FUNCTION_SYMMETRIC = 10


def zero_pad_center(X, points):
    """zero_pad(points, PaddingOption::Center) (data_reorganization.rs:343-357): the first
    ceil(n/2) points stay in front, the last floor(n/2) points move to the end, zeros in between."""
    X = np.asarray(X)
    n = len(X)
    right = n // 2
    left = n - right
    out = np.zeros(points, dtype=X.dtype)
    out[:left] = X[:left]
    if right:
        out[points - right:] = X[left:left + right]
    return out


def linear_phase_table(points, delay, dtype):
    """apply_linear_phase (interpolation.rs:319-339): element i < points/2 is rotated by
    exp(j*inc*i), element i >= points/2 by exp(j*inc*(i - points)), inc = 2*pi*delay/points in T.
    The reference advances the phasor by repeated multiplication (complex_ops.rs:95-102); the restatement
    evaluates each angle directly (the difference is rounding drift of the reference's recurrence)."""
    T = _T(dtype)
    pos = points // 2
    neg = points - pos
    inc = T(T(2) * T(np.pi) * T(delay) / T(points))
    ang = np.empty(points, dtype=np.float64)
    ang[:pos] = float(inc) * np.arange(pos)
    ang[pos:] = float(T(-T(neg) * inc)) + float(inc) * np.arange(neg)
    return np.exp(1j * ang)


def interpolate(x, f, dest_points, delay, dtype, delta=1.0):
    """InterpolationOps::interpolate (interpolation.rs:541-604); f = None is interpft (:533-539).
    plain_fft -> linear phase (delay/delta) -> [upsample: zero_pad Center, * factor * f(shifted x * factor)
    (or * factor without f) | downsample: keep the first ceil(d/2) and the last floor(d/2) bins, scale d/n]
    -> plain_ifft -> scale(1/dest_points) (-> real part for real input)."""
    T = _T(dtype)
    x = np.asarray(x)
    is_complex = np.iscomplexobj(x)
    n = len(x)
    factor = T(dest_points) / T(n)
    X = plain_fft(x.astype(np.complex128))
    if delay != 0:
        X = X * linear_phase_table(n, T(delay) / T(delta), dtype)
    if dest_points > n:
        X = zero_pad_center(X, dest_points)
        if f is None:
            X = X * float(factor)
        else:
            X = X * shifted_response_table(f, dest_points, factor, dtype).astype(np.float64)
    elif dest_points < n:
        neg = dest_points // 2
        pos = dest_points - neg
        X = np.concatenate([X[:pos], X[n - neg:]]) if neg else X[:pos].copy()
        X = X * float(T(2 * dest_points) / T(2 * n))
    y = plain_ifft(X) / dest_points
    return y if is_complex else y.real.copy()


def interpft(x, dest_points, dtype):
    return interpolate(x, None, dest_points, 0.0, dtype)


def conj(x):
    return np.conj(np.asarray(x))


def multiply_complex_exponential(x, a, b, dtype, delta=1.0):
    """ComplexOps::multiply_complex_exponential (complex_ops.rs:81-105): x[i] *= exp(j*(a*delta*i + b*delta))."""
    T = _T(dtype)
    a = T(T(a) * T(delta))
    b = T(T(b) * T(delta))
    i = np.arange(len(x))
    return np.asarray(x).astype(np.complex128) * np.exp(1j * (float(a) * i + float(b)))


def mirror(X):
    """FrequencyDomainOperations::mirror (freq.rs:52-83): [X0, X1 .. X(p-1)] -> [X0, X1 .. X(p-1),
    conj X(p-1) .. conj X1]  (2p - 1 points)."""
    X = np.asarray(X)
    return np.concatenate([X, np.conj(X[1:][::-1])])


def plain_sfft(x):
    """SymmetricTimeToFrequencyDomainOperations::plain_sfft (time_to_freq.rs:197-230) for a statically
    real vector with an odd number n of points: the first (n + 1)/2 bins of the complex transform.
    (Through the interop's dynamically typed vector the reference computes the kept length from the
    complex point count and keeps n/2 + 1 SCALARS - an odd, rejected length for n = 1 mod 4; the drop-in
    follows the statically typed behaviour its own test real_fft_test32 exercises.)"""
    x = np.asarray(x)
    assert not np.iscomplexobj(x) and len(x) % 2 == 1
    return plain_fft(x.astype(np.complex128))[: (len(x) + 1) // 2]


def sfft(x):
    """sfft (time_to_freq.rs:232-264): fft (shifted) then the same truncation: bins -(n-1)/2 .. 0."""
    x = np.asarray(x)
    assert not np.iscomplexobj(x) and len(x) % 2 == 1
    return fft(x.astype(np.complex128))[: (len(x) + 1) // 2]


def windowed_sfft(x, kind, dtype):
    """windowed_sfft (time_to_freq.rs:266-298): window on the complexified vector, then sfft."""
    return sfft_of_complexified(apply_window(np.asarray(x).astype(dtype), kind, dtype))


def sfft_of_complexified(x):
    return fft(np.asarray(x).astype(np.complex128))[: (len(x) + 1) // 2]


def plain_sifft(X):
    """plain_sifft (freq_to_time.rs:190-221): needs Im X[0] ~ 0 (|.| <= 1e-10, else
    InputMustBeConjSymmetric); mirror -> unnormalised inverse transform -> real part (2p - 1 points)."""
    X = np.asarray(X).astype(np.complex128)
    if len(X) and abs(X[0].imag) > 1e-10:
        return ERR_CONJ_SYMMETRIC
    return plain_ifft(mirror(X)).real.copy()


def sifft(X):
    """sifft (freq_to_time.rs:223-234): scale(1/points) with the HALF spectrum's point count,
    ifft_shift of the half spectrum, plain_sifft."""
    X = np.asarray(X).astype(np.complex128)
    return plain_sifft(ifft_shift(X / len(X)))


def windowed_sifft(X, kind, dtype):
    y = sifft(X)
    if isinstance(y, int):
        return y
    return y * window_table(kind, len(y), dtype, unapply=True).astype(np.float64)


# --------------------------------------------------------------------------------------------------
# elementwise math (trigonometry_and_powers.rs:198-377, real_ops.rs:243-289)
# Real vectors call the scalar libm function of T.  Complex vectors call num-complex (dependency
# `num-complex = "^0.4"`, vector/Cargo.toml:39; not vendored in the reference tree): its published
# formulas are restated below in precision T on separate re / im arrays.
# --------------------------------------------------------------------------------------------------
def _split(x, dtype):
    x = np.asarray(x)
    return np.ascontiguousarray(x.real, dtype=dtype), np.ascontiguousarray(x.imag, dtype=dtype)


def _join(re, im, dtype):
    ct = np.complex64 if dtype == np.float32 else np.complex128
    out = np.empty(len(re), dtype=ct)
    out.real = re
    out.imag = im
    return out


def _c_mul(a, b):
    return a[0] * b[0] - a[1] * b[1], a[0] * b[1] + a[1] * b[0]


def _c_polar(a):
    return np.hypot(a[0], a[1]), np.arctan2(a[1], a[0])


def _c_from_polar(r, th):
    return r * np.cos(th), r * np.sin(th)


def _c_ln(a):
    r, th = _c_polar(a)
    return np.log(r), th


def _c_sqrt(a):
    """num-complex Complex::sqrt: exact branches for purely real / purely imaginary input, polar form otherwise."""
    re, im = a
    T = re.dtype.type
    r, th = _c_polar(a)
    gre, gim = _c_from_polar(np.sqrt(r), th / T(2))
    # re == 0, im != 0
    x = np.sqrt(np.abs(im) / T(2))
    ore = np.where(re == 0, x, gre)
    oim = np.where(re == 0, np.where(np.signbit(im), -x, x), gim)
    # im == 0
    pos = ~np.signbit(re)
    sre = np.sqrt(np.abs(re))
    ore = np.where(im == 0, np.where(pos, sre, T(0)), ore)
    oim = np.where(im == 0, np.where(pos, im, np.where(np.signbit(im), -sre, sre)), oim)
    return ore.astype(re.dtype), oim.astype(re.dtype)


def complex_math(name, x, dtype, arg=None):
    """pure_complex_operation with the num-complex method `name`."""
    T = _T(dtype)
    re, im = _split(x, dtype)
    z = (re, im)
    one = (np.ones_like(re), np.zeros_like(re))
    with np.errstate(all="ignore"):
        if name == "sin":
            r = (np.sin(re) * np.cosh(im), np.cos(re) * np.sinh(im))
        elif name == "cos":
            r = (np.cos(re) * np.cosh(im), -np.sin(re) * np.sinh(im))
        elif name == "tan":
            tr, ti = re + re, im + im
            d = np.cos(tr) + np.cosh(ti)
            r = (np.sin(tr) / d, np.sinh(ti) / d)
        elif name == "sinh":
            r = (np.sinh(re) * np.cos(im), np.cosh(re) * np.sin(im))
        elif name == "cosh":
            r = (np.cosh(re) * np.cos(im), np.sinh(re) * np.sin(im))
        elif name == "tanh":
            tr, ti = re + re, im + im
            d = np.cosh(tr) + np.cos(ti)
            r = (np.sinh(tr) / d, np.sin(ti) / d)
        elif name == "asin":      # -i ln(sqrt(1 - z^2) + i z)
            zz = _c_mul(z, z)
            s = _c_sqrt((one[0] - zz[0], one[1] - zz[1]))
            w = _c_ln((s[0] - im, s[1] + re))
            r = (w[1], -w[0])
        elif name == "acos":      # -i ln(i sqrt(1 - z^2) + z)
            zz = _c_mul(z, z)
            s = _c_sqrt((one[0] - zz[0], one[1] - zz[1]))
            w = _c_ln((-s[1] + re, s[0] + im))
            r = (w[1], -w[0])
        elif name == "atan":      # (ln(1 + i z) - ln(1 - i z)) / (2 i)
            a = _c_ln((one[0] - im, one[1] + re))
            b = _c_ln((one[0] + im, one[1] - re))
            d = (a[0] - b[0], a[1] - b[1])
            r = (d[1] / T(2), -d[0] / T(2))
        elif name == "asinh":     # ln(z + sqrt(1 + z^2))
            zz = _c_mul(z, z)
            s = _c_sqrt((one[0] + zz[0], one[1] + zz[1]))
            r = _c_ln((re + s[0], im + s[1]))
        elif name == "acosh":     # 2 ln(sqrt((z + 1)/2) + sqrt((z - 1)/2))
            a = _c_sqrt(((re + T(1)) / T(2), im / T(2)))
            b = _c_sqrt(((re - T(1)) / T(2), im / T(2)))
            w = _c_ln((a[0] + b[0], a[1] + b[1]))
            r = (T(2) * w[0], T(2) * w[1])
        elif name == "atanh":     # (ln(1 + z) - ln(1 - z)) / 2
            a = _c_ln((one[0] + re, one[1] + im))
            b = _c_ln((one[0] - re, one[1] - im))
            r = ((a[0] - b[0]) / T(2), (a[1] - b[1]) / T(2))
        elif name == "sqrt":
            r = _c_sqrt(z)
        elif name == "square":
            r = _c_mul(z, z)
        elif name == "ln":
            r = _c_ln(z)
        elif name == "exp":
            r = _c_from_polar(np.exp(re), im)
        elif name == "powf":
            rr, th = _c_polar(z)
            r = _c_from_polar(np.power(rr, T(arg)), th * T(arg))
            if T(arg) == 0:
                r = (np.ones_like(re), np.zeros_like(re))
        elif name == "log":
            rr, th = _c_polar(z)
            lb = np.log(T(arg))
            r = (np.log(rr) / lb, th / lb)
        elif name == "expf":      # base^z = from_polar(base^re, im * ln(base))
            r = _c_from_polar(np.power(T(arg), re), im * np.log(T(arg)))
        else:
            raise ValueError(name)
    return _join(np.asarray(r[0], dtype=dtype), np.asarray(r[1], dtype=dtype), dtype)


def real_math(name, x, dtype, arg=None):
    """pure_real_operation / simd_real_operation with the scalar function of T."""
    T = _T(dtype)
    x = np.asarray(x, dtype=dtype)
    f = {"sin": np.sin, "cos": np.cos, "tan": np.tan, "asin": np.arcsin, "acos": np.arccos, "atan": np.arctan,
         "sinh": np.sinh, "cosh": np.cosh, "tanh": np.tanh, "asinh": np.arcsinh, "acosh": np.arccosh,
         "atanh": np.arctanh, "sqrt": np.sqrt, "ln": np.log, "exp": np.exp, "abs": np.abs}
    with np.errstate(all="ignore"):
        if name in f:
            return f[name](x).astype(dtype)
        if name == "square":
            return (x * x).astype(dtype)
        if name == "powf":
            return np.power(x, T(arg)).astype(dtype)
        if name == "root":
            return np.power(x, T(1) / T(arg)).astype(dtype)
        if name == "log":
            return (np.log(x) / np.log(T(arg))).astype(dtype)
        if name == "expf":
            return np.power(T(arg), x).astype(dtype)
        if name == "wrap":        # Rust `%` on floats: fmod
            return np.fmod(x, T(arg)).astype(dtype)
    raise ValueError(name)


def unwrap(x, divisor, dtype):
    """ModuloOps::unwrap (real_ops.rs:266-288), sequential: each element is compared with its already
    unwrapped predecessor."""
    T = _T(dtype)
    d = np.asarray(x, dtype=dtype).copy()
    div = T(divisor)
    half = T(div / T(2))
    for j in range(1, len(d)):
        diff = T(d[j] - d[j - 1])
        if diff > half:
            diff = T(np.fmod(diff, div))
            diff = T(diff - div)
            d[j] = T(d[j - 1] + diff)
        elif diff < -half:
            diff = T(np.fmod(diff, div))
            diff = T(diff + div)
            d[j] = T(d[j - 1] + diff)
    return d


def diff(x, with_start=False):
    """DiffSumOps::diff / diff_with_start (diff_sum.rs:63-109)."""
    x = np.asarray(x)
    if with_start:
        return np.concatenate([x[:1], x[1:] - x[:-1]]).astype(x.dtype)
    return (x[1:] - x[:-1]).astype(x.dtype)


def cum_sum(x):
    """DiffSumOps::cum_sum (diff_sum.rs:111-122): sequential running sum in T."""
    return np.cumsum(np.asarray(x), dtype=np.asarray(x).dtype)


def binary_smaller(op, x, w, dtype):
    """add/sub/mul/div_smaller (elementary.rs:457-517,601-639): operand element i % operand.len()."""
    x = np.asarray(x)
    w = np.asarray(w)
    if len(x) % len(w) != 0:
        return ERR_INVALID_ARG_LEN
    ww = np.tile(w, len(x) // len(w))
    return {"add": add, "sub": sub, "mul": mul, "div": div}[op](x, ww, dtype)


def split_into(x, n):
    """data_reorganization.rs:484-512: element i goes to target i % n at position i / n."""
    x = np.asarray(x)
    if n == 0 or len(x) % n != 0:
        return ERR_INVALID_ARG_LEN
    return [x[i::n].copy() for i in range(n)]


def merge(sources):
    """data_reorganization.rs:522-557: inverse of split_into."""
    n = len(sources)
    if n == 0 or any(len(s) != len(sources[0]) for s in sources):
        return ERR_INVALID_ARG_LEN
    out = np.empty(n * len(sources[0]), dtype=np.asarray(sources[0]).dtype)
    for i, s in enumerate(sources):
        out[i::n] = s
    return out


def set_mag_phase(mag, phase, dtype):
    """complex_to_real.rs:749-770: Complex::from_polar(mag, phase) = (mag cos(phase), mag sin(phase))."""
    mag = np.asarray(mag, dtype=dtype)
    phase = np.asarray(phase, dtype=dtype)
    return _join(mag * np.cos(phase), mag * np.sin(phase), dtype)


def interpolate_hermite(x, factor, delay, dtype):
    """RealInterpolationOps::interpolate_hermite (real_interpolation.rs:73-178), every operation in T,
    including the output counter `i = i + 1` kept in T."""
    T = _T(dtype)
    x = np.asarray(x, dtype=dtype)
    n = len(x)
    F, d = T(factor), T(delay)
    dest_len = round_half_away(T(n - 1) * F) + 1
    start = int(np.ceil((T(1) - d) * F))
    end = start + 1
    half, c15, two, c25 = T(0.5), T(1.5), T(2.0), T(2.5)
    out = np.empty(dest_len, dtype=dtype)
    i = T(0)
    for k in range(dest_len):
        rounded = T(i / F + d)
        bf = T(np.floor(rounded))
        b = int(bf)
        if k < start:
            y1, y2, y3 = x[b], x[b + 1], x[b + 2]
            y0 = T(y1 - T(y2 - y1))
        elif k < dest_len - end:
            y0, y1, y2, y3 = x[b - 1], x[b], x[b + 1], x[b + 2]
        else:
            y0, y1 = x[b - 1], x[b]
            y2 = x[b + 1] if b < n - 1 else T(y1 + T(y1 - y0))
            y3 = x[b + 2] if b < n - 2 else T(y2 + T(y2 - y1))
        xx = T(rounded - bf)
        x2 = T(xx * xx)
        a0 = T(T(T(T(-half * y0) + T(c15 * y1)) - T(c15 * y2)) + T(half * y3))
        a1 = T(T(T(y0 - T(c25 * y1)) + T(two * y2)) - T(half * y3))
        a2 = T(T(-half * y0) + T(half * y2))
        out[k] = T(T(T(T(T(a0 * xx) * x2) + T(a1 * x2)) + T(a2 * xx)) + y1)
        i = T(i + T(1))
    return out


# --------------------------------------------------------------------------------------------------
# reductions (statistics.rs, precise_stats.rs, dot_products.rs)
# --------------------------------------------------------------------------------------------------
def statistics(x):
    """StatisticsOps::statistics (statistics.rs:179-340) as computed on ONE chunk (the reference merges
    per-thread chunk results; its merge drops a chunk's minimum when the same chunk also raised the
    maximum, :230-236 - the restatement is the single-chunk result).  Complex: min / max by norm,
    rms = sqrt(sum(z^2) / count) (complex)."""
    x = np.asarray(x)
    n = len(x)
    acc = x.astype(np.complex128 if np.iscomplexobj(x) else np.float64)
    s = acc.sum()
    ssq = (acc * acc).sum()
    if n == 0:
        nan = float("nan")
        return dict(sum=s, count=0, average=nan, rms=nan, min=float("inf"), min_index=0, max=float("-inf"), max_index=0)
    key = np.abs(acc) if np.iscomplexobj(x) else acc
    imin, imax = int(np.argmin(key)), int(np.argmax(key))
    return dict(sum=s, count=n, average=s / n, rms=np.sqrt(ssq / n), min=x[imin], min_index=imin, max=x[imax], max_index=imax)


def statistics_split(x, parts):
    """statistics_split (statistics.rs:395-440): element j belongs to part j % parts with index j / parts."""
    if parts > 16:
        return ERR_INVALID_ARG_LEN
    x = np.asarray(x)
    return [statistics(x[i::parts]) for i in range(parts)]


def dot_product(a, b):
    """DotProductOps::dot_product (dot_products.rs:67-160): sum(a[i] * b[i]) (no conjugation)."""
    a = np.asarray(a)
    b = np.asarray(b)
    n = min(len(a), len(b))
    wide = np.complex128 if np.iscomplexobj(a) else np.float64
    return (a[:n].astype(wide) * b[:n].astype(wide)).sum()


def reverse(x):
    return np.asarray(x)[::-1].copy()


def decimatei(x, factor, delay):
    """interpolation.rs:606-632: keeps points delay, delay+factor, ..."""
    return np.asarray(x)[delay::factor].copy()


def ulp_diff(a, b, dtype):
    """Distance in units in the last place of `dtype` between two real arrays."""
    a = np.asarray(a, dtype=dtype)
    b = np.asarray(b, dtype=dtype)
    it = np.int32 if dtype == np.float32 else np.int64
    ai = a.view(it).astype(np.int64)
    bi = b.view(it).astype(np.int64)
    mask = np.int64(0x7FFFFFFF) if dtype == np.float32 else np.iinfo(np.int64).max
    ai = np.where(ai < 0, -(ai & mask), ai)  # sign-magnitude -> monotone integer line
    bi = np.where(bi < 0, -(bi & mask), bi)
    return np.abs(ai - bi)


def rel_l2(a, b):
    a = np.asarray(a).astype(np.complex128).ravel()
    b = np.asarray(b).astype(np.complex128).ravel()
    den = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / den) if den > 0 else float(np.linalg.norm(a - b))
