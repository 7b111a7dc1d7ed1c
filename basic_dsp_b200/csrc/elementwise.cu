// Single-pass elementwise kernels: scale/offset, add/sub/mul/div, magnitude/phase and the fused
// scale -> mul -> (magnitude, phase) chain, half swaps, zero interleave.
//
// Reference: vector/src/vector_types/general/elementary.rs:283-360,420-455,540-589 and
// vector/src/vector_types/complex/complex_to_real.rs:374-478,595-712.  Arithmetic follows the
// reference's CPU path operation by operation (no FMA contraction: mul_rn/add_rn of common.cuh), so results
// are within the 4-ulp budget of BASELINE.json (bit-identical for the ring operations).
// All kernels are grid-stride, 16 B per thread per access where alignment allows.
#include "elementwise.cuh"

namespace bdsp {

// correctly rounded square root in T (norm and argument: the float / double overloads of hypot and atan2)
__device__ __forceinline__ float sqrt_rn(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ double sqrt_rn(double a) { return __dsqrt_rn(a); }

// ---- unary ops on T scalars (real scale / offset) ------------------------------------------------
template <typename T, int OP>
__global__ void scalar_op_kernel(const T* __restrict__ in, T* __restrict__ out, long long n, T c) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        T v = in[i];
        out[i] = OP == EW_SCALE ? mul_rn(v, c) : add_rn(v, c);
    }
}

// ---- complex-constant ops ---------------------------------------------------------------------------
template <typename T, int OP>
__global__ void complex_const_kernel(const typename CpxOf<T>::type* __restrict__ in,
                                     typename CpxOf<T>::type* __restrict__ out, long long n, T cre, T cim) {
    typedef typename CpxOf<T>::type C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const C c = mk<T>(cre, cim);
    for (; i < n; i += stride) {
        C v = in[i];
        if (OP == EW_SCALE) v = cmul_nofma(v, c);
        else if (OP == EW_OFFSET) { v.x = add_rn(v.x, cre); v.y = add_rn(v.y, cim); }
        else if (OP == EW_CONJ) v.y = -v.y;
        out[i] = v;
    }
}

// ---- binary vector ops --------------------------------------------------------------------------------
template <typename T, int OP>
__global__ void binary_real_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = ew_real_op<OP>(a[i], b[i]);
}

template <typename T, int OP>
__global__ void binary_complex_kernel(const typename CpxOf<T>::type* __restrict__ a,
                                      const typename CpxOf<T>::type* __restrict__ b,
                                      typename CpxOf<T>::type* __restrict__ out, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = ew_complex_op<OP>(a[i], b[i]);
}

// ---- complex -> real ------------------------------------------------------------------------------------
template <typename T, int OP> __device__ __forceinline__ T c2r(typename CpxOf<T>::type v) {
    if (OP == C2R_MAG_HYPOT) return hypot(v.x, v.y);
    if (OP == C2R_MAG_SQRT) return sqrt_rn(add_rn(mul_rn(v.x, v.x), mul_rn(v.y, v.y)));
    if (OP == C2R_MAG_SQ) return add_rn(mul_rn(v.x, v.x), mul_rn(v.y, v.y));
    if (OP == C2R_PHASE) return atan2(v.y, v.x);
    if (OP == C2R_REAL) return v.x;
    return v.y;
}

// In-place capable: out may alias the front half of `in` (the reference writes the real result
// into the front half of the same storage, vector_types/mod.rs:437-452).  Each thread reads its
// element pair before any thread of a *later* index range can overwrite it only when whole blocks
// are processed in order, which a grid cannot guarantee -> the C ABI always passes a separate
// destination (the vector's scratch) and swaps.
template <typename T, int OP>
__global__ void complex_to_real_kernel(const typename CpxOf<T>::type* __restrict__ in, T* __restrict__ out, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = c2r<T, OP>(in[i]);
}

template <typename T>
__global__ void mag_phase_kernel(const typename CpxOf<T>::type* __restrict__ in, T* __restrict__ mag, T* __restrict__ ph, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        typename CpxOf<T>::type v = in[i];
        mag[i] = hypot(v.x, v.y);   // Complex::to_polar = (norm, arg), complex_to_real.rs:707
        ph[i] = atan2(v.y, v.x);
    }
}

// fused chain of sequential trait calls: v.scale(c); v.mul(&w); (mag, phase) = v.get_mag_phase()
// one read of v and w, one write of mag and phase (48 B/point for c64 instead of 128 B unfused)
template <typename T, bool WRITE_V>
__global__ void scale_mul_mag_phase_kernel(typename CpxOf<T>::type* __restrict__ v, const typename CpxOf<T>::type* __restrict__ w,
                                           T* __restrict__ mag, T* __restrict__ ph, long long n, T cre, T cim, int complex_scale) {
    typedef typename CpxOf<T>::type C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const C c = mk<T>(cre, cim);
    for (; i < n; i += stride) {
        C x = v[i];
        if (complex_scale) x = cmul_nofma(x, c);
        else { x.x = mul_rn(x.x, cre); x.y = mul_rn(x.y, cre); }
        x = cmul_nofma(x, w[i]);
        if (WRITE_V) v[i] = x;
        mag[i] = hypot(x.x, x.y);
        ph[i] = atan2(x.y, x.x);
    }
}

// ---- data reorganisation ------------------------------------------------------------------------------
// out[(i + rot) mod n] = in[i] for elements of `esz` T scalars (swap_halves / fft_shift / ifft_shift)
template <typename T>
__global__ void rotate_kernel(const T* __restrict__ in, T* __restrict__ out, long long n_elems, long long rot, int esz) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long total = n_elems * esz;
    for (; i < total; i += stride) {
        long long e = i / esz, c = i - e * esz;
        long long d = e + rot; if (d >= n_elems) d -= n_elems;
        out[d * esz + c] = in[i];
    }
}

// out[i*factor] = in[i], other slots zero, for elements of esz scalars (zero_interleave_b, to_complex)
template <typename T>
__global__ void zero_interleave_kernel(const T* __restrict__ in, T* __restrict__ out, long long n_elems, int factor, int esz) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long total = n_elems * factor * esz;
    for (; i < total; i += stride) {
        long long e = i / esz, c = i - e * esz;
        long long src = e / factor;
        out[i] = (e - src * factor == 0) ? in[src * esz + c] : (T)0;
    }
}

// out[i] = in[n-1-i] for elements of esz scalars (ReorganizeDataOps::reverse, data_reorganization.rs:237-246)
template <typename T>
__global__ void reverse_kernel(const T* __restrict__ in, T* __restrict__ out, long long n_elems, int esz) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long total = n_elems * esz;
    for (; i < total; i += stride) {
        long long e = i / esz, c = i - e * esz;
        out[(n_elems - 1 - e) * esz + c] = in[i];
    }
}

// out[j] = in[delay + j*factor] (InterpolationOps::decimatei, interpolation.rs:606-632)
template <typename T>
__global__ void decimate_kernel(const T* __restrict__ in, T* __restrict__ out, long long out_elems, long long factor, long long delay, int esz) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long total = out_elems * esz;
    for (; i < total; i += stride) {
        long long e = i / esz, c = i - e * esz;
        out[i] = in[(delay + e * factor) * esz + c];
    }
}

template <typename T>
__global__ void fill_kernel(T* __restrict__ out, long long n, T v) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = v;
}

// multiply_function_priv for the built-in frequency responses (time_freq/mod.rs:612-648,
// conv_types.rs:434-449,498-505): X[i] *= ratio * f((j/max) * ratio), j = i - (points - points%2)/2
template <typename T>
__global__ void mul_freq_resp_kernel(T* __restrict__ data, long long points, int is_complex, int kind, T rolloff, T ratio) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long offset = points % 2;
    const T mx = (T)(points - offset) / (T)2;
    for (; i < points; i += stride) {
        T j = add_rn(-mx, (T)i);
        T x = mul_rn(div_rn(j, mx), ratio);
        T ax = fabs(x);
        T f;
        if (kind == 0) f = ax <= (T)1 ? (T)1 : (T)0;
        else {
            const T one = (T)1, two = (T)2, pi = (T)3.14159265358979323846;
            if (ax <= (one - rolloff)) f = one;
            else if (ax <= (one + rolloff)) f = one / two * (one + cos(pi / rolloff * (ax - (one - rolloff)) / two));
            else f = (T)0;
        }
        if (is_complex) {
            // (*num) * scale * fun(..) with scale, fun converted to Complex (imag 0): two complex products
            typename CpxOf<T>::type v = reinterpret_cast<typename CpxOf<T>::type*>(data)[i];
            v = cmul_nofma(v, mk<T>(ratio, (T)0));
            v = cmul_nofma(v, mk<T>(f, (T)0));
            reinterpret_cast<typename CpxOf<T>::type*>(data)[i] = v;
        } else {
            data[i] = mul_rn(mul_rn(data[i], ratio), f);
        }
    }
}


// apply_window / unapply_window for the built-in windows (window_functions.rs:25-129; time.rs:33-66; symmetric windows are
// evaluated for the first half and mirrored, vector_types/mod.rs:528-598), evaluated on the device in precision T
template <typename T>
__global__ void window_kernel(T* __restrict__ data, long long points, int is_complex, int kind, int unapply) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < points; i += stride) {
        const long long j = i < (points + 1) / 2 ? i : points - 1 - i;
        T w = window_value_dev<T>(kind, j, points);
        if (unapply) w = div_rn((T)1, w);
        if (is_complex) {
            typedef typename CpxOf<T>::type C;
            reinterpret_cast<C*>(data)[i] = cmul_nofma(reinterpret_cast<C*>(data)[i], mk<T>(w, (T)0));
        } else data[i] = mul_rn(data[i], w);
    }
}

// X[i] *= table[i] (complex or real table) - host-evaluated custom responses / windows
template <typename T>
__global__ void mul_table_kernel(T* __restrict__ data, const T* __restrict__ table, long long points, int is_complex, int table_complex) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < points; i += stride) {
        if (is_complex) {
            typedef typename CpxOf<T>::type C;
            C v = reinterpret_cast<C*>(data)[i];
            C t = table_complex ? reinterpret_cast<const C*>(table)[i] : mk<T>(table[i], (T)0);
            reinterpret_cast<C*>(data)[i] = cmul_nofma(v, t);
        } else data[i] = mul_rn(data[i], table[i]);
    }
}



// multiplier of multiply_function_priv with is_fft_shifted = true for the built-in frequency responses
// (time_freq/mod.rs:612-723, fft_swap_x :67-78; symmetric: first half evaluated, second half mirrored):
// ratio * f(x * ratio), x = 1 + (i' - mx)/mx for the mirrored index i' <= mx
template <typename T> __device__ __forceinline__ T shifted_resp_dev(long long i, long long points, int kind, T rolloff, T ratio) {
    const long long offset = points % 2;
    const long long c = (points - offset) / 2;
    const T mx = (T)(points - offset) / (T)2;
    const long long ip = i <= c ? i : (offset == 0 ? points - i : points - 1 - i);
    const T j = -mx + (T)ip;
    const T xv = j <= (T)0 ? (T)1 + j / mx : -(mx - j + (T)1) / mx;
    const T x = xv * ratio;
    const T ax = fabs(x);
    T f;
    if (kind == 0) f = ax <= (T)1 ? (T)1 : (T)0;
    else {
        const T one = (T)1, two = (T)2, pi = (T)3.14159265358979323846;
        if (ax <= (one - rolloff)) f = one;
        else if (ax <= (one + rolloff)) f = one / two * (one + cos(pi / rolloff * (ax - (one - rolloff)) / two));
        else f = (T)0;
    }
    return ratio * f;
}
template <typename T>
__global__ void mul_shifted_resp_kernel(typename CpxOf<T>::type* __restrict__ data, long long points, int kind, T rolloff, T ratio) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < points; i += stride) data[i] = cmul_nofma(data[i], mk<T>(shifted_resp_dev<T>(i, points, kind, rolloff, ratio), (T)0));
}

// ---- FFT-based resampling: spectrum re-binning (interpolation.rs:541-604) ----------------------------
// out[k] (dest bins) = in[src(k)] * phase(src) * (table ? table[k] : 1) * scale, zero where the padded
// spectrum has no source bin.  n > dest: keep the first ceil(dest/2) and last floor(dest/2) bins;
// n < dest: zero_pad Center (first ceil(n/2) bins in front, last floor(n/2) at the end).
// phase: apply_linear_phase (interpolation.rs:319-339): bin i < n/2 -> exp(j*inc*i), else exp(j*inc*(i-n)).
template <typename T>
__global__ void resample_spectrum_kernel(const typename CpxOf<T>::type* __restrict__ in, typename CpxOf<T>::type* __restrict__ out,
                                         long long n, long long dest, const T* __restrict__ table, T scale, int use_scale,
                                         double phase_inc, int use_phase, int resp_kind, T resp_rolloff, T resp_ratio) {
    typedef typename CpxOf<T>::type C;
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; k < dest; k += stride) {
        long long src;
        if (dest >= n) {
            const long long right = n / 2, left = n - right;
            src = k < left ? k : (k >= dest - right ? k - (dest - n) : -1);
        } else {
            const long long neg = dest / 2, pos = dest - neg;
            src = k < pos ? k : k + (n - dest);
        }
        C v = mk<T>((T)0, (T)0);
        if (src >= 0) {
            v = in[src];
            if (use_phase) {
                const long long m = src < n / 2 ? src : src - n;
                double sn, cs;
                sincos(phase_inc * (double)m, &sn, &cs);
                v = cmul_nofma(v, mk<T>((T)cs, (T)sn));
            }
            if (table) { const T w = table[k]; v = cmul_nofma(v, mk<T>(w, (T)0)); }
            else if (resp_kind >= 0) v = cmul_nofma(v, mk<T>(shifted_resp_dev<T>(k, dest, resp_kind, resp_rolloff, resp_ratio), (T)0));
            if (use_scale) { v.x = mul_rn(v.x, scale); v.y = mul_rn(v.y, scale); }
        }
        out[k] = v;
    }
}

// mirror (freq.rs:52-83): p points -> 2p - 1 points, out[p + i] = conj(in[p - 1 - i])
template <typename T>
__global__ void mirror_kernel(const typename CpxOf<T>::type* __restrict__ in, typename CpxOf<T>::type* __restrict__ out, long long p) {
    typedef typename CpxOf<T>::type C;
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long total = 2 * p - 1;
    for (; k < total; k += stride) {
        if (k < p) out[k] = in[k];
        else { C v = in[total - k]; out[k] = mk<T>(v.x, -v.y); }
    }
}

// multiply_complex_exponential (complex_ops.rs:81-105)
template <typename T>
__global__ void mul_cexp_kernel(typename CpxOf<T>::type* __restrict__ data, long long points, double a, double b) {
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; k < points; k += stride) {
        double sn, cs;
        sincos(a * (double)k + b, &sn, &cs);
        data[k] = cmul_nofma(data[k], mk<T>((T)cs, (T)sn));
    }
}

// spectrum product of a fast convolution over rows: a[r * M + i] = a[r * M + i] * bspec[i] * scale.  Contraction allowed,
// as in the transforms around it; one thread per point.
template <typename T>
__global__ void spectrum_mul_rows_kernel(typename CpxOf<T>::type* __restrict__ a,
                                         const typename CpxOf<T>::type* __restrict__ bspec, long long M,
                                         long long batch, T scale) {
    typedef typename CpxOf<T>::type C;
    long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= M * batch) return;
    C v = cmul(a[gid], bspec[gid % M]);
    v.x *= scale; v.y *= scale;
    a[gid] = v;
}

// ------------------------------------------------------------------------------------------
// host wrappers
// ------------------------------------------------------------------------------------------
template <typename T>
int ew_scalar(int op, const void* in, void* out, size_t n_scalars, double c, cudaStream_t st) {
    const T* i = reinterpret_cast<const T*>(in); T* o = reinterpret_cast<T*>(out);
    const long long n = (long long)n_scalars;
    if (op == EW_SCALE) return launch_grid_stride(scalar_op_kernel<T, EW_SCALE>, n, st, i, o, n, (T)c);
    return launch_grid_stride(scalar_op_kernel<T, EW_OFFSET>, n, st, i, o, n, (T)c);
}

template <typename T>
int ew_complex_const(int op, const void* in, void* out, size_t points, double re, double im, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const C* i = reinterpret_cast<const C*>(in); C* o = reinterpret_cast<C*>(out);
    const long long n = (long long)points;
    if (op == EW_SCALE) return launch_grid_stride(complex_const_kernel<T, EW_SCALE>, n, st, i, o, n, (T)re, (T)im);
    if (op == EW_OFFSET) return launch_grid_stride(complex_const_kernel<T, EW_OFFSET>, n, st, i, o, n, (T)re, (T)im);
    return launch_grid_stride(complex_const_kernel<T, EW_CONJ>, n, st, i, o, n, (T)re, (T)im);
}

template <typename T>
int ew_binary(int op, const void* a, const void* b, void* out, size_t n_scalars, int is_complex, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    if (is_complex && (op == EW_MUL || op == EW_DIV)) {
        const C* x = reinterpret_cast<const C*>(a); const C* y = reinterpret_cast<const C*>(b); C* o = reinterpret_cast<C*>(out);
        const long long n = (long long)(n_scalars / 2);
        if (op == EW_MUL) return launch_grid_stride(binary_complex_kernel<T, EW_MUL>, n, st, x, y, o, n);
        return launch_grid_stride(binary_complex_kernel<T, EW_DIV>, n, st, x, y, o, n);
    }
    // complex add / sub are the real ops on the interleaved scalars
    const T* x = reinterpret_cast<const T*>(a); const T* y = reinterpret_cast<const T*>(b); T* o = reinterpret_cast<T*>(out);
    const long long n = (long long)n_scalars;
    if (op == EW_ADD) return launch_grid_stride(binary_real_kernel<T, EW_ADD>, n, st, x, y, o, n);
    if (op == EW_SUB) return launch_grid_stride(binary_real_kernel<T, EW_SUB>, n, st, x, y, o, n);
    if (op == EW_MUL) return launch_grid_stride(binary_real_kernel<T, EW_MUL>, n, st, x, y, o, n);
    return launch_grid_stride(binary_real_kernel<T, EW_DIV>, n, st, x, y, o, n);
}

template <typename T>
int ew_complex_to_real(int op, const void* in, void* out, size_t points, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const C* i = reinterpret_cast<const C*>(in); T* o = reinterpret_cast<T*>(out);
    const long long n = (long long)points;
    switch (op) {
        case C2R_MAG_HYPOT: return launch_grid_stride(complex_to_real_kernel<T, C2R_MAG_HYPOT>, n, st, i, o, n);
        case C2R_MAG_SQRT: return launch_grid_stride(complex_to_real_kernel<T, C2R_MAG_SQRT>, n, st, i, o, n);
        case C2R_MAG_SQ: return launch_grid_stride(complex_to_real_kernel<T, C2R_MAG_SQ>, n, st, i, o, n);
        case C2R_PHASE: return launch_grid_stride(complex_to_real_kernel<T, C2R_PHASE>, n, st, i, o, n);
        case C2R_REAL: return launch_grid_stride(complex_to_real_kernel<T, C2R_REAL>, n, st, i, o, n);
        default: return launch_grid_stride(complex_to_real_kernel<T, C2R_IMAG>, n, st, i, o, n);
    }
}

template <typename T>
int ew_mag_phase(const void* in, void* mag, void* phase, size_t points, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    return launch_grid_stride(mag_phase_kernel<T>, (long long)points, st, reinterpret_cast<const C*>(in), reinterpret_cast<T*>(mag),
                              reinterpret_cast<T*>(phase), (long long)points);
}

template <typename T>
int ew_scale_mul_mag_phase(void* v, const void* w, void* mag, void* phase, size_t points, double cre, double cim,
                           int complex_scale, int write_v, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    auto run = [&](auto kernel) {
        return launch_grid_stride(kernel, (long long)points, st, reinterpret_cast<C*>(v), reinterpret_cast<const C*>(w),
                                  reinterpret_cast<T*>(mag), reinterpret_cast<T*>(phase), (long long)points, (T)cre, (T)cim, complex_scale);
    };
    return write_v ? run(scale_mul_mag_phase_kernel<T, true>) : run(scale_mul_mag_phase_kernel<T, false>);
}

template <typename T>
int ew_rotate(const void* in, void* out, size_t n_elems, size_t rot, int esz, cudaStream_t st) {
    return launch_grid_stride(rotate_kernel<T>, (long long)(n_elems * esz), st, reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out),
                              (long long)n_elems, (long long)rot, esz);
}

template <typename T>
int ew_zero_interleave(const void* in, void* out, size_t n_elems, int factor, int esz, cudaStream_t st) {
    return launch_grid_stride(zero_interleave_kernel<T>, (long long)(n_elems * factor * esz), st, reinterpret_cast<const T*>(in),
                              reinterpret_cast<T*>(out), (long long)n_elems, factor, esz);
}

template <typename T> int ew_reverse(const void* in, void* out, size_t n_elems, int esz, cudaStream_t st) {
    return launch_grid_stride(reverse_kernel<T>, (long long)(n_elems * esz), st, reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out),
                              (long long)n_elems, esz);
}

template <typename T> int ew_decimate(const void* in, void* out, size_t out_elems, size_t factor, size_t delay, int esz, cudaStream_t st) {
    return launch_grid_stride(decimate_kernel<T>, (long long)(out_elems * esz), st, reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out),
                              (long long)out_elems, (long long)factor, (long long)delay, esz);
}

template <typename T> int ew_fill(void* out, size_t n, double v, cudaStream_t st) {
    return launch_grid_stride(fill_kernel<T>, (long long)n, st, reinterpret_cast<T*>(out), (long long)n, (T)v);
}

template <typename T>
int ew_mul_freq_resp(void* data, size_t points, int is_complex, int kind, double rolloff, double ratio, cudaStream_t st) {
    return launch_grid_stride(mul_freq_resp_kernel<T>, (long long)points, st, reinterpret_cast<T*>(data), (long long)points, is_complex, kind,
                              (T)rolloff, (T)ratio);
}

template <typename T>
int ew_window(void* data, size_t points, int is_complex, int kind, int unapply, cudaStream_t st) {
    if (!points) return 0;
    return launch_grid_stride(window_kernel<T>, (long long)points, st, reinterpret_cast<T*>(data), (long long)points, is_complex, kind, unapply);
}

template <typename T>
int ew_mul_table(void* data, const void* table, size_t points, int is_complex, int table_complex, cudaStream_t st) {
    return launch_grid_stride(mul_table_kernel<T>, (long long)points, st, reinterpret_cast<T*>(data), reinterpret_cast<const T*>(table),
                              (long long)points, is_complex, table_complex);
}

template <typename T>
int ew_resample_spectrum(const void* in, void* out, size_t n, size_t dest, const void* table, double scale, int use_scale,
                         double phase_inc, int use_phase, int resp_kind, double resp_rolloff, double resp_ratio, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    if (!dest) return 0;
    return launch_grid_stride(resample_spectrum_kernel<T>, (long long)dest, st, reinterpret_cast<const C*>(in), reinterpret_cast<C*>(out),
                              (long long)n, (long long)dest, reinterpret_cast<const T*>(table), (T)scale, use_scale, phase_inc, use_phase,
                              resp_kind, (T)resp_rolloff, (T)resp_ratio);
}

template <typename T>
int ew_mul_shifted_resp(void* data, size_t points, int kind, double rolloff, double ratio, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    if (!points) return 0;
    return launch_grid_stride(mul_shifted_resp_kernel<T>, (long long)points, st, reinterpret_cast<C*>(data), (long long)points, kind,
                              (T)rolloff, (T)ratio);
}

template <typename T>
int ew_mirror(const void* in, void* out, size_t points, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    if (!points) return 0;
    return launch_grid_stride(mirror_kernel<T>, (long long)(2 * points - 1), st, reinterpret_cast<const C*>(in), reinterpret_cast<C*>(out),
                              (long long)points);
}
template <typename T>
int ew_mul_cexp(void* data, size_t points, double a, double b, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    if (!points) return 0;
    return launch_grid_stride(mul_cexp_kernel<T>, (long long)points, st, reinterpret_cast<C*>(data), (long long)points, a, b);
}

template <typename T>
int ew_spectrum_mul_rows(void* x, const void* h, size_t n, size_t rows, double scale, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const long long tot = (long long)(n * rows);
    spectrum_mul_rows_kernel<T><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(reinterpret_cast<C*>(x), reinterpret_cast<const C*>(h),
                                                                                (long long)n, (long long)rows, (T)scale);
    BDSP_LAUNCHED();
    return 0;
}

#define BDSP_INST(T)                                                                                     \
    template int ew_resample_spectrum<T>(const void*, void*, size_t, size_t, const void*, double, int, double, int, int, double, double, cudaStream_t); \
    template int ew_mul_shifted_resp<T>(void*, size_t, int, double, double, cudaStream_t);            \
    template int ew_mirror<T>(const void*, void*, size_t, cudaStream_t);                                  \
    template int ew_mul_cexp<T>(void*, size_t, double, double, cudaStream_t);                             \
    template int ew_scalar<T>(int, const void*, void*, size_t, double, cudaStream_t);                     \
    template int ew_complex_const<T>(int, const void*, void*, size_t, double, double, cudaStream_t);      \
    template int ew_binary<T>(int, const void*, const void*, void*, size_t, int, cudaStream_t);           \
    template int ew_complex_to_real<T>(int, const void*, void*, size_t, cudaStream_t);                    \
    template int ew_mag_phase<T>(const void*, void*, void*, size_t, cudaStream_t);                        \
    template int ew_scale_mul_mag_phase<T>(void*, const void*, void*, void*, size_t, double, double, int, int, cudaStream_t); \
    template int ew_rotate<T>(const void*, void*, size_t, size_t, int, cudaStream_t);                     \
    template int ew_zero_interleave<T>(const void*, void*, size_t, int, int, cudaStream_t);               \
    template int ew_fill<T>(void*, size_t, double, cudaStream_t);                                         \
    template int ew_reverse<T>(const void*, void*, size_t, int, cudaStream_t);                            \
    template int ew_decimate<T>(const void*, void*, size_t, size_t, size_t, int, cudaStream_t);           \
    template int ew_mul_freq_resp<T>(void*, size_t, int, int, double, double, cudaStream_t);              \
    template int ew_window<T>(void*, size_t, int, int, int, cudaStream_t);                                \
    template int ew_mul_table<T>(void*, const void*, size_t, int, int, cudaStream_t);                     \
    template int ew_spectrum_mul_rows<T>(void*, const void*, size_t, size_t, double, cudaStream_t);
BDSP_INST(float)
BDSP_INST(double)
#undef BDSP_INST

}  // namespace bdsp
