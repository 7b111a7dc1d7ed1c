// Elementwise math family of the reference's C facade (SURVEY 8f row 4): trigonometry / powers
// (trigonometry_and_powers.rs:198-377), abs / wrap / unwrap (real_ops.rs:243-289), diff / cum_sum
// (diff_sum.rs:63-122), *_smaller (elementary.rs:457-517), split_into / merge
// (data_reorganization.rs:484-557), set_real_imag / set_mag_phase (complex_to_real.rs:726-770) and
// interpolate_hermite (real_interpolation.rs:73-178).
//
// Real vectors: the CUDA libm function of T.  Complex vectors: the formulas of num-complex 0.4 (the
// reference's dependency) written out on (re, im) in precision T.  All kernels are one pass over HBM
// (grid-stride, 8 or 16 bytes per thread and access).
#include <cuda_runtime.h>
#include <math_constants.h>

#include "common.cuh"
#include "elementwise.cuh"
#include "mathops.cuh"

namespace bdsp {
namespace {

__device__ __forceinline__ void sc_(float x, float* s, float* c) { sincosf(x, s, c); }
__device__ __forceinline__ void sc_(double x, double* s, double* c) { sincos(x, s, c); }
template <typename T> __device__ __forceinline__ typename CpxOf<T>::type c_from_polar(T r, T th) {
    T s, c;
    sc_(th, &s, &c);
    return mk<T>(mul_rn(r, c), mul_rn(r, s));
}
template <typename T> __device__ __forceinline__ typename CpxOf<T>::type c_ln(typename CpxOf<T>::type a) {
    return mk<T>((T)log(hypot(a.x, a.y)), (T)atan2(a.y, a.x));
}
template <typename T> __device__ __forceinline__ typename CpxOf<T>::type c_sqrt(typename CpxOf<T>::type a) {
    // num-complex Complex::sqrt: exact branches for purely real / purely imaginary input
    if (a.y == (T)0) {
        if (!signbit(a.x)) return mk<T>((T)sqrt(a.x), a.y);
        const T im = (T)sqrt(-a.x);
        return mk<T>((T)0, signbit(a.y) ? -im : im);
    }
    if (a.x == (T)0) {
        const T x = (T)sqrt(div_rn((T)fabs(a.y), (T)2));
        return mk<T>(x, signbit(a.y) ? -x : x);
    }
    return c_from_polar((T)sqrt(hypot(a.x, a.y)), div_rn((T)atan2(a.y, a.x), (T)2));
}

template <typename T> __device__ typename CpxOf<T>::type complex_fn(int op, typename CpxOf<T>::type z, T arg, T ln_arg) {
    typedef typename CpxOf<T>::type C;
    const T re = z.x, im = z.y;
    switch (op) {
    case M_SIN: return mk<T>(mul_rn((T)sin(re), (T)cosh(im)), mul_rn((T)cos(re), (T)sinh(im)));
    case M_COS: return mk<T>(mul_rn((T)cos(re), (T)cosh(im)), mul_rn(-(T)sin(re), (T)sinh(im)));
    case M_TAN: {
        const T tr = add_rn(re, re), ti = add_rn(im, im);
        const T d = add_rn((T)cos(tr), (T)cosh(ti));
        return mk<T>(div_rn((T)sin(tr), d), div_rn((T)sinh(ti), d));
    }
    case M_SINH: return mk<T>(mul_rn((T)sinh(re), (T)cos(im)), mul_rn((T)cosh(re), (T)sin(im)));
    case M_COSH: return mk<T>(mul_rn((T)cosh(re), (T)cos(im)), mul_rn((T)sinh(re), (T)sin(im)));
    case M_TANH: {
        const T tr = add_rn(re, re), ti = add_rn(im, im);
        const T d = add_rn((T)cosh(tr), (T)cos(ti));
        return mk<T>(div_rn((T)sinh(tr), d), div_rn((T)sin(ti), d));
    }
    case M_ASIN: {   // -i ln(sqrt(1 - z^2) + i z)
        const C zz = cmul_nofma(z, z);
        const C s = c_sqrt<T>(mk<T>(sub_rn((T)1, zz.x), sub_rn((T)0, zz.y)));
        const C w = c_ln<T>(mk<T>(sub_rn(s.x, im), add_rn(s.y, re)));
        return mk<T>(w.y, -w.x);
    }
    case M_ACOS: {   // -i ln(i sqrt(1 - z^2) + z)
        const C zz = cmul_nofma(z, z);
        const C s = c_sqrt<T>(mk<T>(sub_rn((T)1, zz.x), sub_rn((T)0, zz.y)));
        const C w = c_ln<T>(mk<T>(add_rn(-s.y, re), add_rn(s.x, im)));
        return mk<T>(w.y, -w.x);
    }
    case M_ATAN: {   // (ln(1 + i z) - ln(1 - i z)) / (2 i)
        if (re == (T)0 && im == (T)1) return mk<T>((T)0, (T)CUDART_INF);
        if (re == (T)0 && im == (T)-1) return mk<T>((T)0, -(T)CUDART_INF);
        const C a = c_ln<T>(mk<T>(sub_rn((T)1, im), add_rn((T)0, re)));
        const C b = c_ln<T>(mk<T>(add_rn((T)1, im), sub_rn((T)0, re)));
        return mk<T>(div_rn(sub_rn(a.y, b.y), (T)2), -div_rn(sub_rn(a.x, b.x), (T)2));
    }
    case M_ASINH: {  // ln(z + sqrt(1 + z^2))
        const C zz = cmul_nofma(z, z);
        const C s = c_sqrt<T>(mk<T>(add_rn((T)1, zz.x), add_rn((T)0, zz.y)));
        return c_ln<T>(mk<T>(add_rn(re, s.x), add_rn(im, s.y)));
    }
    case M_ACOSH: {  // 2 ln(sqrt((z + 1) / 2) + sqrt((z - 1) / 2))
        const C a = c_sqrt<T>(mk<T>(div_rn(add_rn(re, (T)1), (T)2), div_rn(im, (T)2)));
        const C b = c_sqrt<T>(mk<T>(div_rn(sub_rn(re, (T)1), (T)2), div_rn(im, (T)2)));
        const C w = c_ln<T>(mk<T>(add_rn(a.x, b.x), add_rn(a.y, b.y)));
        return mk<T>(mul_rn((T)2, w.x), mul_rn((T)2, w.y));
    }
    case M_ATANH: {  // (ln(1 + z) - ln(1 - z)) / 2
        if (re == (T)1 && im == (T)0) return mk<T>((T)CUDART_INF, (T)0);
        if (re == (T)-1 && im == (T)0) return mk<T>(-(T)CUDART_INF, (T)0);
        const C a = c_ln<T>(mk<T>(add_rn((T)1, re), add_rn((T)0, im)));
        const C b = c_ln<T>(mk<T>(sub_rn((T)1, re), sub_rn((T)0, im)));
        return mk<T>(div_rn(sub_rn(a.x, b.x), (T)2), div_rn(sub_rn(a.y, b.y), (T)2));
    }
    case M_SQRT: return c_sqrt<T>(z);
    case M_SQUARE: return cmul_nofma(z, z);
    case M_LN: return c_ln<T>(z);
    case M_EXP: return c_from_polar((T)exp(re), im);
    case M_POWF:
        if (arg == (T)0) return mk<T>((T)1, (T)0);
        return c_from_polar((T)pow(hypot(re, im), arg), mul_rn((T)atan2(im, re), arg));
    case M_LOG: return mk<T>(div_rn((T)log(hypot(re, im)), ln_arg), div_rn((T)atan2(im, re), ln_arg));
    case M_EXPF: return c_from_polar((T)pow(arg, re), mul_rn(im, ln_arg));
    default: return z;
    }
}

template <typename T> __device__ T real_fn(int op, T x, T arg, T ln_arg) {
    switch (op) {
    case M_SIN: return (T)sin(x);
    case M_COS: return (T)cos(x);
    case M_TAN: return (T)tan(x);
    case M_ASIN: return (T)asin(x);
    case M_ACOS: return (T)acos(x);
    case M_ATAN: return (T)atan(x);
    case M_SINH: return (T)sinh(x);
    case M_COSH: return (T)cosh(x);
    case M_TANH: return (T)tanh(x);
    case M_ASINH: return (T)asinh(x);
    case M_ACOSH: return (T)acosh(x);
    case M_ATANH: return (T)atanh(x);
    case M_SQRT: return (T)sqrt(x);
    case M_SQUARE: return mul_rn(x, x);
    case M_LN: return (T)log(x);
    case M_EXP: return (T)exp(x);
    case M_ABS: return (T)fabs(x);
    case M_POWF: return (T)pow(x, arg);
    case M_LOG: return div_rn((T)log(x), ln_arg);
    case M_EXPF: return (T)pow(arg, x);
    case M_WRAP: return (T)fmod(x, arg);
    default: return x;
    }
}

// 16 bytes per thread and access; the n % W tail is handled by the first threads
template <typename T> struct alignas(16) Pack { T v[16 / sizeof(T)]; };
template <typename T>
__global__ void math_real_kernel(T* __restrict__ data, long long n, int op, T arg, T ln_arg) {
    constexpr int W = 16 / sizeof(T);
    const long long nv = n / W;
    Pack<T>* dv = reinterpret_cast<Pack<T>*>(data);
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = tid; i < nv; i += stride) {
        Pack<T> p = dv[i];
#pragma unroll
        for (int k = 0; k < W; k++) p.v[k] = real_fn<T>(op, p.v[k], arg, ln_arg);
        dv[i] = p;
    }
    const long long t = nv * W + tid;
    if (t < n) data[t] = real_fn<T>(op, data[t], arg, ln_arg);
}
template <typename T>
__global__ void math_complex_kernel(typename CpxOf<T>::type* __restrict__ data, long long n, int op, T arg, T ln_arg) {
    typedef typename CpxOf<T>::type C;
    constexpr int W = 16 / sizeof(C);   // 2 (f32) or 1 (f64)
    const long long nv = n / W;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    Pack<T>* dv = reinterpret_cast<Pack<T>*>(data);
    for (long long i = tid; i < nv; i += stride) {
        Pack<T> p = dv[i];
#pragma unroll
        for (int k = 0; k < W; k++) {
            const C r = complex_fn<T>(op, mk<T>(p.v[2 * k], p.v[2 * k + 1]), arg, ln_arg);
            p.v[2 * k] = r.x; p.v[2 * k + 1] = r.y;
        }
        dv[i] = p;
    }
    const long long t = nv * W + tid;
    if (t < n) data[t] = complex_fn<T>(op, data[t], arg, ln_arg);
}

// ---- unwrap: loop-carried through rounded values -> one warp, lane 0 walks 128-element tiles staged in
// shared memory by the whole warp (coalesced loads / stores, sequential arithmetic) -------------------
template <typename T>
__global__ void unwrap_kernel(T* __restrict__ data, long long n, T divisor) {
    __shared__ T tile[2][1024];
    const int lane = threadIdx.x;
    const T half = div_rn(divisor, (T)2);
    T prev = (T)0;
    const long long tiles = (n + 1023) / 1024;
    for (int k = lane; k < 1024 && k < n; k += 32) tile[0][k] = data[k];
    __syncwarp();
    for (long long t = 0; t < tiles; t++) {
        const int cur = (int)(t & 1);
        const long long base = t * 1024;
        const int cnt = (int)((n - base) < 1024 ? (n - base) : 1024);
        // prefetch the next tile while lane 0 works (loads are issued before the serial loop)
        T nxt[32];
        const long long nb = base + 1024;
        if (t + 1 < tiles) {
#pragma unroll
            for (int k = 0; k < 32; k++) { const long long j = nb + lane + 32 * k; nxt[k] = j < n ? data[j] : (T)0; }
        }
        if (lane == 0) {
            int j0 = 0;
            if (t == 0) { prev = tile[cur][0]; j0 = 1; }
            for (int j = j0; j < cnt; j++) {
                T v = tile[cur][j];
                T diff = sub_rn(v, prev);
                if (diff > half) { diff = sub_rn((T)fmod(diff, divisor), divisor); v = add_rn(prev, diff); }
                else if (diff < -half) { diff = add_rn((T)fmod(diff, divisor), divisor); v = add_rn(prev, diff); }
                tile[cur][j] = v;
                prev = v;
            }
        }
        __syncwarp();
        for (int k = lane; k < cnt; k += 32) data[base + k] = tile[cur][k];
        if (t + 1 < tiles) {
#pragma unroll
            for (int k = 0; k < 32; k++) tile[cur ^ 1][lane + 32 * k] = nxt[k];
        }
        __syncwarp();
    }
}

// ---- diff ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void diff_kernel(const T* __restrict__ in, T* __restrict__ out, long long n_out, int step, int with_start) {
    // scalars; complex = step 2.  with_start: out[0..step) = in[0..step), out[j] = in[j] - in[j - step]
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n_out; i += stride) {
        if (with_start) out[i] = i < step ? in[i] : sub_rn(in[i], in[i - step]);
        else out[i] = sub_rn(in[i + step], in[i]);
    }
}

// ---- cum_sum: three-phase scan over LANES interleaved sequences (1 real, 2 complex) ---------------------
// phase 1: per-block totals; phase 2: exclusive scan of the totals (one block per lane); phase 3: block-local scan +
// offsets.  A thread owns CS_PER consecutive points (all lanes) and moves them with 16-byte accesses.
constexpr int CS_THREADS = 256;
constexpr int CS_PER = 8;

template <typename T, int LANES>
__device__ __forceinline__ void cs_load(const T* __restrict__ in, long long base, long long points, T (&v)[CS_PER * LANES]) {
    constexpr int W = 16 / sizeof(T);                 // scalars per pack
    constexpr int NP = CS_PER * LANES / W;            // packs per thread
    if (base + CS_PER <= points) {
        const Pack<T>* pv = reinterpret_cast<const Pack<T>*>(in + base * LANES);
#pragma unroll
        for (int q = 0; q < NP; q++) {
            const Pack<T> pk = pv[q];
#pragma unroll
            for (int e = 0; e < W; e++) v[q * W + e] = pk.v[e];
        }
    } else {
#pragma unroll
        for (int k = 0; k < CS_PER * LANES; k++) v[k] = (base * LANES + k < points * LANES) ? in[base * LANES + k] : (T)0;
    }
}

template <typename T, int LANES>
__global__ void __launch_bounds__(CS_THREADS) cumsum_totals_kernel(const T* __restrict__ in, T* __restrict__ totals, long long points) {
    __shared__ T sh[LANES][CS_THREADS];
    const long long base = ((long long)blockIdx.x * CS_THREADS + threadIdx.x) * CS_PER;
    T v[CS_PER * LANES];
    cs_load<T, LANES>(in, base, points, v);
#pragma unroll
    for (int l = 0; l < LANES; l++) {
        T s = (T)0;
#pragma unroll
        for (int k = 0; k < CS_PER; k++) s = add_rn(s, v[k * LANES + l]);
        sh[l][threadIdx.x] = s;
    }
    __syncthreads();
    for (int off = CS_THREADS / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off)
#pragma unroll
            for (int l = 0; l < LANES; l++) sh[l][threadIdx.x] = add_rn(sh[l][threadIdx.x], sh[l][threadIdx.x + off]);
        __syncthreads();
    }
    if (threadIdx.x < LANES) totals[(long long)threadIdx.x * gridDim.x + blockIdx.x] = sh[threadIdx.x][0];
}
template <typename T>
__global__ void __launch_bounds__(1024) cumsum_scan_totals_kernel(T* __restrict__ totals, long long nblocks, int lanes) {
    // one block per lane: exclusive scan of the per-block totals (thread t owns a contiguous run)
    __shared__ T sh[1024];
    T* t = totals + (long long)blockIdx.x * nblocks;
    const long long per = (nblocks + 1023) / 1024;
    const long long b0 = (long long)threadIdx.x * per;
    T s = (T)0;
    for (long long b = b0; b < b0 + per && b < nblocks; b++) s = add_rn(s, t[b]);
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        T add = (T)0;
        if (threadIdx.x >= off) add = sh[threadIdx.x - off];
        __syncthreads();
        if (threadIdx.x >= off) sh[threadIdx.x] = add_rn(sh[threadIdx.x], add);
        __syncthreads();
    }
    T run = threadIdx.x ? sh[threadIdx.x - 1] : (T)0;
    for (long long b = b0; b < b0 + per && b < nblocks; b++) { const T v = t[b]; t[b] = run; run = add_rn(run, v); }
}
template <typename T, int LANES>
__global__ void __launch_bounds__(CS_THREADS) cumsum_apply_kernel(const T* __restrict__ in, T* __restrict__ out, const T* __restrict__ totals,
                                                                long long points) {
    __shared__ T sh[LANES][CS_THREADS];
    const long long base = ((long long)blockIdx.x * CS_THREADS + threadIdx.x) * CS_PER;
    T v[CS_PER * LANES];
    cs_load<T, LANES>(in, base, points, v);
#pragma unroll
    for (int l = 0; l < LANES; l++) {
        T s = (T)0;
#pragma unroll
        for (int k = 0; k < CS_PER; k++) { s = add_rn(s, v[k * LANES + l]); v[k * LANES + l] = s; }
        sh[l][threadIdx.x] = s;
    }
    __syncthreads();
    // Hillis-Steele inclusive scan of the per-thread sums
    for (int off = 1; off < CS_THREADS; off <<= 1) {
        T add[LANES];
#pragma unroll
        for (int l = 0; l < LANES; l++) add[l] = threadIdx.x >= off ? sh[l][threadIdx.x - off] : (T)0;
        __syncthreads();
        if (threadIdx.x >= off)
#pragma unroll
            for (int l = 0; l < LANES; l++) sh[l][threadIdx.x] = add_rn(sh[l][threadIdx.x], add[l]);
        __syncthreads();
    }
    T offset[LANES];
#pragma unroll
    for (int l = 0; l < LANES; l++)
        offset[l] = add_rn(totals[(long long)l * gridDim.x + blockIdx.x], threadIdx.x ? sh[l][threadIdx.x - 1] : (T)0);
#pragma unroll
    for (int k = 0; k < CS_PER * LANES; k++) v[k] = add_rn(offset[k % LANES], v[k]);
    constexpr int W = 16 / sizeof(T);
    constexpr int NP = CS_PER * LANES / W;
    if (base + CS_PER <= points) {
        Pack<T>* pv = reinterpret_cast<Pack<T>*>(out + base * LANES);
#pragma unroll
        for (int q = 0; q < NP; q++) {
            Pack<T> pk;
#pragma unroll
            for (int e = 0; e < W; e++) pk.v[e] = v[q * W + e];
            pv[q] = pk;
        }
    } else {
#pragma unroll
        for (int k = 0; k < CS_PER * LANES; k++)
            if (base * LANES + k < points * LANES) out[base * LANES + k] = v[k];
    }
}

// ---- binary op with a shorter, repeated operand: data[i] = data[i] OP w[i % w_points] (points) -----------------------
template <typename T, int OP, bool CPX>
__global__ void smaller_kernel(T* __restrict__ data, const T* __restrict__ w, long long points, long long w_points) {
    typedef typename CpxOf<T>::type C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < points; i += stride) {
        const long long j = i % w_points;
        if (CPX) reinterpret_cast<C*>(data)[i] = ew_complex_op<OP>(reinterpret_cast<const C*>(data)[i], reinterpret_cast<const C*>(w)[j]);
        else data[i] = ew_real_op<OP>(data[i], w[j]);
    }
}

// ---- split / merge: element i <-> part i % parts, position i / parts ------------------------------------
template <typename T> struct PartPtrs { T* p[64]; };
template <typename T>
__global__ void split_merge_kernel(T* __restrict__ whole, PartPtrs<T> parts, int nparts, long long elems, int esz, int merge) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < elems; i += stride) {
        T* part = parts.p[i % nparts];
        const long long pos = i / nparts;
        for (int c = 0; c < esz; c++) {
            if (merge) whole[i * esz + c] = part[pos * esz + c];
            else part[pos * esz + c] = whole[i * esz + c];
        }
    }
}

// ---- set_real_imag / set_mag_phase ------------------------------------------------------------------------
template <typename T>
__global__ void compose_kernel(const T* __restrict__ a, const T* __restrict__ b, typename CpxOf<T>::type* __restrict__ out, long long points,
                               int polar) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < points; i += stride) out[i] = polar ? c_from_polar(a[i], b[i]) : mk<T>(a[i], b[i]);
}

// ---- interpolate_hermite -----------------------------------------------------------------------------------
__device__ __forceinline__ float ctr(long long i, float) { return i >= 16777216ll ? 16777216.0f : (float)i; }
__device__ __forceinline__ double ctr(long long i, double) { return i >= 9007199254740992ll ? 9007199254740992.0 : (double)i; }
template <typename T>
__global__ void hermite_kernel(const T* __restrict__ x, T* __restrict__ y, long long n, long long dest_len, long long start, T F, T d) {
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long end = start + 1;
    const T half = (T)0.5, c15 = (T)1.5, two = (T)2, c25 = (T)2.5;
    for (; k < dest_len; k += stride) {
        const T rounded = add_rn(div_rn(ctr(k, (T)0), F), d);
        const T bf = (T)floor(rounded);
        long long b = (long long)bf;
        T y0, y1, y2, y3;
        if (k < start) {
            if (b < 0) b = 0;
            if (b > n - 3) b = n - 3;                    // the reference asserts b == 0 here; clamp instead of panicking
            y1 = x[b]; y2 = x[b + 1]; y3 = x[b + 2];
            y0 = sub_rn(y1, sub_rn(y2, y1));
        } else if (k < dest_len - end) {
            if (b < 1) b = 1;
            if (b > n - 3) b = n - 3;
            y0 = x[b - 1]; y1 = x[b]; y2 = x[b + 1]; y3 = x[b + 2];
        } else {
            if (b < 1) b = 1;
            if (b > n - 1) b = n - 1;
            y0 = x[b - 1]; y1 = x[b];
            y2 = b < n - 1 ? x[b + 1] : add_rn(y1, sub_rn(y1, y0));
            y3 = b < n - 2 ? x[b + 2] : add_rn(y2, sub_rn(y2, y1));
        }
        const T xx = sub_rn(rounded, bf), x2 = mul_rn(xx, xx);
        const T a0 = add_rn(sub_rn(add_rn(mul_rn(-half, y0), mul_rn(c15, y1)), mul_rn(c15, y2)), mul_rn(half, y3));
        const T a1 = sub_rn(add_rn(sub_rn(y0, mul_rn(c25, y1)), mul_rn(two, y2)), mul_rn(half, y3));
        const T a2 = add_rn(mul_rn(-half, y0), mul_rn(half, y2));
        y[k] = add_rn(add_rn(add_rn(mul_rn(mul_rn(a0, xx), x2), mul_rn(a1, x2)), mul_rn(a2, xx)), y1);
    }
}

}  // namespace

template <typename T>
int math_unary(int op, void* data, size_t elems, int is_complex, double arg, cudaStream_t st) {
    if (!elems) return 0;
    const T a = (T)arg;
    T ln_arg;   // `base.ln()` evaluated in T
    if (sizeof(T) == 4) ln_arg = (T)logf((float)a); else ln_arg = (T)log((double)a);
    const long long items = (long long)elems * (is_complex ? 2 : 1) * (long long)sizeof(T) / 16 + 1;
    const unsigned grid = grid_stride_blocks(items);
    if (is_complex)
        math_complex_kernel<T><<<grid, GRID_STRIDE_THREADS, 0, st>>>(reinterpret_cast<typename CpxOf<T>::type*>(data), (long long)elems, op, a, ln_arg);
    else math_real_kernel<T><<<grid, GRID_STRIDE_THREADS, 0, st>>>(reinterpret_cast<T*>(data), (long long)elems, op, a, ln_arg);
    BDSP_LAUNCHED();
    return 0;
}

template <typename T>
int math_unwrap(void* data, size_t n, double divisor, cudaStream_t st) {
    if (n < 2) return 0;
    unwrap_kernel<T><<<1, 32, 0, st>>>(reinterpret_cast<T*>(data), (long long)n, (T)divisor);
    BDSP_LAUNCHED();
    return 0;
}

template <typename T>
int math_diff(const void* in, void* out, size_t n_out_scalars, int step, int with_start, cudaStream_t st) {
    if (!n_out_scalars) return 0;
    return launch_grid_stride(diff_kernel<T>, (long long)n_out_scalars, st, reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out),
                              (long long)n_out_scalars, step, with_start);
}

size_t math_cumsum_workspace(size_t points, int lanes, size_t elem_size) {
    const size_t per_block = (size_t)CS_THREADS * CS_PER;
    return ((points + per_block - 1) / per_block) * (size_t)lanes * elem_size;
}

template <typename T>
int math_cumsum(const void* in, void* out, void* work, size_t points, int lanes, cudaStream_t st) {
    if (!points) return 0;
    const size_t per_block = (size_t)CS_THREADS * CS_PER;
    const unsigned nblocks = (unsigned)((points + per_block - 1) / per_block);
    const T* i = reinterpret_cast<const T*>(in);
    T* o = reinterpret_cast<T*>(out);
    T* w = reinterpret_cast<T*>(work);
    if (lanes == 1) cumsum_totals_kernel<T, 1><<<nblocks, CS_THREADS, 0, st>>>(i, w, (long long)points);
    else cumsum_totals_kernel<T, 2><<<nblocks, CS_THREADS, 0, st>>>(i, w, (long long)points);
    BDSP_LAUNCHED();
    cumsum_scan_totals_kernel<T><<<lanes, 1024, 0, st>>>(w, (long long)nblocks, lanes);
    BDSP_LAUNCHED();
    if (lanes == 1) cumsum_apply_kernel<T, 1><<<nblocks, CS_THREADS, 0, st>>>(i, o, w, (long long)points);
    else cumsum_apply_kernel<T, 2><<<nblocks, CS_THREADS, 0, st>>>(i, o, w, (long long)points);
    BDSP_LAUNCHED();
    return 0;
}

template <typename T>
int math_binary_smaller(int op, void* data, const void* w, size_t points, size_t w_points, int is_complex, cudaStream_t st) {
    if (!points) return 0;
    auto run = [&](auto kernel) {
        return launch_grid_stride(kernel, (long long)points, st, reinterpret_cast<T*>(data), reinterpret_cast<const T*>(w), (long long)points,
                                  (long long)w_points);
    };
    if (is_complex) {
        if (op == EW_ADD) return run(smaller_kernel<T, EW_ADD, true>);
        if (op == EW_SUB) return run(smaller_kernel<T, EW_SUB, true>);
        if (op == EW_MUL) return run(smaller_kernel<T, EW_MUL, true>);
        return run(smaller_kernel<T, EW_DIV, true>);
    }
    if (op == EW_ADD) return run(smaller_kernel<T, EW_ADD, false>);
    if (op == EW_SUB) return run(smaller_kernel<T, EW_SUB, false>);
    if (op == EW_MUL) return run(smaller_kernel<T, EW_MUL, false>);
    return run(smaller_kernel<T, EW_DIV, false>);
}

template <typename T>
int math_split_merge(void* whole, void* const* parts, int nparts, size_t elems, int esz, int merge, cudaStream_t st) {
    if (!elems) return 0;
    if (nparts > 64) { set_last_error("split_into / merge: at most 64 parts"); return 7; }
    PartPtrs<T> pp;
    for (int i = 0; i < nparts; i++) pp.p[i] = reinterpret_cast<T*>(parts[i]);
    return launch_grid_stride(split_merge_kernel<T>, (long long)elems, st, reinterpret_cast<T*>(whole), pp, nparts, (long long)elems, esz, merge);
}

template <typename T>
int math_compose(const void* a, const void* b, void* out, size_t points, int polar, cudaStream_t st) {
    if (!points) return 0;
    return launch_grid_stride(compose_kernel<T>, (long long)points, st, reinterpret_cast<const T*>(a), reinterpret_cast<const T*>(b),
                              reinterpret_cast<typename CpxOf<T>::type*>(out), (long long)points, polar);
}

template <typename T>
int math_hermite(const void* x, void* y, size_t n, size_t dest_len, size_t start, double factor, double delay, cudaStream_t st) {
    if (!dest_len) return 0;
    return launch_grid_stride(hermite_kernel<T>, (long long)dest_len, st, reinterpret_cast<const T*>(x), reinterpret_cast<T*>(y), (long long)n,
                              (long long)dest_len, (long long)start, (T)factor, (T)delay);
}

#define BDSP_INST(T)                                                                                   \
    template int math_unary<T>(int, void*, size_t, int, double, cudaStream_t);                         \
    template int math_unwrap<T>(void*, size_t, double, cudaStream_t);                                  \
    template int math_diff<T>(const void*, void*, size_t, int, int, cudaStream_t);                     \
    template int math_cumsum<T>(const void*, void*, void*, size_t, int, cudaStream_t);                 \
    template int math_binary_smaller<T>(int, void*, const void*, size_t, size_t, int, cudaStream_t);   \
    template int math_split_merge<T>(void*, void* const*, int, size_t, int, int, cudaStream_t);        \
    template int math_compose<T>(const void*, const void*, void*, size_t, int, cudaStream_t);          \
    template int math_hermite<T>(const void*, void*, size_t, size_t, size_t, double, double, cudaStream_t);
BDSP_INST(float)
BDSP_INST(double)
#undef BDSP_INST

}  // namespace bdsp
