// Interpolation kernels: interpolatef (polyphase FIR, integer factor; per-output taps otherwise)
// and interpolate_lin.  Reference: vector/src/vector_types/time_freq/interpolation.rs:92-482 and
// real_interpolation.rs:33-71.
#include "interp.cuh"

namespace bdsp {

// ------------------------------------------------------------------------------------------
// Integer-factor polyphase kernel.
//   y[r*F + s] = sum_{j < J} x[(r - L - 1 + j) mod N] * tab[sel][s][j],   J = 2L + 3
// `tab` holds two tables over the same window superset [r-L-1, r+L+1]:
//   sel 0 = interior outputs  (interpolate_priv_simd, interpolation.rs:244-275; taps reversed)
//   sel 1 = edge outputs      (interpolate_priv_simd_step, :293-315)
// built on the host in precision T exactly as function_to_vectors (:133-181) evaluates them.
// ------------------------------------------------------------------------------------------
#define IP_THREADS 256

// generic-factor variant of the same polyphase kernel for F > 8: one thread per output
template <typename T, bool CPLX>
__global__ void interp_poly_generic_kernel(const void* __restrict__ x_, void* __restrict__ y_, const T* __restrict__ tab,
                                           long long N, long long new_points, int F, int L, long long scalar_len) {
    typedef typename CpxOf<T>::type C;
    typedef typename std::conditional<CPLX, C, T>::type X;
    const int J = 2 * L + 3;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= new_points) return;
    long long r = i / F; int s = (int)(i - r * F);
    bool interior = (i >= scalar_len) && (i < new_points - scalar_len);
    const T* t = tab + (interior ? 0 : F * J) + s * J;
    long long g = (r - L - 1) % N; if (g < 0) g += N;
    X acc = X();
    for (int j = 0; j < J; j++) {
        X xv = reinterpret_cast<const X*>(x_)[g];
        if constexpr (CPLX) { acc.x += xv.x * t[j]; acc.y += xv.y * t[j]; } else acc += xv * t[j];
        g++; if (g >= N) g -= N;
    }
    reinterpret_cast<X*>(y_)[i] = acc;
}

// ------------------------------------------------------------------------------------------
// Register-tiled polyphase kernel (the one used for F <= 8): a thread owns RP consecutive input
// positions x F phases = RP*F accumulators; per tap it issues ONE shared load for the sliding input
// window and one (vector, warp-uniform) load for the F taps, i.e. RP*F FMAs per two shared loads.
// CTAs whose outputs touch the first/last (2L+1)*F outputs (different tap window there, see the header
// comment) take the per-output path of interp_poly_generic_kernel's logic.
// ------------------------------------------------------------------------------------------
#define IP2_THREADS 256
__device__ __forceinline__ int ip_skew(int i) { return i + (i >> 5); }   // lanes are RP elements apart

template <typename T, bool CPLX, int FMAX, int RP>
__global__ void __launch_bounds__(IP2_THREADS)
interp_poly_tiled_kernel(const void* __restrict__ x_, void* __restrict__ y_, const T* __restrict__ tab, long long N,
                         long long new_points, int F, int L, long long scalar_len) {
    typedef typename CpxOf<T>::type C;
    typedef typename std::conditional<CPLX, C, T>::type X;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int J = 2 * L + 3;
    constexpr int POS = IP2_THREADS * RP;                     // input positions per CTA
    T* stab = reinterpret_cast<T*>(smem_raw);                 // interior taps, [J][FMAX]
    X* sx = reinterpret_cast<X*>(stab + ((J * FMAX + 3) & ~3));
    // the LAST tile of a vector takes the slow per-output path with wrap-around: it runs first (CTA 0), next to the first tile
    // (CTA 1), so that its latency-bound loop overlaps the whole grid instead of forming the kernel's tail
    const long long tile_ix = blockIdx.x == 0 ? (long long)gridDim.x - 1 : (long long)blockIdx.x - 1;
    const long long r0 = tile_ix * POS;
    const bool interior = (r0 * F >= scalar_len) && ((r0 + POS) * F <= new_points - scalar_len);
    if (!interior) {
        // edge CTA: one output at a time, tap table chosen per output
        for (long long i = r0 * F + threadIdx.x; i < (r0 + POS) * F && i < new_points; i += IP2_THREADS) {
            const long long r = i / F; const int s = (int)(i - r * F);
            const bool in = (i >= scalar_len) && (i < new_points - scalar_len);
            const T* t = tab + (in ? 0 : F * J) + s * J;
            long long g = (r - L - 1) % N; if (g < 0) g += N;
            X acc = X();
            for (int j = 0; j < J; j++) {
                const X xv = reinterpret_cast<const X*>(x_)[g];
                if constexpr (CPLX) { acc.x += xv.x * t[j]; acc.y += xv.y * t[j]; } else acc += xv * t[j];
                g++; if (g >= N) g -= N;
            }
            reinterpret_cast<X*>(y_)[i] = acc;
        }
        return;
    }
    for (int i = threadIdx.x; i < J * FMAX; i += IP2_THREADS) {
        const int j = i / FMAX, s = i - j * FMAX;
        stab[i] = s < F ? tab[s * J + j] : (T)0;
    }
    const int W = POS + J - 1;
    {
        long long g = r0 - L - 1 + threadIdx.x;               // interior: no wrap-around
        for (int w = threadIdx.x; w < W; w += IP2_THREADS) {
            sx[ip_skew(w)] = reinterpret_cast<const X*>(x_)[g];
            g += IP2_THREADS;
        }
    }
    __syncthreads();
    X acc[RP][FMAX];
#pragma unroll
    for (int p = 0; p < RP; p++)
#pragma unroll
        for (int s = 0; s < FMAX; s++) acc[p][s] = X();
    const int base = threadIdx.x * RP;
    X win[RP];                                                 // win[(j + p) % RP] = window[base + j + p]
#pragma unroll
    for (int p = 0; p < RP; p++) win[p] = sx[ip_skew(base + p)];
    for (int jb = 0; jb < J; jb += RP) {
#pragma unroll
        for (int jj = 0; jj < RP; jj++) {
            const int j = jb + jj;
            if (j < J) {
                T tp[FMAX];
#pragma unroll
                for (int s = 0; s < FMAX; s++) tp[s] = stab[j * FMAX + s];
#pragma unroll
                for (int p = 0; p < RP; p++) {
                    const X xv = win[(jj + p) % RP];
                    if constexpr (std::is_same<T, float>::value && !CPLX) {
                        // packed FP32x2: two phases per FFMA2 (scalar 3-register FFMA issues at ~0.55/clk/SMSP on sm_100)
                        const float2 xx = make_float2(xv, xv);
#pragma unroll
                        for (int s = 0; s < FMAX; s += 2) {
                            const float2 r = __ffma2_rn(xx, make_float2(tp[s], tp[s + 1]), make_float2(acc[p][s], acc[p][s + 1]));
                            acc[p][s] = r.x; acc[p][s + 1] = r.y;
                        }
                    } else if constexpr (std::is_same<T, float>::value && CPLX) {
#pragma unroll
                        for (int s = 0; s < FMAX; s++) acc[p][s] = __ffma2_rn(xv, make_float2(tp[s], tp[s]), acc[p][s]);
                    } else {
#pragma unroll
                        for (int s = 0; s < FMAX; s++) {
                            if constexpr (CPLX) { acc[p][s].x += xv.x * tp[s]; acc[p][s].y += xv.y * tp[s]; }
                            else acc[p][s] += xv * tp[s];
                        }
                    }
                }
                win[jj] = sx[ip_skew(base + j + RP)];
            }
        }
    }
    // stage the RP*F results of every thread in shared memory (padded rows) and write them out with
    // fully coalesced stores: consecutive threads -> consecutive outputs
    __syncthreads();
    X* so = reinterpret_cast<X*>(smem_raw);
    constexpr int ROW = RP * FMAX + 4;
#pragma unroll
    for (int p = 0; p < RP; p++)
#pragma unroll
        for (int s = 0; s < FMAX; s++)
            if (s < F) so[threadIdx.x * ROW + p * F + s] = acc[p][s];
    __syncthreads();
    const int per_thread = RP * F;
    const int total = POS * F;
    X* yo = reinterpret_cast<X*>(y_) + r0 * F;
    for (int o = threadIdx.x; o < total; o += IP2_THREADS) {
        const int tt = o / per_thread, e = o - tt * per_thread;
        yo[o] = so[tt * ROW + e];
    }
}

// ------------------------------------------------------------------------------------------
// Real f32, F <= 4 (BASELINE config C4a): 8 positions x 4 phases per thread, everything packed FP32x2.
// The input window is stored DUPLICATED ({x, x} pairs) so that one 64-bit shared load yields the splat
// operand of FFMA2 without a MOV; per tap and thread: 1 LDS.128 (4 taps, warp-uniform) + 1 LDS.64 +
// 16 FFMA2 for 32 outputs.  y16: y is 16-byte aligned, so F == 4 can be written with float4 stores (the row entry point
// accepts any float-aligned output).
// ------------------------------------------------------------------------------------------
// threads per CTA: small CTAs keep the barrier-separated load / compute / store phases of different CTAs overlapping on
// the SM.  Measured on B200 (C4a, 2^24 samples x4): 256 threads 0.160 ms, 128: 0.142, 64: 0.133, 32: 0.136 while the vector's last
// tile was the kernel's tail (+ ~25 us on every variant); with the end tiles first: 256: 0.117, 128: 0.109, 64: 0.111, 32: 0.118.
#define IPF_THREADS 64
// positions per thread (IPF_LRP = log2): 8 -> 64 registers, 1024 threads per SM; 16 -> half the shared loads and loop overhead
// per FFMA2, but 127 registers and 512 threads per SM.  Measured on B200 (C4a): 8 positions 0.131 ms; 16 positions 0.162 ms
// (64-thread CTAs), 0.160 (32), 0.185 (128): the FMA pipe needs the resident warps more than it needs fewer instructions
#define IPF_LRP 3
#define IPF_RP (1 << IPF_LRP)
#define IPF_POS (IPF_THREADS * IPF_RP)
#define IPF_ROW (4 * IPF_RP + 2)   // staging row stride in floats (odd number of 8-byte words: conflict-free 64-bit stores)
__device__ __forceinline__ int ipf_skew(int i) { return i + (i >> IPF_LRP); }

__global__ void __launch_bounds__(IPF_THREADS, 1024 / IPF_THREADS)
interp_poly_f32_kernel(const float* __restrict__ x, float* __restrict__ y, const float* __restrict__ tab, long long N,
                       long long new_points, int F, int L, long long scalar_len, bool y16) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int J = 2 * L + 3;
    const int JI = 2 * L + 2;                                  // the last window slot has no interior tap
    float4* stab = reinterpret_cast<float4*>(smem_raw);        // interior taps, [J] x {s0, s1, s2, s3}
    float2* sxx = reinterpret_cast<float2*>(stab + J);         // duplicated window
    // Tiles that touch the ends of the vector run the same packed path over a window loaded with wrap-around (interior
    // outputs never need wrapped samples; the read-ahead slots and the outputs of the edge regions merely have to stay in
    // bounds) and then overwrite the (2 L + 1) F outputs of each edge region with the per-output form below.  They used to
    // take the per-output form for all their 2048 outputs - 27 latency-bound loads per output on 64 threads - and the last
    // tile, scheduled last, was the kernel's tail (ncu: SMs active for 70 % of the duration).  Edge tiles still go first.
    const long long tile_ix = blockIdx.x == 0 ? (long long)gridDim.x - 1 : (long long)blockIdx.x - 1;
    const long long r0 = tile_ix * IPF_POS;
    const bool interior = (r0 * F >= scalar_len) && ((r0 + IPF_POS) * F <= new_points - scalar_len);
    for (int j = threadIdx.x; j < J; j += IPF_THREADS) {
        float4 t4;
        t4.x = tab[j];
        t4.y = F > 1 ? tab[J + j] : 0.f;
        t4.z = F > 2 ? tab[2 * J + j] : 0.f;
        t4.w = F > 3 ? tab[3 * J + j] : 0.f;
        stab[j] = t4;
    }
    const int W = IPF_POS + JI - 1 + IPF_RP;
    {
        if (interior) {
            const float* xs = x + (r0 - L - 1);
            const long long wmax = N - 1 - (r0 - L - 1);      // the last IPF_RP slots are read ahead of use: keep them inside the vector
            for (int w = threadIdx.x; w < W; w += IPF_THREADS) {
                const float v = xs[w <= wmax ? w : (int)wmax];
                sxx[ipf_skew(w)] = make_float2(v, v);
            }
        } else {
            long long g = (r0 - L - 1 + threadIdx.x) % N; if (g < 0) g += N;
            const long long adv = IPF_THREADS % N;
            for (int w = threadIdx.x; w < W; w += IPF_THREADS) {
                const float v = x[g];
                sxx[ipf_skew(w)] = make_float2(v, v);
                g += adv; if (g >= N) g -= N;
            }
        }
    }
    __syncthreads();
    float2 acc[IPF_RP][2];
#pragma unroll
    for (int p = 0; p < IPF_RP; p++) { acc[p][0] = make_float2(0.f, 0.f); acc[p][1] = make_float2(0.f, 0.f); }
    // window slot k of this thread lives at sxx[ipf_skew(8*tid + k)] = wbase[k + (k >> 3)]: within one block of 8 taps
    // the 8 slots that enter the window are contiguous, and the block start advances by 9 float2
    const float2* wbase = sxx + threadIdx.x * (IPF_RP + 1);
    float2 win[IPF_RP];
#pragma unroll
    for (int p = 0; p < IPF_RP; p++) win[p] = wbase[p];
    const int full = JI & ~(IPF_RP - 1);
    const float2* wp = wbase + (IPF_RP + 1);
    const float4* tp = stab;
    for (int jb = 0; jb < full; jb += IPF_RP, wp += IPF_RP + 1, tp += IPF_RP) {
#pragma unroll
        for (int jj = 0; jj < IPF_RP; jj++) {
            const float4 t4 = tp[jj];
            const float2 ta = make_float2(t4.x, t4.y), tb = make_float2(t4.z, t4.w);
#pragma unroll
            for (int p = 0; p < IPF_RP; p++) {
                const float2 xx = win[(jj + p) % IPF_RP];
                acc[p][0] = __ffma2_rn(xx, ta, acc[p][0]);
                acc[p][1] = __ffma2_rn(xx, tb, acc[p][1]);
            }
            win[jj] = wp[jj];
        }
    }
#pragma unroll
    for (int jj = 0; jj < IPF_RP; jj++) {
        if (full + jj < JI) {      // remaining taps (warp-uniform condition)
            const float4 t4 = tp[jj];
            const float2 ta = make_float2(t4.x, t4.y), tb = make_float2(t4.z, t4.w);
#pragma unroll
            for (int p = 0; p < IPF_RP; p++) {
                const float2 xx = win[(jj + p) % IPF_RP];
                acc[p][0] = __ffma2_rn(xx, ta, acc[p][0]);
                acc[p][1] = __ffma2_rn(xx, tb, acc[p][1]);
            }
            win[jj] = wp[jj];
        }
    }
    __syncthreads();
    float* so = reinterpret_cast<float*>(smem_raw);
    if (F == 4) {
#pragma unroll
        for (int p = 0; p < IPF_RP; p++) {
            *reinterpret_cast<float2*>(so + threadIdx.x * IPF_ROW + 4 * p) = acc[p][0];
            *reinterpret_cast<float2*>(so + threadIdx.x * IPF_ROW + 4 * p + 2) = acc[p][1];
        }
    } else {
#pragma unroll
        for (int p = 0; p < IPF_RP; p++) {
            const float a4[4] = {acc[p][0].x, acc[p][0].y, acc[p][1].x, acc[p][1].y};
#pragma unroll
            for (int s = 0; s < 4; s++)
                if (s < F) so[threadIdx.x * IPF_ROW + p * F + s] = a4[s];
        }
    }
    __syncthreads();
    float* yo = y + r0 * F;
    if (F == 4 && y16) {   // 32 outputs per staging row: no integer division in the copy-out loop; 16-byte stores (y 16-byte aligned)
#pragma unroll
        for (int it = 0; it < IPF_RP; it++) {
            const int o = 4 * (threadIdx.x + IPF_THREADS * it);
            const float* sp = so + (o >> (IPF_LRP + 2)) * IPF_ROW + (o & (4 * IPF_RP - 1));
            const float2 a = *reinterpret_cast<const float2*>(sp), b = *reinterpret_cast<const float2*>(sp + 2);
            if (interior || r0 * F + o + 3 < new_points) *reinterpret_cast<float4*>(yo + o) = make_float4(a.x, a.y, b.x, b.y);
            else
                for (int e = 0; e < 4; e++)
                    if (r0 * F + o + e < new_points) yo[o + e] = sp[e];
        }
    } else {
        const int per_thread = IPF_RP * F;
        const int total = IPF_POS * F;
        for (int o = threadIdx.x; o < total; o += IPF_THREADS) {
            const int tt = o / per_thread, e = o - tt * per_thread;
            if (interior || r0 * F + o < new_points) yo[o] = so[tt * IPF_ROW + e];
        }
    }
    if (!interior) {
        // outputs of the two edge regions inside this tile: taps chosen per output, circular window (interpolation.rs:191-290)
        __syncthreads();
        const long long lo = r0 * F, hi = (r0 + IPF_POS) * F < new_points ? (r0 + IPF_POS) * F : new_points;
        const long long b0 = hi < scalar_len ? hi : scalar_len;                     // end of the leading edge region in this tile
        long long a1 = lo > new_points - scalar_len ? lo : new_points - scalar_len;   // start of the trailing one
        if (a1 < b0) a1 = b0;                                                        // (short vectors: the regions meet)
        for (int pass = 0; pass < 2; pass++) {
            const long long a = pass == 0 ? lo : a1;
            const long long b = pass == 0 ? b0 : hi;
            for (long long i = a + threadIdx.x; i < b; i += IPF_THREADS) {
                const long long r = i / F; const int s = (int)(i - r * F);
                const float* t = tab + F * J + s * J;
                long long g = (r - L - 1) % N; if (g < 0) g += N;
                float acc = 0.f;
                for (int j = 0; j < J; j++) {
                    acc += x[g] * t[j];
                    g++; if (g >= N) g -= N;
                }
                y[i] = acc;
            }
        }
    }
}

template <typename T>
int interp_poly(const void* x, void* y, const T* tab_dev, size_t N, size_t new_points, int F, int L, int is_complex,
                cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const long long scalar_len = (long long)(2 * L + 1) * F;
    const int J = 2 * L + 3;
    if (F <= 8) {
        const size_t xs = is_complex ? sizeof(C) : sizeof(T);
        const long long rows = ((long long)new_points + F - 1) / F;
#define BDSP_IP2(CP, FM, RPV)                                                                                          \
    do {                                                                                                               \
        const int pos = IP2_THREADS * RPV;                                                                             \
        const size_t wlen = (size_t)pos + J + RPV + 1;                                                                 \
        size_t smem = (((size_t)J * FM + 3) & ~(size_t)3) * sizeof(T) + (wlen + wlen / 32 + 2) * xs;                   \
        const size_t stage = (size_t)IP2_THREADS * (RPV * FM + 4) * xs;                                                \
        if (smem < stage) smem = stage;                                                                                \
        const long long grid = (rows + pos - 1) / pos;                                                                 \
        if (smem > 48 * 1024) BDSP_CUDA_OK(cudaFuncSetAttribute(interp_poly_tiled_kernel<T, CP, FM, RPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        interp_poly_tiled_kernel<T, CP, FM, RPV><<<(unsigned)grid, IP2_THREADS, smem, st>>>(x, y, tab_dev, (long long)N, (long long)new_points, F, L, scalar_len); \
    } while (0)
        if (is_complex) { if (F <= 4) BDSP_IP2(true, 4, 2); else BDSP_IP2(true, 8, 1); }
        else if (F <= 4 && sizeof(T) == 4) {
            const size_t wlen = (size_t)IPF_POS + J + 2 * IPF_RP;
            size_t smem = (size_t)J * 16 + (wlen + wlen / IPF_RP + 2) * 8;
            const size_t stage = (size_t)IPF_THREADS * IPF_ROW * 4;
            if (smem < stage) smem = stage;
            const long long grid = (rows + IPF_POS - 1) / IPF_POS;
            static PerDeviceOnce configured;
            if (configured.need()) {
                BDSP_CUDA_OK(cudaFuncSetAttribute(interp_poly_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem > 48 * 1024 ? smem : 48 * 1024)));
                BDSP_CUDA_OK(cudaFuncSetAttribute(interp_poly_f32_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                configured.mark();
            }
            interp_poly_f32_kernel<<<(unsigned)grid, IPF_THREADS, smem, st>>>(reinterpret_cast<const float*>(x), reinterpret_cast<float*>(y),
                                                                              reinterpret_cast<const float*>(tab_dev), (long long)N,
                                                                              (long long)new_points, F, L, scalar_len,
                                                                              (reinterpret_cast<uintptr_t>(y) & 15) == 0);
        }
        else { if (F <= 4) BDSP_IP2(false, 4, 4); else BDSP_IP2(false, 8, 2); }
#undef BDSP_IP2
    } else {
        const long long grid = ((long long)new_points + 255) / 256;
        if (is_complex) interp_poly_generic_kernel<T, true><<<(unsigned)grid, 256, 0, st>>>(x, y, tab_dev, (long long)N, (long long)new_points, F, L, scalar_len);
        else interp_poly_generic_kernel<T, false><<<(unsigned)grid, 256, 0, st>>>(x, y, tab_dev, (long long)N, (long long)new_points, F, L, scalar_len);
    }
    BDSP_LAUNCHED();
    return 0;
}

// ------------------------------------------------------------------------------------------
// Non-integer factor: interpolate_priv_scalar (interpolation.rs:92-131).  Taps are evaluated per
// output on the device in precision T for the two built-in impulse responses
// (conv_types.rs:406-423 RaisedCosine, :479-487 Sinc).
// ------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ T pi_t() { return (T)3.14159265358979323846; }

template <typename T> __device__ __forceinline__ T sinc_calc(T x) {
    if (x == (T)0) return (T)1;
    T pi_x = pi_t<T>() * x;
    return sin(pi_x) / pi_x;
}

template <typename T> __device__ __forceinline__ T rc_calc(T x, T rolloff) {
    if (x == (T)0) return (T)1;
    const T one = (T)1, two = (T)2, pi = pi_t<T>();
    const T four = two * two;
    if (fabs(x) == one / (two * rolloff)) {
        T arg = pi / two / rolloff;
        return sin(arg) / arg * pi / four;
    }
    T pi_x = pi * x;
    T arg = two * rolloff * x;
    return sin(pi_x) * cos(pi_x * rolloff) / pi_x / (one - (arg * arg));
}

template <typename T, bool CPLX>
__global__ void interp_frac_kernel(const void* __restrict__ x_, void* __restrict__ y_, long long N, long long new_points,
                                   T factor, T delay, int L, int kind, T rolloff) {
    typedef typename CpxOf<T>::type C;
    typedef typename std::conditional<CPLX, C, T>::type X;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= new_points) return;
    const T center = (T)i / factor;
    const T rounded = floor(center);
    long long r = (long long)rounded;
    T j = -(T)L - (center - rounded) + delay;
    long long g = (r - L) % N; if (g < 0) g += N;
    X acc = X();
    for (int k = 0; k < 2 * L + 1; k++) {
        const T t = kind == 0 ? sinc_calc<T>(j) : rc_calc<T>(j, rolloff);
        X xv = reinterpret_cast<const X*>(x_)[g];
        if constexpr (CPLX) { acc.x += xv.x * t; acc.y += xv.y * t; } else acc += xv * t;
        j = j + (T)1;
        g++; if (g >= N) g -= N;
    }
    reinterpret_cast<X*>(y_)[i] = acc;
}

template <typename T>
int interp_frac(const void* x, void* y, size_t N, size_t new_points, double factor, double delay, int L, int kind,
                double rolloff, int is_complex, cudaStream_t st) {
    const long long grid = ((long long)new_points + 255) / 256;
    if (is_complex) interp_frac_kernel<T, true><<<(unsigned)grid, 256, 0, st>>>(x, y, (long long)N, (long long)new_points, (T)factor, (T)delay, L, kind, (T)rolloff);
    else interp_frac_kernel<T, false><<<(unsigned)grid, 256, 0, st>>>(x, y, (long long)N, (long long)new_points, (T)factor, (T)delay, L, kind, (T)rolloff);
    BDSP_LAUNCHED();
    return 0;
}

// ------------------------------------------------------------------------------------------
// interpolate_lin (real_interpolation.rs:33-71): every operation individually rounded in T.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float lin_eval(float i, float F, float d, const float* __restrict__ x, long long n) {
    float p = __fadd_rn(__fdiv_rn(i, F), d);
    float bf = floorf(p);
    long long b = (long long)bf;
    if (b < 0) b = 0;                // the reference panics on an out-of-range index; clamp instead
    if (b > n - 2) b = n - 2;
    float y0 = x[b], y1 = x[b + 1];
    return __fadd_rn(y0, __fmul_rn(__fsub_rn(y1, y0), __fsub_rn(p, bf)));
}
__device__ __forceinline__ double lin_eval(double i, double F, double d, const double* __restrict__ x, long long n) {
    double p = __dadd_rn(__ddiv_rn(i, F), d);
    double bf = floor(p);
    long long b = (long long)bf;
    if (b < 0) b = 0;
    if (b > n - 2) b = n - 2;
    double y0 = x[b], y1 = x[b + 1];
    return __dadd_rn(y0, __dmul_rn(__dsub_rn(y1, y0), __dsub_rn(p, bf)));
}

// The reference counts the output index in precision T by repeated `+ 1.0` (real_interpolation.rs:53,65);
// in f32 that counter stops advancing at 2^24 (Q7).  The same saturation is applied here so that the
// result is bit-identical to the reference for every length (and the read index stays in bounds).
__device__ __forceinline__ float counter_value(long long i, float) { return i >= 16777216ll ? 16777216.0f : (float)i; }
__device__ __forceinline__ double counter_value(long long i, double) { return i >= 9007199254740992ll ? 9007199254740992.0 : (double)i; }

template <typename T> struct alignas(16) LinPack { T v[16 / sizeof(T)]; };
// 16 bytes of output per thread and step (4 f32 / 2 f64 consecutive results)
template <typename T>
__global__ void interp_lin_kernel(const T* __restrict__ x, T* __restrict__ y, long long n, long long dest_len, T F, T d) {
    constexpr int W = 16 / sizeof(T);
    const long long nv = (dest_len - 1) / W;          // packs that do not contain the last element
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long v = i; v < nv; v += stride) {
        LinPack<T> p;
#pragma unroll
        for (int k = 0; k < W; k++) p.v[k] = lin_eval(counter_value(v * W + k, (T)0), F, d, x, n);
        reinterpret_cast<LinPack<T>*>(y)[v] = p;
    }
    const long long t = nv * W + i;
    if (t < dest_len) y[t] = t == dest_len - 1 ? x[n - 1] : lin_eval(counter_value(t, (T)0), F, d, x, n);
}

// Fast path, bit-identical to the kernel above: F is a power of two (i / F == i * (1/F) exactly, every other operation is
// the same individually rounded one), all indices fit 32 bits, one thread per pack of 4 outputs (no grid-stride loop).
// The generic kernel is issue-bound (IEEE division + 64-bit integer -> float conversion per output: ~40 instructions for
// 4 bytes written); this one needs about half of that.
__global__ void __launch_bounds__(256) interp_lin_pow2_f32_kernel(const float* __restrict__ x, float* __restrict__ y, unsigned n,
                                                                  unsigned dest_len, float invF, float d) {
    const unsigned nv = (dest_len - 1) / 4;
    const unsigned v = blockIdx.x * 256u + threadIdx.x;
    if (v < nv) {
        float4 r;
        float* rp = reinterpret_cast<float*>(&r);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float ci = fminf(__uint2float_rn(v * 4u + k), 16777216.0f);   // the reference's saturating f32 counter (Q7)
            const float p = __fadd_rn(__fmul_rn(ci, invF), d);
            const float bf = floorf(p);
            int b = __float2int_rz(bf);
            b = max(0, min(b, (int)n - 2));
            const float y0 = __ldg(x + b), y1 = __ldg(x + b + 1);
            rp[k] = __fadd_rn(y0, __fmul_rn(__fsub_rn(y1, y0), __fsub_rn(p, bf)));
        }
        reinterpret_cast<float4*>(y)[v] = r;
    } else if (v < nv + 4) {
        const unsigned t = nv * 4u + (v - nv);
        if (t < dest_len) {
            if (t == dest_len - 1) y[t] = x[n - 1];
            else {
                const float ci = fminf(__uint2float_rn(t), 16777216.0f);
                const float p = __fadd_rn(__fmul_rn(ci, invF), d);
                const float bf = floorf(p);
                int b = __float2int_rz(bf);
                b = max(0, min(b, (int)n - 2));
                const float y0 = x[b], y1 = x[b + 1];
                y[t] = __fadd_rn(y0, __fmul_rn(__fsub_rn(y1, y0), __fsub_rn(p, bf)));
            }
        }
    }
}

template <typename T>
int interp_lin(const void* x, void* y, size_t n, size_t dest_len, double factor, double delay, cudaStream_t st) {
    if (sizeof(T) == 4 && n >= 2 && dest_len >= 2 && dest_len < (1ull << 31) && n < (1ull << 31) && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
        const float F = (float)factor;
        int e = 0;
        const float m = frexpf(F, &e);
        if (F > 0.f && m == 0.5f && e > -100 && e < 100) {   // power of two: the quotient is an exact scaling
            const unsigned nv = (unsigned)((dest_len - 1) / 4);
            const unsigned grid = (nv + 4 + 255) / 256;
            interp_lin_pow2_f32_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), reinterpret_cast<float*>(y), (unsigned)n,
                                                            (unsigned)dest_len, 1.0f / F, (float)delay);
            BDSP_LAUNCHED();
            return 0;
        }
    }
    long long grid = ((long long)dest_len / (16 / (long long)sizeof(T)) + 255) / 256 + 1;
    const long long cap = (long long)sm_count() * 32;
    if (grid > cap) grid = cap;
    interp_lin_kernel<T><<<(unsigned)grid, 256, 0, st>>>(reinterpret_cast<const T*>(x), reinterpret_cast<T*>(y), (long long)n,
                                                       (long long)dest_len, (T)factor, (T)delay);
    BDSP_LAUNCHED();
    return 0;
}

#define BDSP_INST(T)                                                                                                  \
    template int interp_poly<T>(const void*, void*, const T*, size_t, size_t, int, int, int, cudaStream_t);             \
    template int interp_frac<T>(const void*, void*, size_t, size_t, double, double, int, int, double, int, cudaStream_t); \
    template int interp_lin<T>(const void*, void*, size_t, size_t, double, double, cudaStream_t);
BDSP_INST(float)
BDSP_INST(double)
#undef BDSP_INST

}  // namespace bdsp
