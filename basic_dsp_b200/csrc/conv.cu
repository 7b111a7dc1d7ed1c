// Convolution kernels: fused overlap-save fast convolution and direct circular FIR.
//
// Both compute the reference's centred circular convolution
//     y[i] = sum_{k<L} x[(i + cl - 1 - k) mod N] * h[k],   cl = L - L/2
// (ConvolutionOps::convolve_signal, vector/src/vector_types/time_freq/convolution.rs:477-542;
//  convolve_iteration, time_freq/mod.rs:456-473).  They replace the reference's overlap_discard
// (convolution.rs:304-461), its SIMD FIR (time_freq/mod.rs:531-610) and its OpenCL kernels
// conv_vecs_r/conv_vecs_c/multiply_vector (gpu_support/ocl/ocl_kernels32.rs).
#include <math.h>

#include <map>
#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

#include "conv.cuh"
#include "elementwise.cuh"
#include "fft.cuh"
#include "fft_core.cuh"
#include "olsi.cuh"

namespace bdsp {

// ------------------------------------------------------------------------------------------
// Overlap-save: one CTA = one block of M points of one vector, everything in shared memory:
//   load M inputs (circular) -> FFT -> * Hs (H/M, L2 resident) -> IFFT -> store M-L+1 outputs.
// HBM traffic per output sample: 8 B read * M/(M-L+1) + 8 B write (c32).
// ------------------------------------------------------------------------------------------
template <typename T, bool REAL>
__global__ void __launch_bounds__(sizeof(T) == 4 ? 1024 : 512)
ols_conv_kernel(const void* __restrict__ x_, void* __restrict__ y_, long long N, long long batch, int L, int log2M,
                long long blocks_per_vec, const typename CpxOf<T>::type* __restrict__ Hs,
                const typename CpxOf<T>::type* __restrict__ tw) {
    typedef typename CpxOf<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C* s = reinterpret_cast<C*>(smem_raw);
    const int M = 1 << log2M;
    const int step = M - L + 1;
    const int cl = L - L / 2;
    const long long vec = blockIdx.x / blocks_per_vec;
    const long long blk = blockIdx.x - vec * blocks_per_vec;
    const long long i0 = blk * step;              // first output index of this block
    long long p0 = (i0 - (L - cl)) % N;            // first input index (may be negative before wrap)
    if (p0 < 0) p0 += N;
    // ---- load (circular) ----
    {
        long long g = (p0 + threadIdx.x) % N;
        const long long adv = blockDim.x % N;
        for (int idx = threadIdx.x; idx < M; idx += blockDim.x) {
            C v;
            if (REAL) { v.x = reinterpret_cast<const T*>(x_)[vec * N + g]; v.y = 0; }
            else v = reinterpret_cast<const C*>(x_)[vec * N + g];
            s[spad(idx)] = v;
            g += adv; if (g >= N) g -= N;
        }
    }
    __syncthreads();
    block_fft<T, false>(s, log2M, 1, tw);
    // ---- spectrum multiply (Hs already holds the 1/M scaling) ----
    for (int idx = threadIdx.x; idx < M; idx += blockDim.x) {
        C v = s[spad(idx)];
        s[spad(idx)] = cmul(v, __ldg(&Hs[idx]));
    }
    __syncthreads();
    block_fft<T, true>(s, log2M, 1, tw);
    // ---- store the valid part: m in [L-1, M) -> y[i0 + m - (L-1)] ----
    for (int idx = threadIdx.x; idx < step; idx += blockDim.x) {
        long long i = i0 + idx;
        if (i < N) {
            C v = s[spad(idx + L - 1)];
            if (REAL) reinterpret_cast<T*>(y_)[vec * N + i] = v.x;
            else reinterpret_cast<C*>(y_)[vec * N + i] = v;
        }
    }
}

// Hs[k] = FFT_M(pad(h))[k] / M
template <typename T>
__global__ void ols_pad_h_kernel(const void* __restrict__ h_, typename CpxOf<T>::type* __restrict__ hp, int L, int M,
                                 int h_is_real) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    typename CpxOf<T>::type v = mk<T>(0, 0);
    if (i < L) {
        if (h_is_real) v.x = reinterpret_cast<const T*>(h_)[i];
        else v = reinterpret_cast<const typename CpxOf<T>::type*>(h_)[i];
    }
    hp[i] = v;
}

template <typename T> size_t ols_block_len(size_t L, bool complex_signal) {
    // same rule as the reference (fft_len >= 4*overlap, convolution.rs:323-331) with a 4096 floor so
    // that the block transform amortises its overlap; capped by the shared-memory transform limit.
    // c32 signals: fused 4096-point blocks up to 2046 taps (+ an 8192-point plan next to it, see OlsPlan::M2),
    // fused 8192-point blocks up to 4094 taps.
    if (sizeof(T) == 4 && complex_signal && L >= 2 && L <= 2046) return 4096;
    if (sizeof(T) == 4 && complex_signal && L >= 2 && L <= 4094) return 8192;
    // c64 signals: the fused 4096-point kernel (ols64.cu) up to 2048 taps - beyond 1025 taps its block efficiency drops below
    // the reference's 75 % rule, but it still beats the generic 8192-point blocks (2047 taps: 1.07 against 1.28 ms per 2^25 samples)
    if (sizeof(T) == 8 && complex_signal && L <= 2048) return 4096;
    size_t m = next_pow2(4 * (L > 1 ? L - 1 : 1));
    if (m < 4096) m = 4096;
    if (m > fft_block_max_n<T>()) m = fft_block_max_n<T>();
    return m;
}

// largest L the overlap-save blocks take
template <typename T> static size_t ols_max_taps() { return fft_block_max_n<T>() / 2; }

int ols4096_prepare(const void* Hs, void* Hpos, size_t L, cudaStream_t st);
int ols4096_convolve(const void* x, void* y, size_t N, size_t batch, size_t L, cudaTextureObject_t htex, cudaStream_t st);
int ols8192_prepare(const void* Hs, void* Hpos, size_t L, cudaStream_t st);
int ols8192_convolve(const void* x, void* y, size_t N, size_t batch, size_t L, cudaTextureObject_t htex, cudaStream_t st);
bool ols64_applicable(size_t N, size_t L, size_t M);
int ols64_convolve(const void* x, void* y, size_t N, size_t batch, size_t L, const void* Hs, cudaStream_t st);

namespace {
// Hs (2*M complex) <- FFT_M(pad(h)) / M, then the fused kernel's layout behind it (c32, M = 4096 / 8192)
template <typename T>
int ols_spectrum(const void* h, size_t L, int h_is_real, size_t M, bool fused, void** Hs_out, cudaTextureObject_t* tex, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    void* Hs = nullptr;
    BDSP_CUDA_OK(cudaMalloc(&Hs, 2 * M * sizeof(C)));
    ols_pad_h_kernel<T><<<(unsigned)((M + 255) / 256), 256, 0, st>>>(h, reinterpret_cast<C*>(Hs), (int)L, (int)M, h_is_real);
    int rc = cudaGetLastError() == cudaSuccess ? 0 : -1;
    count_launch();
    FftOpts o;
    o.scale = 1.0 / (double)M;
    if (!rc) rc = fft_exec<T>(Hs, Hs, M, 1, o, nullptr, 0, st);
    if (!rc && fused) {
        void* Hpos = reinterpret_cast<C*>(Hs) + M;
        rc = M == 4096 ? ols4096_prepare(Hs, Hpos, L, st) : ols8192_prepare(Hs, Hpos, L, st);
        if (!rc) {
            cudaResourceDesc rd = {};
            rd.resType = cudaResourceTypeLinear;
            rd.res.linear.devPtr = Hpos;
            rd.res.linear.desc = cudaCreateChannelDesc<float4>();
            rd.res.linear.sizeInBytes = 2 * M * sizeof(float);
            cudaTextureDesc td = {};
            td.readMode = cudaReadModeElementType;
            if (cudaCreateTextureObject(tex, &rd, &td, nullptr) != cudaSuccess) { set_last_error("ols plan: texture object"); rc = -1; }
        }
    }
    if (rc) { cudaFree(Hs); return rc; }
    *Hs_out = Hs;
    return 0;
}
}  // namespace

template <typename T>
OlsPlan* ols_plan_create(const void* h, size_t L, int h_is_real, bool complex_signal, cudaStream_t st) {
    if (!h || !L || L > ols_max_taps<T>()) { set_last_error("ols plan: unsupported impulse response length %zu", L); return nullptr; }
    OlsPlan* p = new OlsPlan();
    p->is64 = sizeof(T) == 8; p->L = L; p->h_is_real = h_is_real;
    if (cudaGetDevice(&p->device) != cudaSuccess) { delete p; return nullptr; }
    p->M = ols_block_len<T>(L, complex_signal);
    const bool fused = sizeof(T) == 4 && complex_signal && L >= 2 && (p->M == 4096 || p->M == 8192);
    int rc = ols_spectrum<T>(h, L, h_is_real, p->M, fused, &p->Hs, &p->htex, st);
    if (!rc && fused && p->M == 4096) {
        p->M2 = 8192;
        rc = ols_spectrum<T>(h, L, h_is_real, p->M2, true, &p->Hs2, &p->htex2, st);
    }
    if (rc) { ols_plan_destroy(p); return nullptr; }
    return p;
}

void ols_plan_destroy(OlsPlan* p) {
    if (!p) return;
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != p->device) cudaSetDevice(p->device);
    cudaDeviceSynchronize();    // kernels of any stream may still read the spectra
    if (p->htex) cudaDestroyTextureObject(p->htex);
    if (p->htex2) cudaDestroyTextureObject(p->htex2);
    if (p->Hs) cudaFree(p->Hs);
    if (p->Hs2) cudaFree(p->Hs2);
    if (cur != p->device) cudaSetDevice(cur);
    delete p;
}

const float2* olsi_twiddles(int M) {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) { set_last_error("ols%d: cudaGetDevice failed", M); return nullptr; }
    static std::mutex mu;
    static std::map<std::pair<int, int>, float2*> tables;   // (device, M)
    std::lock_guard<std::mutex> lk(mu);
    auto it = tables.find({d, M});
    if (it != tables.end()) return it->second;
    const int n1 = M / 16, n2 = M / 256;
    std::vector<float2> h(2 * n1);
    const long double tau = 2.0L * 3.14159265358979323846264338327950288L;
    for (int c = 0; c < n1; c++) {
        h[c].x = (float)cosl(-tau * (long double)c / (long double)M);
        h[c].y = (float)sinl(-tau * (long double)c / (long double)M);
    }
    for (int k = 0; k < 16; k++)
        for (int c = 0; c < n2; c++) {
            const long double a = -tau * (long double)((k * c) % n1) / (long double)n1;
            h[n1 + n2 * k + c].x = (float)cosl(a);
            h[n1 + n2 * k + c].y = (float)sinl(a);
        }
    float2* dev = nullptr;
    if (cudaMalloc(&dev, h.size() * sizeof(float2)) != cudaSuccess ||
        cudaMemcpy(dev, h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) {
        if (dev) cudaFree(dev);
        cudaGetLastError();
        set_last_error("ols%d: twiddle table allocation failed", M);
        return nullptr;
    }
    tables[{d, M}] = dev;
    return dev;
}

// generic overlap-save blocks of the plan's length M
template <typename T>
static int ols_generic_convolve(const OlsPlan* p, const void* x, void* y, size_t N, size_t batch, int is_real, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const size_t L = p->L, M = p->M;
    const size_t step = M - L + 1;
    const long long bpv = (long long)((N + step - 1) / step);
    const int log2M = ilog2(M);
    const int threads = block_fft_threads((int)M, 1);
    const size_t smem = spad_host(M) * sizeof(C);
    const long long grid = bpv * (long long)batch;
    if (grid > 0x7fffffffll) { set_last_error("ols_convolve: grid too large"); return -2; }
    const C* tw = twiddle_table<T>();
    if (!tw) return -1001;
    if (is_real) {
        if (smem > 48 * 1024) BDSP_CUDA_OK(cudaFuncSetAttribute(ols_conv_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ols_conv_kernel<T, true><<<(unsigned)grid, threads, smem, st>>>(x, y, (long long)N, (long long)batch, (int)L, log2M, bpv,
                                                                       reinterpret_cast<const C*>(p->Hs), tw);
    } else {
        if (smem > 48 * 1024) BDSP_CUDA_OK(cudaFuncSetAttribute(ols_conv_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ols_conv_kernel<T, false><<<(unsigned)grid, threads, smem, st>>>(x, y, (long long)N, (long long)batch, (int)L, log2M, bpv,
                                                                        reinterpret_cast<const C*>(p->Hs), tw);
    }
    BDSP_LAUNCHED();
    return 0;
}

// ------------------------------------------------------------------------------------------
// Direct circular FIR.  Tile of FIR_TILE outputs per CTA; the input window (tile + L - 1 halo,
// circular) and the taps are staged in shared memory; each thread produces FIR_U consecutive
// outputs from a sliding register window (one shared load of x and one broadcast load of a tap per
// FIR_U multiply-accumulates).
//   XC: x complex (else real), HC: taps complex (else real)
// ------------------------------------------------------------------------------------------
#define FIR_THREADS 256
#define FIR_U 8
#define FIR_TILE (FIR_THREADS * FIR_U)
// skewed window index: threads are FIR_U elements apart, the skew makes their banks distinct
__device__ __forceinline__ int fpad(int w) { return w + (w >> 3); }

template <typename T, bool XC, bool HC> struct FirTypes {
    typedef typename CpxOf<T>::type C;
};

template <typename T, bool XC, bool HC>
__global__ void __launch_bounds__(FIR_THREADS)
fir_kernel(const void* __restrict__ x_, void* __restrict__ y_, const void* __restrict__ h_, long long N, long long batch,
           int L, int cl, long long tiles_per_vec) {
    typedef typename CpxOf<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: taps (L entries of C), then the window (FIR_TILE + L - 1 entries of C, +pad)
    C* sh = reinterpret_cast<C*>(smem_raw);
    C* sx = sh + L;
    const unsigned tpv = (unsigned)tiles_per_vec;            // (the grid has fewer than 2^31 tiles)
    const unsigned vec_u = blockIdx.x / tpv;
    const long long vec = vec_u;
    const long long tile = blockIdx.x - vec_u * tpv;
    const long long i0 = tile * FIR_TILE;
    const int W = FIR_TILE + L - 1;
    // window element w corresponds to x[(i0 - (L - cl) + w) mod N]
    // (64-bit remainders cost ~100 instructions each: vectors longer than a tile + taps need conditional corrections only)
    const bool big = N >= (long long)FIR_TILE + L;
    long long p0 = i0 - (L - cl);
    if (big) { if (p0 < 0) p0 += N; }
    else { p0 %= N; if (p0 < 0) p0 += N; }
    for (int k = threadIdx.x; k < L; k += FIR_THREADS) {
        C t;
        if (HC) t = reinterpret_cast<const C*>(h_)[k];
        else { t.x = reinterpret_cast<const T*>(h_)[k]; t.y = (sizeof(T) == 4 && XC) ? t.x : (T)0; }   // f32: {t, t} splat for FFMA2
        sh[k] = t;
    }
    {
        long long g = p0 + threadIdx.x;
        if (big) { if (g >= N) g -= N; } else g %= N;
        const long long adv = big ? FIR_THREADS : FIR_THREADS % N;
        for (int w = threadIdx.x; w < W; w += FIR_THREADS) {
            C v;
            if (XC) v = reinterpret_cast<const C*>(x_)[vec * N + g];
            else { v.x = reinterpret_cast<const T*>(x_)[vec * N + g]; v.y = 0; }
            sx[fpad(w)] = v;
            g += adv; if (g >= N) g -= N;
        }
    }
    __syncthreads();
    // thread t produces outputs u0..u0+U-1 (u0 = t*U) from a circular register window:
    // at tap offset o = L-1-k the window holds x_window[u0 + o + u] in r[(o + u) % U]
    const int u0 = threadIdx.x * FIR_U;
    C acc[FIR_U];
    C r[FIR_U];
#pragma unroll
    for (int u = 0; u < FIR_U; u++) { acc[u] = mk<T>(0, 0); r[u] = sx[fpad(u0 + u)]; }
    for (int ob = 0; ob < L; ob += FIR_U) {
#pragma unroll
        for (int oo = 0; oo < FIR_U; oo++) {
            const int o = ob + oo;
            if (o < L) {
                const C t = sh[L - 1 - o];
#pragma unroll
                for (int u = 0; u < FIR_U; u++) {
                    const C xv = r[(oo + u) % FIR_U];
                    if constexpr (std::is_same<T, float>::value && XC && !HC) {
                        acc[u] = __ffma2_rn(xv, t, acc[u]);   // {re, im} * {t, t} + acc: one packed instruction per tap
                    } else if (HC) {
                        acc[u].x += xv.x * t.x - xv.y * t.y;
                        acc[u].y += xv.x * t.y + xv.y * t.x;
                    } else {
                        acc[u].x += xv.x * t.x;
                        if (XC) acc[u].y += xv.y * t.x;
                    }
                }
                r[oo] = sx[fpad(u0 + o + FIR_U)];
            }
        }
    }
    // stage the 8 consecutive outputs of every thread in (skewed) shared memory and copy out coalesced
    __syncthreads();
#pragma unroll
    for (int u = 0; u < FIR_U; u++) sx[fpad(u0 + u)] = acc[u];
    __syncthreads();
    for (int o = threadIdx.x; o < FIR_TILE; o += FIR_THREADS) {
        const long long i = i0 + o;
        if (i < N) {
            const C v = sx[fpad(o)];
            if (XC) reinterpret_cast<C*>(y_)[vec * N + i] = v;
            else reinterpret_cast<T*>(y_)[vec * N + i] = v.x;
        }
    }
}

template <typename T>
static int fir_convolve(const void* x, void* y, const void* h, size_t N, size_t batch, size_t L, int x_complex, int h_complex,
                        cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const size_t cl = L - L / 2;
    if (x == y) { set_last_error("fir_convolve: in-place operation is not supported"); return -3; }
    const long long tpv = (long long)((N + FIR_TILE - 1) / FIR_TILE);
    const size_t W = FIR_TILE + L - 1 + FIR_U + 1;
    const size_t smem = (L + W + W / 8 + 2) * sizeof(C);
    if (smem > 200 * 1024) { set_last_error("fir_convolve: too many taps (%zu)", L); return -2; }
    const long long grid = tpv * (long long)batch;
#define BDSP_FIR(XC_, HC_)                                                                                             \
    do {                                                                                                               \
        if (smem > 48 * 1024) BDSP_CUDA_OK(cudaFuncSetAttribute(fir_kernel<T, XC_, HC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        fir_kernel<T, XC_, HC_><<<(unsigned)grid, FIR_THREADS, smem, st>>>(x, y, h, (long long)N, (long long)batch, (int)L, (int)cl, tpv); \
    } while (0)
    if (x_complex && h_complex) BDSP_FIR(true, true);
    else if (x_complex) BDSP_FIR(true, false);
    else if (!h_complex) BDSP_FIR(false, false);
    else { set_last_error("fir_convolve: real vector with complex taps"); return -2; }
#undef BDSP_FIR
    BDSP_LAUNCHED();
    return 0;
}

// ------------------------------------------------------------------------------------------
// full-length frequency-domain path for impulse responses too long for a block transform:
//   y = IFFT(FFT(x) * FFT(roll(pad(h, N), -(cl-1)))) / N
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void pad_roll_h_kernel(const void* __restrict__ h_, typename CpxOf<T>::type* __restrict__ hp, long long L,
                                  long long N, long long shift, int h_is_real) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    // hp[i] = padded[(i + shift) mod N]
    long long src = (i + shift) % N;
    typename CpxOf<T>::type v = mk<T>(0, 0);
    if (src < L) {
        if (h_is_real) v.x = reinterpret_cast<const T*>(h_)[src];
        else v = reinterpret_cast<const typename CpxOf<T>::type*>(h_)[src];
    }
    hp[i] = v;
}

template <typename T>
static int fft_convolve_full(const void* x, void* y, const void* h, size_t N, size_t batch, size_t L, int is_real,
                             int h_is_real, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    const size_t cl = L - L / 2;
    // slots 4 / 5: fft_exec below uses slots 0..2 for its own passes (mixed-radix interleave, chirp-z ping-pong)
    BDSP_WS(Hf, C*, N * sizeof(C), 4);
    BDSP_WS(X, C*, N * batch * sizeof(C), 5);
    pad_roll_h_kernel<T><<<(unsigned)((N + 255) / 256), 256, 0, st>>>(h, Hf, (long long)L, (long long)N, (long long)(cl - 1), h_is_real);
    BDSP_LAUNCHED();
    FftOpts f;
    int rc = fft_exec<T>(Hf, Hf, N, 1, f, nullptr, 0, st);
    if (rc) return rc;
    FftOpts fx;
    fx.real_input = is_real;
    rc = fft_exec<T>(x, X, N, batch, fx, nullptr, 0, st);
    if (rc) return rc;
    // spectrum multiply (convolution.rs:427-429,444-446) and the 1/N of the inverse: fused into the first load of the
    // inverse transform (FftOpts::in_mul) wherever that transform carries a multiplier - every length except c32 powers of
    // two up to 16384, whose packed single-pass kernels keep the separate pass
    FftOpts inv;
    inv.inverse = 1;
    if (sizeof(T) == 4 && is_pow2(N) && N >= 64 && N <= 16384) {
        rc = ew_spectrum_mul_rows<T>(X, Hf, N, batch, 1.0 / (double)N, st);
        if (rc) return rc;
    } else {
        inv.in_mul.p = Hf; inv.in_mul.kind = 2;
        inv.scale = 1.0 / (double)N;
    }
    if (!is_real) return fft_exec<T>(X, y, N, batch, inv, nullptr, 0, st);
    rc = fft_exec<T>(X, X, N, batch, inv, nullptr, 0, st);
    if (rc) return rc;
    return ew_complex_to_real<T>(C2R_REAL, X, y, N * batch, st);
}

// Choice between the two fused block lengths where both apply (2 <= L <= 2046).  Measured on B200, 64 x 2^20 points
// (profiles/r2_ols_block_choice.txt): per POINT the 4096-point kernel is ~20 % faster (four independently phased CTAs per
// SM against two), so the 8192-point kernel only wins once its better block efficiency (M - L)/M outweighs that.
#define BDSP_OLS8192_MIN_TAPS 1450
#define BDSP_OLS8192_MIN_BLOCKS 592

// direct FIR up to this many taps
static size_t fir_max_taps(int h_is_real) { return h_is_real ? 96 : 24; }

template <typename T> bool conv_needs_plan(size_t L, int h_is_real) { return L > fir_max_taps(h_is_real) && L <= ols_max_taps<T>(); }

template <typename T>
int convolve(const void* x, void* y, size_t N, size_t batch, int x_is_real, const void* h, size_t L, int h_is_real,
             const OlsPlan* p, cudaStream_t st) {
    if (L <= fir_max_taps(h_is_real)) return fir_convolve<T>(x, y, h, N, batch, L, !x_is_real, !h_is_real, st);
    if (L > ols_max_taps<T>()) return fft_convolve_full<T>(x, y, h, N, batch, L, x_is_real, h_is_real, st);
    if (!p || p->is64 != (sizeof(T) == 8) || p->L != L) { set_last_error("convolve: %zu taps need their overlap-save plan", L); return -2; }
    if (x == y) { set_last_error("ols_convolve: in-place operation is not supported"); return -3; }
    const size_t M = p->M;
    if (sizeof(T) == 4 && !x_is_real) {
        // c32 responses beyond the fused blocks (4095 .. 8192 taps) on power-of-two vectors with packed multi-pass transforms:
        // forward transform + inverse transform with the spectrum multiply on its first load (2 x 2 passes over HBM) beats
        // the generic 16384-point overlap-save blocks (64 x 2^20, 8191 taps: 1.79 ms)
        if (L > 4094 && is_pow2(N) && N >= (1u << 15) && N <= (1u << 24))
            return fft_convolve_full<T>(x, y, h, N, batch, L, 0, h_is_real, st);
        // (olsi_blocks divides by the block step, which is only positive for applicable lengths)
        const bool want8 = olsi_applicable(8192, N, L) && L >= BDSP_OLS8192_MIN_TAPS &&
                           olsi_blocks(8192, N, L) * (long long)batch >= BDSP_OLS8192_MIN_BLOCKS;
        if (p->htex2 && want8)
            return ols8192_convolve(x, y, N, batch, L, p->htex2, st);
        if (p->htex && M == 4096 && olsi_applicable(4096, N, L))
            return ols4096_convolve(x, y, N, batch, L, p->htex, st);
        if (p->htex && M == 8192 && olsi_applicable(8192, N, L))
            return ols8192_convolve(x, y, N, batch, L, p->htex, st);
    }
    if (sizeof(T) == 8 && !x_is_real && ols64_applicable(N, L, M)) return ols64_convolve(x, y, N, batch, L, p->Hs, st);   // fused 4096-point c64 blocks
    return ols_generic_convolve<T>(p, x, y, N, batch, x_is_real, st);
}

#define BDSP_INST(T)                                                                                                    \
    template OlsPlan* ols_plan_create<T>(const void*, size_t, int, bool, cudaStream_t);                                 \
    template bool conv_needs_plan<T>(size_t, int);                                                                      \
    template int convolve<T>(const void*, void*, size_t, size_t, int, const void*, size_t, int, const OlsPlan*, cudaStream_t);
BDSP_INST(float)
BDSP_INST(double)
#undef BDSP_INST

}  // namespace bdsp
