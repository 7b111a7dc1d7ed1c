// Fused overlap-save block for c64 signals: 4096-point blocks, FFT -> * H -> IFFT in one CTA, data in registers between
// global memory and the first / last radix-8 stage.
//
// Replaces the reference's overlap_discard loop for f64 (convolution.rs:304-461: rustfft forward, spectrum multiply
// :427-429, inverse, copy of the valid part) and, inside this library, the generic ols_conv_kernel<double>, whose
// run-time-indexed stages and separate load / multiply / store sweeps cost 14 shared-memory round trips per block.
//
// 512 threads x 8 points.  Both transforms are Stockham radix-8 x 4 (8^4 = 4096) in natural order:
//   forward: thread j loads x[j + 512 r] (coalesced) = inputs of its first butterfly; after the fourth stage it holds
//            X[j + 512 r], multiplies by Hs[j + 512 r] (H / 4096, natural order: OlsPlan::Hs) and these ARE the inputs
//            of the inverse transform's first butterfly - no exchange between the two transforms;
//   inverse: after its fourth stage the thread holds y[j + 512 r] and stores the valid ones (m >= L - 1) coalesced.
// Six shared-memory exchanges per block, 16 B words, one word of padding per 8 (stride-8 first-stage writes).
#include "conv.cuh"
#include "fft.cuh"
#include "fft_core.cuh"

namespace bdsp {

namespace {

constexpr int O64_M = 4096;
constexpr int O64_T = 512;
constexpr int O64_WORDS = O64_M + O64_M / 8;
constexpr int O64_TWL = 16384;   // master table W_16384^i (fft.cu)

__device__ __forceinline__ double2& o64_at(double2* s, int idx) { return s[idx + (idx >> 3)]; }

// v[r] *= w1^r, r = 1..7 (product tree of depth 3)
__device__ __forceinline__ void o64_twiddle(double2* v, double2 w1) {
    const double2 w2 = cmul(w1, w1), w3 = cmul(w2, w1), w4 = cmul(w2, w2);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], w3);
    v[4] = cmul(v[4], w4);
    v[5] = cmul(v[5], cmul(w4, w1));
    v[6] = cmul(v[6], cmul(w3, w3));
    v[7] = cmul(v[7], cmul(w4, w3));
}

// 4096-point transform of the 8 x 512 values held as v[r] = a[j + 512 r]; result v[r] = A[j + 512 r]
template <bool INV>
__device__ __forceinline__ void o64_fft(double2* v, double2* s, int j, const double2* __restrict__ tw) {
    RegFFT<double, 8, INV>::run(v);                                   // Ns = 1
#pragma unroll
    for (int r = 0; r < 8; r++) o64_at(s, 8 * j + r) = v[r];
    __syncthreads();
#pragma unroll
    for (int st = 1; st < 4; st++) {                                   // Ns = 8, 64, 512
        const int Ns = 1 << (3 * st);
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = o64_at(s, j + 512 * r);
        const int k = j & (Ns - 1);
        double2 w1 = __ldg(&tw[k * (O64_TWL / (8 * Ns))]);
        if (INV) w1.y = -w1.y;
        o64_twiddle(v, w1);
        RegFFT<double, 8, INV>::run(v);
        if (st < 3) {
            __syncthreads();
#pragma unroll
            for (int r = 0; r < 8; r++) o64_at(s, (j - k) * 8 + k + Ns * r) = v[r];
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(O64_T, 2)
ols64_kernel(const double2* __restrict__ x, double2* __restrict__ y, long long N, int L, int step, unsigned blocks_per_vec,
             const double2* __restrict__ Hs, const double2* __restrict__ tw) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* s = reinterpret_cast<double2*>(smem_raw);
    const int j = threadIdx.x;
    const unsigned vec = blockIdx.x / blocks_per_vec;
    const unsigned blk = blockIdx.x - vec * blocks_per_vec;
    const int i0 = (int)blk * step;                      // first output of this block (N < 2^31)
    const int cl = L - L / 2;
    const int n = (int)N;
    int g = i0 - (L - cl) + j;                            // first input: -N < g < N, block length <= N
    if (g < 0) g += n;
    else if (g >= n) g -= n;                              // (last block of a vector)
    const double2* xv = x + (long long)vec * N;
    double2 v[8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        v[r] = xv[g];
        g += 512;
        if (g >= n) g -= n;
    }
    o64_fft<false>(v, s, j, tw);
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = cmul(v[r], __ldg(&Hs[j + 512 * r]));
    __syncthreads();                                      // the forward transform's last reads precede the inverse's first writes
    o64_fft<true>(v, s, j, tw);
    double2* yv = y + (long long)vec * N;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int m = j + 512 * r;
        const int i = i0 + m - (L - 1);
        if (m >= L - 1 && i < n) yv[i] = v[r];
    }
}

}  // namespace

bool ols64_applicable(size_t N, size_t L, size_t M) { return M == (size_t)O64_M && L >= 1 && L <= (size_t)O64_M / 2 && N >= (size_t)O64_M && N < (1ull << 30); }

int ols64_convolve(const void* x, void* y, size_t N, size_t batch, size_t L, const void* Hs, cudaStream_t st) {
    const int step = O64_M - (int)L + 1;
    const unsigned long long bpv = (N + step - 1) / step;
    if (bpv * batch > 0x7fffffffull) { set_last_error("ols64: grid too large"); return -2; }
    const double2* tw = twiddle_table<double>();
    if (!tw) return -1001;
    const size_t smem = (size_t)O64_WORDS * sizeof(double2);
    static PerDeviceOnce configured;
    if (configured.need()) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(ols64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        BDSP_CUDA_OK(cudaFuncSetAttribute(ols64_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured.mark();
    }
    ols64_kernel<<<(unsigned)(bpv * batch), O64_T, smem, st>>>(reinterpret_cast<const double2*>(x), reinterpret_cast<double2*>(y), (long long)N,
                                                               (int)L, step, (unsigned)bpv, reinterpret_cast<const double2*>(Hs), tw);
    BDSP_LAUNCHED();
    return 0;
}

}  // namespace bdsp
