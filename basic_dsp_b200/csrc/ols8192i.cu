// Fused 8192-point overlap-save block (interleaved-complex FP32x2 arithmetic, cxmath.cuh): forward FFT, spectrum
// multiply and inverse FFT of one block in ONE kernel pass with the block resident in shared memory (the reference's
// overlap_discard, convolution.rs:304-461, whose blocks are 2 rustfft calls + a scalar multiply loop).
//
// Why a second block length next to ols4096i: the reference derives fft_len from the tap count (convolution.rs:323-331).
// The fused block is bound by the L1 / shared-memory data pipe (profiles/r2_ols_ablation.txt), whose load is proportional
// to the points pushed through the four exchanges, i.e. per OUTPUT sample to M / (M - L + 1): 1.33 for a 4096-point block
// at 1023 taps, 1.14 for an 8192-point block - and a 4096-point block cannot take more than 2046 taps at all.
//
// Structure (M = 8192 = 16 * 16 * 32, 256 threads, 32 points per thread and stage; block position p = 512 a + 32 b + c):
//   F1  radix-16 DIF over a, columns (2t, 2t+1) straight from global memory (128-bit loads)           -> smem | CTA barrier
//   F2  radix-16 DIF over b inside row a = t >> 4                                                       -> smem | warp barrier
//   F3  radix-32 DIF over the 32 contiguous c of (a, b = t & 15) | * H | radix-32 DIT  (registers)     -> smem | warp barrier
//   I2  radix-16 DIT over b                                                                             -> smem | CTA barrier
//   I1  radix-16 DIT over a, valid outputs straight to global memory (128-bit stores)
// Row a (512 points) is owned by half-warp a in F2, F3 and I2: two CTA-wide barriers per block.
// Shared layout: point p lives in float2 slot 512 a + 32 b + (c ^ 2 (b & 7)): the low three bits of the 16-byte chunk
// index are XOR-swizzled by the row number, which keeps the 128-bit accesses of every quarter-warp in eight different
// bank windows in all three access patterns, without padding (64 KB per CTA, two CTAs per SM).
#include <mutex>

#include "conv.cuh"
#include "olsi.cuh"

namespace bdsp {

using namespace cx;

#define O8_M 8192
#define O8_T 256
#define O8_MIN_CTAS 2
#define O8_SMEM_BYTES (O8_M * sizeof(float2))

// twiddle table olsi_twiddles(8192): [0,512) W8192^col; [512 + 32 k + c] W512^{k c}, k in [0,16), c in [0,32)
#define O8_TW2 512

template <bool ALIGNED>
__global__ void __launch_bounds__(O8_T, O8_MIN_CTAS)
ols8192i_kernel(const float2* __restrict__ x, float2* __restrict__ y, int N, int m_first, int step, int shift,
                int blocks_per_vec, const float2* __restrict__ tw, cudaTextureObject_t htex) {
    extern __shared__ __align__(16) float2 o8_sm[];
    float2* sm = o8_sm;
    const int t = threadIdx.x;
    const int vec = blockIdx.x / blocks_per_vec;
    const int blk = blockIdx.x - vec * blocks_per_vec;
    const int i0 = blk * step;
    const float2* xr = x + (size_t)vec * (size_t)N;
    float2* yr = y + (size_t)vec * (size_t)N;
    const int hi = t >> 4, lo = t & 15;        // half-warp index / lane inside it

    c2 v[16], u[16];                           // the thread's two columns
    // ------------------------------------------------------------------ F1: over a, columns (2t, 2t+1) = (b = hi, c = 2 lo, 2 lo + 1)
    {
        const int col = 2 * t;
        // block position p holds x[(p0 + p) mod N], p0 = i0 + shift - m_first  (p0 > -8192, even)
        const int p0 = i0 + shift - m_first;
        if (p0 >= 0 && p0 + O8_M <= N) {   // block-uniform: no wrap-around inside this block
            const float2* px = xr + p0 + col;
#pragma unroll
            for (int a = 0; a < 16; a++) {
                if (ALIGNED) {
                    const float4 ab = ld_x4(px + 512 * a);
                    v[a] = make_float2(ab.x, ab.y);
                    u[a] = make_float2(ab.z, ab.w);
                } else {
                    v[a] = __ldg(px + 512 * a);
                    u[a] = __ldg(px + 512 * a + 1);
                }
            }
        } else {                             // first / last block of a vector: circular indexing
            int idx = (p0 + col) % N;
            if (idx < 0) idx += N;
            const int adv = 512 % N;
#pragma unroll
            for (int a = 0; a < 16; a++) {
                int i1 = idx + 1; if (i1 >= N) i1 -= N;
                v[a] = __ldg(&xr[idx]);
                u[a] = __ldg(&xr[i1]);
                idx += adv; if (idx >= N) idx -= N;
            }
        }
        r16<false>(v);
        r16<false>(u);
        const float4 w = __ldg(reinterpret_cast<const float4*>(tw + col));
        apply_twiddles<true>(v, make_float2(w.x, w.y));
        apply_twiddles<true>(u, make_float2(w.z, w.w));
        float2* dst = sm + 32 * hi + ((2 * lo) ^ (2 * (hi & 7)));
#pragma unroll
        for (int s = 0; s < 16; s++)
            *reinterpret_cast<float4*>(dst + 512 * r16_k(s)) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
    }
    __syncthreads();
    // ------------------------------------------------------------------ F2: over b inside row a = hi, columns c = 2 lo, 2 lo + 1
    float2* row = sm + 512 * hi;
    const float4* tw2 = reinterpret_cast<const float4*>(tw + O8_TW2) + lo;   // tw2[16 k]: W512^{k c}, c = 2 lo, 2 lo + 1
    {
#pragma unroll
        for (int b = 0; b < 16; b++) {
            const float4 f = *reinterpret_cast<const float4*>(row + 32 * b + ((2 * lo) ^ (2 * (b & 7))));
            v[b] = make_float2(f.x, f.y);
            u[b] = make_float2(f.z, f.w);
        }
        r16<false>(v);
        r16<false>(u);
        oi_tw2<true, false, 16>(v, u, tw2);
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int k1 = r16_k(s);
            *reinterpret_cast<float4*>(row + 32 * k1 + ((2 * lo) ^ (2 * (k1 & 7)))) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
        }
    }
    __syncwarp();
    // ------------------------------------------------------------------ F3 | *H | I3 on the 32 contiguous points of (a = hi, b = lo)
    {
        float2* grp = row + 32 * lo;
        const int sw = lo & 7;
        c2 P[32];
#pragma unroll
        for (int q = 0; q < 16; q++) {
            const float4 f = *reinterpret_cast<const float4*>(grp + 2 * (q ^ sw));
            P[2 * q] = make_float2(f.x, f.y);
            P[2 * q + 1] = make_float2(f.z, f.w);
        }
        fft_dif<5, false>(P);                // slot j holds k2 = bitrev5(j)
#pragma unroll
        for (int q = 0; q < 16; q++) {
            // plan layout: [q][thread] float4 = H of positions c = 2q, 2q + 1 -> a warp reads 512 contiguous bytes
            const float4 h = tex1Dfetch<float4>(htex, q * O8_T + t);
            P[2 * q] = mul(P[2 * q], make_float2(h.x, h.y));
            P[2 * q + 1] = mul(P[2 * q + 1], make_float2(h.z, h.w));
        }
        fft_dit<5, true>(P);
#pragma unroll
        for (int q = 0; q < 16; q++)
            *reinterpret_cast<float4*>(grp + 2 * (q ^ sw)) = make_float4(P[2 * q].x, P[2 * q].y, P[2 * q + 1].x, P[2 * q + 1].y);
    }
    __syncwarp();
    // ------------------------------------------------------------------ I2: over b (DIT: twiddle first)
    {
#pragma unroll
        for (int k1 = 0; k1 < 16; k1++) {
            const float4 f = *reinterpret_cast<const float4*>(row + 32 * k1 + ((2 * lo) ^ (2 * (k1 & 7))));
            v[k1] = make_float2(f.x, f.y);
            u[k1] = make_float2(f.z, f.w);
        }
        oi_tw2<false, true, 16>(v, u, tw2);
        r16<true>(v);
        r16<true>(u);
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int b = r16_k(s);
            *reinterpret_cast<float4*>(row + 32 * b + ((2 * lo) ^ (2 * (b & 7)))) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
        }
    }
    __syncthreads();
    // ------------------------------------------------------------------ I1: over a, valid outputs to global
    {
        const int col = 2 * t;
        const float2* src = sm + 32 * hi + ((2 * lo) ^ (2 * (hi & 7)));
#pragma unroll
        for (int k0 = 0; k0 < 16; k0++) {
            const float4 f = *reinterpret_cast<const float4*>(src + 512 * k0);
            v[k0] = make_float2(f.x, f.y);
            u[k0] = make_float2(f.z, f.w);
        }
        const float4 w = __ldg(reinterpret_cast<const float4*>(tw + col));
        apply_twiddles<false>(v, make_float2(w.x, -w.y));
        apply_twiddles<false>(u, make_float2(w.z, -w.w));
        r16<true>(v);
        r16<true>(u);
        // output i = i0 + m, m = col + 512 a - m_first in [0, step) and i < N
        const int mlo = col - m_first;                     // m for a = 0
        int mhi = step;                                    // exclusive bound on m
        if (i0 + step > N) mhi = N - i0;                   // last block of the vector
        float2* py = yr + i0 + mlo;
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int a = r16_k(s);
            const int m = mlo + 512 * a;
            if (ALIGNED) {
                if (m >= 0 && m < mhi) *reinterpret_cast<float4*>(py + 512 * a) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
            } else {
                if (m >= 0 && m < mhi) py[512 * a] = v[s];
                if (m + 1 >= 0 && m + 1 < mhi) py[512 * a + 1] = u[s];
            }
        }
    }
}

// frequency index held at block position p after F1, F2, F3
__host__ __device__ __forceinline__ int o8_freq_of_pos(int p) {
    const int k0 = p >> 9, k1 = (p >> 5) & 15, c = p & 31;
    return k0 + 16 * k1 + 256 * bitrev5(c);
}

// Hpos (kernel layout, interleaved) <- Hs (interleaved, natural order, already scaled by 1/M), delayed by d samples:
// H_d[k] = H[k] * exp(-2 pi i k d / M).  Position p = 512 a + 32 b + c is owned by thread t = 16 a + b and stored at
// float2 index 2 * ((c / 2) * 256 + t) + (c & 1).
__global__ void ols8192i_permute_h_kernel(const float2* __restrict__ Hs, float2* __restrict__ Hpos, int d) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= O8_M) return;
    const int k = o8_freq_of_pos(p);
    float2 h = Hs[k];
    if (d) h = cmul(h, unit_root<float>((unsigned long long)k * (unsigned long long)d, O8_M, -1));
    const int t = p >> 5, c = p & 31;
    Hpos[2 * ((c >> 1) * O8_T + t) + (c & 1)] = h;
}

// Hpos: 8192 float2 <- Hs = FFT_8192(pad(h)) / 8192 (natural order)
int ols8192_prepare(const void* Hs, void* Hpos, size_t L, cudaStream_t st) {
    int d, shift, m_first, step;
    olsi_geometry(O8_M, L, &d, &shift, &m_first, &step);
    ols8192i_permute_h_kernel<<<O8_M / 256, 256, 0, st>>>(reinterpret_cast<const float2*>(Hs), reinterpret_cast<float2*>(Hpos), d);
    BDSP_LAUNCHED();
    return 0;
}

int ols8192_convolve(const void* x, void* y, size_t N, size_t batch, size_t L, cudaTextureObject_t htex, cudaStream_t st) {
    if (x == y) { set_last_error("ols8192_convolve: in-place operation is not supported"); return -3; }
    int d, shift, m_first, step;
    olsi_geometry(O8_M, L, &d, &shift, &m_first, &step);
    const long long bpv = ((long long)N + step - 1) / step;
    const long long grid = bpv * (long long)batch;
    if (grid > 0x7fffffffll) { set_last_error("ols8192_convolve: grid too large"); return -2; }
    const float2* tw = olsi_twiddles(O8_M);
    if (!tw) return -1;
    static std::mutex mu;   // launches from threads on different devices: PerDeviceOnce is not thread-safe on its own
    static PerDeviceOnce configured;
    std::lock_guard<std::mutex> lk(mu);
    if (configured.need()) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(ols8192i_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)O8_SMEM_BYTES));
        BDSP_CUDA_OK(cudaFuncSetAttribute(ols8192i_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)O8_SMEM_BYTES));
        configured.mark();
    }
    const bool aligned = (N % 2 == 0) && ((reinterpret_cast<uintptr_t>(y) & 15) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    if (aligned)
        ols8192i_kernel<true><<<(unsigned)grid, O8_T, O8_SMEM_BYTES, st>>>(reinterpret_cast<const float2*>(x), reinterpret_cast<float2*>(y),
                                                                          (int)N, m_first, step, shift, (int)bpv, tw, htex);
    else
        ols8192i_kernel<false><<<(unsigned)grid, O8_T, O8_SMEM_BYTES, st>>>(reinterpret_cast<const float2*>(x), reinterpret_cast<float2*>(y),
                                                                           (int)N, m_first, step, shift, (int)bpv, tw, htex);
    BDSP_LAUNCHED();
    return 0;
}

}  // namespace bdsp
