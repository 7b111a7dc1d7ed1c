// Fused 4096-point overlap-save block for the fast convolution hot path, interleaved-complex FP32x2 version:
// forward FFT, spectrum multiply and inverse FFT of one block in ONE kernel with the block resident in shared memory
// (the reference's overlap_discard, convolution.rs:304-461: 2 rustfft calls + a scalar multiply loop per block).
//
// Structure (M = 4096 = 16^3, 128 threads, 32 points per thread and stage; block position p = 256 a + 16 b + c):
//   F1  radix-16 DIF over a, columns (2t, 2t+1) of the input in smem (aligned rows: bulk copies)
//       or straight from global memory (other rows)                                                 -> smem  | CTA barrier
//   F2  radix-16 DIF over b inside row a = t >> 3                                                    -> smem  | warp barrier
//   F3  radix-16 DIF over the 16 contiguous c | * H (position order) | radix-16 DIT  (registers)    -> smem  | warp barrier
//   I2  radix-16 DIT over b                                                                          -> smem  | CTA barrier
//   I1  radix-16 DIT over a, valid outputs to global memory: aligned rows through smem in natural order and one
//       bulk copy, other rows with direct stores
// Aligned rows move a block's input and output between global and shared memory by bulk asynchronous copies
// (cp.async.bulk + mbarrier): no load or store instruction per 16 bytes on the L1 data pipe, the kernel's saturated unit.
// The forward transform leaves the spectrum digit-reversed, the plan stores H in that order, the inverse consumes it:
// no reordering pass.  All arithmetic is interleaved-complex packed FP32x2 (cxmath.cuh): two adjacent points travel as
// one 128-bit word through every global and shared access, so a stage costs 16 + 16 shared-memory instructions per
// thread (round 1's planar kernel: 32 + 32), no MOV re-pairing, no constant pairs.
// Shared layout: point p lives in float2 slot 256 a + 16 b + (c ^ 2 (b & 7)): the 16-byte chunks of a 128-byte row
// are XOR-swizzled by the row number, which keeps the 128-bit accesses of every quarter-warp in eight different bank
// windows in all three access patterns, without padding (32 KB per CTA).
#include "conv.cuh"
#include "olsi.cuh"

namespace bdsp {

using namespace cx;

#define OI_M 4096
#define OI_T 128
#define OI_MIN_CTAS 5

// twiddle table olsi_twiddles(4096): [0,256) W4096^col; [256 + 16 k + c] W256^{k c}, k, c in [0,16)
#define OI_TW2 256

// ALIGNED: rows start on 16-byte boundaries (N even, 16-byte aligned base pointers); together with the even block
// offsets chosen by the plan every thread then moves its two adjacent points with one 128-bit access, and every piece
// of a block's input and output is a 16-byte aligned run of a multiple of 16 bytes, as bulk copies require.  `shift` =
// cl - 1 + d is the (even) distance between a block position's input index and its output index.
template <bool ALIGNED>
__global__ void __launch_bounds__(OI_T, OI_MIN_CTAS)
ols4096i_kernel(const float2* __restrict__ x, float2* __restrict__ y, int N, int m_first, int step, int shift,
                int blocks_per_vec, const float2* __restrict__ tw, cudaTextureObject_t htex) {
    __shared__ __align__(128) float2 sm[OI_M];
    __shared__ __align__(8) unsigned long long bar;
    const int t = threadIdx.x;
    const int vec = blockIdx.x / blocks_per_vec;
    const int blk = blockIdx.x - vec * blocks_per_vec;
    const int i0 = blk * step;
    const float2* xr = x + (size_t)vec * (size_t)N;
    float2* yr = y + (size_t)vec * (size_t)N;
    const int hi = t >> 3, lo = t & 7;         // quarter-warp index / lane inside it
    // block position p holds x[(p0 + p) mod N], p0 = i0 + shift - m_first  (-4096 < p0 < N - 1, even)
    const int p0 = i0 + shift - m_first;
    pdl_trigger();                             // the next kernel of the stream may start launching
    pdl_wait();                                // ... and this one touches global memory only after its predecessor is complete
    if (ALIGNED) {
        // the block's 32 KB of input land in sm in natural order through one or two bulk copies (two when it wraps
        // around the end of the vector): no load instruction per 16 bytes on the L1 data pipe, its saturated unit
        if (t == 0) {
            const unsigned b = smem_u32(&bar), s = smem_u32(sm);
            mbar_init(b, 1);
            mbar_arrive_expect_tx(b, OI_M * 8);
            const int first = p0 < 0 ? p0 + N : p0;
            const int n1 = min(OI_M, N - first);
            bulk_g2s(s, xr + first, 8 * n1, b);
            if (n1 < OI_M) bulk_g2s(s + 8 * n1, xr, 8 * (OI_M - n1), b);
        }
        __syncthreads();                       // the barrier is initialised before anyone waits on it
        mbar_wait(smem_u32(&bar), 0);
    }

    c2 v[16], u[16];                           // the thread's two columns
    // ------------------------------------------------------------------ F1: over a, columns (2t, 2t+1) = (b = hi, c = 2 lo, 2 lo + 1)
    {
        const int col = 2 * t;
        if (ALIGNED) {
#pragma unroll
            for (int a = 0; a < 16; a++) {
                const float4 ab = *reinterpret_cast<const float4*>(sm + 256 * a + col);
                v[a] = make_float2(ab.x, ab.y);
                u[a] = make_float2(ab.z, ab.w);
            }
        } else if (p0 >= 0 && p0 + OI_M <= N) {   // block-uniform: no wrap-around inside this block
            const float2* px = xr + p0 + col;
#pragma unroll
            for (int a = 0; a < 16; a++) {
                v[a] = __ldg(px + 256 * a);
                u[a] = __ldg(px + 256 * a + 1);
            }
        } else {                             // first / last block of a vector: circular indexing
            int idx = p0 + col;
            if (idx < 0) idx += N;
            if (idx >= N) idx -= N;
#pragma unroll
            for (int a = 0; a < 16; a++) {
                int i1 = idx + 1; if (i1 >= N) i1 -= N;
                v[a] = __ldg(&xr[idx]);
                u[a] = __ldg(&xr[i1]);
                idx += 256; if (idx >= N) idx -= N;
            }
        }
        r16<false>(v);
        r16<false>(u);
        const float4 w = __ldg(reinterpret_cast<const float4*>(tw + col));
        apply_twiddles<true>(v, make_float2(w.x, w.y));
        apply_twiddles<true>(u, make_float2(w.z, w.w));
        if (ALIGNED) __syncthreads();          // every thread has read the natural-order input before it is overwritten
        float2* dst = sm + 16 * hi + ((2 * lo) ^ (2 * (hi & 7)));
#pragma unroll
        for (int s = 0; s < 16; s++)
            *reinterpret_cast<float4*>(dst + 256 * r16_k(s)) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
    }
    __syncthreads();
    // ------------------------------------------------------------------ F2: over b inside row a = hi, columns c = 2 lo, 2 lo + 1
    float2* row = sm + 256 * hi;
    const float4* tw2 = reinterpret_cast<const float4*>(tw + OI_TW2) + lo;   // tw2[8 k]: W256^{k c}, c = 2 lo, 2 lo + 1
    {
#pragma unroll
        for (int b = 0; b < 16; b++) {
            const float4 f = *reinterpret_cast<const float4*>(row + 16 * b + ((2 * lo) ^ (2 * (b & 7))));
            v[b] = make_float2(f.x, f.y);
            u[b] = make_float2(f.z, f.w);
        }
        r16<false>(v);
        r16<false>(u);
        oi_tw2<true, false, 8>(v, u, tw2);
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int k1 = r16_k(s);
            *reinterpret_cast<float4*>(row + 16 * k1 + ((2 * lo) ^ (2 * (k1 & 7)))) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
        }
    }
    __syncwarp();
    // ------------------------------------------------------------------ F3 | *H | I3 on the 16 contiguous points of rows (hi, b = lo + 8 half)
#pragma unroll 1
    for (int half = 0; half < 2; half++) {
        float2* grp = row + 16 * (lo + 8 * half);
        c2 P[16];
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const float4 f = *reinterpret_cast<const float4*>(grp + 2 * (q ^ lo));
            P[2 * q] = make_float2(f.x, f.y);
            P[2 * q + 1] = make_float2(f.z, f.w);
        }
        fft_dif<4, false>(P);
#pragma unroll
        for (int q = 0; q < 8; q++) {
            // plan layout: [half][q][thread] float4 = H of positions c = 2q, 2q + 1 -> a warp reads 512 contiguous bytes
            const float4 h = tex1Dfetch<float4>(htex, (half * 8 + q) * OI_T + t);
            P[2 * q] = mul(P[2 * q], make_float2(h.x, h.y));
            P[2 * q + 1] = mul(P[2 * q + 1], make_float2(h.z, h.w));
        }
        fft_dit<4, true>(P);
#pragma unroll
        for (int q = 0; q < 8; q++)
            *reinterpret_cast<float4*>(grp + 2 * (q ^ lo)) = make_float4(P[2 * q].x, P[2 * q].y, P[2 * q + 1].x, P[2 * q + 1].y);
    }
    __syncwarp();
    // ------------------------------------------------------------------ I2: over b (DIT: twiddle first)
    {
#pragma unroll
        for (int k1 = 0; k1 < 16; k1++) {
            const float4 f = *reinterpret_cast<const float4*>(row + 16 * k1 + ((2 * lo) ^ (2 * (k1 & 7))));
            v[k1] = make_float2(f.x, f.y);
            u[k1] = make_float2(f.z, f.w);
        }
        oi_tw2<false, true, 8>(v, u, tw2);
        r16<true>(v);
        r16<true>(u);
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int b = r16_k(s);
            *reinterpret_cast<float4*>(row + 16 * b + ((2 * lo) ^ (2 * (b & 7)))) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
        }
    }
    __syncthreads();
    // ------------------------------------------------------------------ I1: over a, valid outputs to global
    {
        const int col = 2 * t;
        const float2* src = sm + 16 * hi + ((2 * lo) ^ (2 * (hi & 7)));
#pragma unroll
        for (int k0 = 0; k0 < 16; k0++) {
            const float4 f = *reinterpret_cast<const float4*>(src + 256 * k0);
            v[k0] = make_float2(f.x, f.y);
            u[k0] = make_float2(f.z, f.w);
        }
        const float4 w = __ldg(reinterpret_cast<const float4*>(tw + col));
        apply_twiddles<false>(v, make_float2(w.x, -w.y));
        apply_twiddles<false>(u, make_float2(w.z, -w.w));
        r16<true>(v);
        r16<true>(u);
        // output i = i0 + m, m = col + 256 a - m_first in [0, step) and i < N
        const int mlo = col - m_first;                     // m for a = 0
        int mhi = step;                                    // exclusive bound on m
        if (i0 + step > N) mhi = N - i0;                   // last block of the vector
        float2* py = yr + i0 + mlo;
        // ALIGNED: the valid outputs go to sm in natural order (position m_first + m) and leave through one bulk copy
        // of the mhi outputs (a 16-byte aligned, even count) instead of a 128-bit store each
        if (ALIGNED) __syncthreads();                      // every thread has read the swizzled layout
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int a = r16_k(s);
            const int m = mlo + 256 * a;
            if (ALIGNED) {
                if (m >= 0 && m < mhi) *reinterpret_cast<float4*>(sm + col + 256 * a) = make_float4(v[s].x, v[s].y, u[s].x, u[s].y);
            } else {
                if (m >= 0 && m < mhi) py[256 * a] = v[s];
                if (m + 1 >= 0 && m + 1 < mhi) py[256 * a + 1] = u[s];
            }
        }
        if (ALIGNED) {
            fence_proxy_async_smem();                      // the stores above precede the bulk copy's reads
            __syncthreads();
            if (t == 0) bulk_s2g_wait_read(yr + i0, smem_u32(sm + m_first), 8 * mhi);   // sm stays valid until read
        }
    }
}

// frequency index held at block position p after F1, F2, F3
__host__ __device__ __forceinline__ int oi_freq_of_pos(int p) {
    const int k0 = p >> 8, k1 = (p >> 4) & 15, c = p & 15;
    return k0 + 16 * k1 + 256 * bitrev4(c);
}

// Hpos (kernel layout, interleaved) <- Hs (interleaved, natural order, already scaled by 1/M), delayed by d samples:
// H_d[k] = H[k] * exp(-2 pi i k d / M).  Position p = 256 a + 16 b + c is owned by thread t = 8 a + (b & 7) in iteration
// half = b >> 3 and stored at float2 index 2 * (((half * 8 + c / 2) * 128) + t) + (c & 1).
__global__ void ols4096i_permute_h_kernel(const float2* __restrict__ Hs, float2* __restrict__ Hpos, int d) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= OI_M) return;
    const int k = oi_freq_of_pos(p);
    float2 h = Hs[k];
    if (d) h = cmul(h, unit_root<float>((unsigned long long)k * (unsigned long long)d, OI_M, -1));
    const int a = p >> 8, b = (p >> 4) & 15, c = p & 15;
    const int t = 8 * a + (b & 7), half = b >> 3;
    Hpos[2 * ((half * 8 + (c >> 1)) * OI_T + t) + (c & 1)] = h;
}

// Hpos: 4096 float2 <- Hs from the plan (FFT_4096(pad(h)) / 4096, natural order)
int ols4096_prepare(const void* Hs, void* Hpos, size_t L, cudaStream_t st) {
    int d, shift, m_first, step;
    olsi_geometry(OI_M, L, &d, &shift, &m_first, &step);
    ols4096i_permute_h_kernel<<<OI_M / 256, 256, 0, st>>>(reinterpret_cast<const float2*>(Hs), reinterpret_cast<float2*>(Hpos), d);
    BDSP_LAUNCHED();
    return 0;
}

int ols4096_convolve(const void* x, void* y, size_t N, size_t batch, size_t L, cudaTextureObject_t htex, cudaStream_t st) {
    if (x == y) { set_last_error("ols4096_convolve: in-place operation is not supported"); return -3; }
    int d, shift, m_first, step;
    olsi_geometry(OI_M, L, &d, &shift, &m_first, &step);
    const long long bpv = ((long long)N + step - 1) / step;
    const long long grid = bpv * (long long)batch;
    if (grid > 0x7fffffffll) { set_last_error("ols4096_convolve: grid too large"); return -2; }
    const float2* tw = olsi_twiddles(OI_M);
    if (!tw) return -1;
    const bool aligned = (N % 2 == 0) && ((reinterpret_cast<uintptr_t>(y) & 15) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    if (aligned)
        BDSP_CUDA_OK(launch_pdl(ols4096i_kernel<true>, dim3((unsigned)grid), dim3(OI_T), 0, st, reinterpret_cast<const float2*>(x),
                                reinterpret_cast<float2*>(y), (int)N, m_first, step, shift, (int)bpv, tw, htex));
    else
        BDSP_CUDA_OK(launch_pdl(ols4096i_kernel<false>, dim3((unsigned)grid), dim3(OI_T), 0, st, reinterpret_cast<const float2*>(x),
                                reinterpret_cast<float2*>(y), (int)N, m_first, step, shift, (int)bpv, tw, htex));
    BDSP_LAUNCHED();
    return 0;
}

}  // namespace bdsp
