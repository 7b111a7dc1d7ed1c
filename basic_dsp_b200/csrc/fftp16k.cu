// 16384-point c32 rows (BASELINE config C3: 4096 x 2^14 fft + magnitude): persistent CTAs with a rolling pipeline.
//
// A 16384-point row needs 139 KB of shared memory, i.e. ONE 512-thread CTA per SM, so nothing hides a CTA's own load /
// compute / store phases: round 1's kernel ran them back to back (profiles/r1_fftp16384_ncu.txt: DRAM 34 %, FMA 39 %,
// LSU 48 % - nothing saturated, 44 % of the HBM roofline).  This kernel keeps the same arithmetic
//   F0  radix-4 DIF over stride 4096 (global -> shared), twiddle W_16384^{k c}
//   F1  radix-16 over stride 256, F2 radix-16 over stride 16 (in place in shared memory)
//   F3  radix-16 over 16 contiguous points in registers -> global, natural order (+ fft_shift, magnitude)
// but overlaps the two memory-bound phases of consecutive rows: the 16 contiguous points a thread quad reads in F3
// (same (k0, k1) group of the four 4096-point sub-blocks) are exactly the shared-memory words that F0 of the NEXT row
// writes for 8 column pairs, so the quad, after its F3 loads, runs F0 of the next row for those columns in place
// (quad-local dependency: __syncwarp only).  The next row's global loads are issued before the F3 arithmetic and
// consumed after it, the current row's result stores and the next row's loads are in flight together, and there is no
// separate load phase any more.  Three CTA-wide barriers per row.
// Replaces rustfft + swap pass + magnitude pass for these rows (time_to_freq.rs:136-165, complex_to_real.rs:374-379).
#include "fftp.cuh"

namespace bdsp {
using namespace ols16;

#define F16_NT 512
#define F16_B FP_B_OF(4)

// the two adjacent column pairs (2*lsb, 2*lsb + 1) of group (k0, k1): F0 inputs of one row, 8 x 128-bit loads
struct F16Raw { float4 v[2][4]; };

template <bool SHIFT_IN>
__device__ __forceinline__ void f16_load(F16Raw& r, const float2* __restrict__ xr, int c0) {
#pragma unroll
    for (int u = 0; u < 2; u++)
#pragma unroll
        for (int n3 = 0; n3 < 4; n3++) {
            const int src = SHIFT_IN ? ((n3 + 2) & 3) : n3;
            r.v[u][n3] = __ldg(reinterpret_cast<const float4*>(xr + c0 + 2 * u + 4096 * src));
        }
}

template <bool INV, bool SHIFT_IN, bool SHIFT_OUT, bool MAG>
__global__ void __launch_bounds__(F16_NT, 1)
fftp16k_kernel(const float2* __restrict__ x, void* __restrict__ out_, long long rows, float scale, const float* __restrict__ tw) {
    constexpr int N = 16384;
    extern __shared__ __align__(16) float smem[];
    float* sre = smem;
    float* sim = smem + 4 * F16_B;
    const int t = threadIdx.x;
    const float* tw0 = tw + 1024 + 8192;        // W_16384^c, c < 4096
    const long long row_step = gridDim.x;
    long long row = blockIdx.x;
    if (row >= rows) return;

    // F3 / F0 geometry of this thread's two groups: gl = t + 512*half = lsb + 4*(k0 + 16*k1)
    int g_k0[2], g_k1[2];
    const int lsb = t & 3;
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const int gl = t + F16_NT * half;
        g_k0[half] = (gl >> 2) & 15;
        g_k1[half] = gl >> 6;
    }
    // column pairs of the quad's group (k0, k1): pi = 128*k0 + 8*k1 + jj, jj = 2*lsb + u; c = 2*pi
    // shared word of column pair (k0, k1, jj): 272*k0 + 16*k1 + ((2*jj + 4*fp_rot(k0, k1)) & 15)
    auto f0_store = [&](const F16Raw& r, int half) {
        const int k0 = g_k0[half], k1 = g_k1[half];
        const int rot4 = 4 * fp_rot(k0, k1);
        const int rowbase = 272 * k0 + 16 * k1;
#pragma unroll
        for (int u = 0; u < 2; u++) {
            cp a[4];
#pragma unroll
            for (int n3 = 0; n3 < 4; n3++) {
                planar_of(r.v[u][n3], a[n3].re, a[n3].im);
            }
            r4<INV>(a[0], a[1], a[2], a[3]);
            const int jj = 2 * lsb + u;
            const int c = 2 * (128 * k0 + 8 * k1 + jj);
            cp w1;
            w1.re = __ldg(reinterpret_cast<const float2*>(tw0 + c));
            w1.im = __ldg(reinterpret_cast<const float2*>(tw0 + 4096 + c));
            if (INV) w1.im = pneg(w1.im);
            const cp w2 = cmul(w1, w1);
            a[1] = cmul(a[1], w1);
            a[2] = cmul(a[2], w2);
            a[3] = cmul(a[3], cmul(w2, w1));
            const int off = rowbase + ((2 * jj + rot4) & 15);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                *reinterpret_cast<float2*>(sre + k * F16_B + off) = a[k].re;
                *reinterpret_cast<float2*>(sim + k * F16_B + off) = a[k].im;
            }
        }
    };
    auto c0_of = [&](int half) { return 2 * (128 * g_k0[half] + 8 * g_k1[half] + 2 * lsb); };

    // ---- prologue: F0 of the first row ------------------------------------------------------------------------
    {
        const float2* xr = x + (size_t)row * (size_t)N;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            F16Raw raw;
            f16_load<SHIFT_IN>(raw, xr, c0_of(half));
            f0_store(raw, half);
        }
    }
    __syncthreads();

    const int sb = t >> 7, tt = t & 127;
    float* bre = sre + sb * F16_B;
    float* bim = sim + sb * F16_B;
    for (; row < rows; row += row_step) {
        const long long nrow = row + row_step;
        const bool has_next = nrow < rows;
        const float2* xn = x + (size_t)(has_next ? nrow : row) * (size_t)N;
        // one thread asks L2 for the row after the next while the current one is computed
        if (t == 0 && nrow + row_step < rows) {
            const float2* pf = x + (size_t)(nrow + row_step) * (size_t)N;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(pf), "r"(N * 8) : "memory");
        }
        cp v[16];
        // ------------------------------------------------------------------ F1: stride 256 inside sub-block sb
        {
            const int c = 2 * tt;
            const int g = tt >> 3, j = 2 * (tt & 7);
            int off[4];   // row>>1 takes 8 values but only (row>>1)&3 matters: 4 rotations
#pragma unroll
            for (int r = 0; r < 4; r++) off[r] = 16 * g + ((j + 4 * (((g >> 1) + r) & 3)) & 15);
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++) {
                v[n2].re = *reinterpret_cast<const float2*>(bre + 272 * n2 + off[(n2 >> 1) & 3]);
                v[n2].im = *reinterpret_cast<const float2*>(bim + 272 * n2 + off[(n2 >> 1) & 3]);
            }
            r16<INV>(v);
            cp w1;
            w1.re = *reinterpret_cast<const float2*>(tw + c);
            w1.im = *reinterpret_cast<const float2*>(tw + 256 + c);
            if (INV) w1.im = pneg(w1.im);
            apply_twiddles<true>(v, w1);
#pragma unroll
            for (int s = 0; s < 16; s++) {
                const int k0 = r16_k(s);
                *reinterpret_cast<float2*>(bre + 272 * k0 + off[(k0 >> 1) & 3]) = v[s].re;
                *reinterpret_cast<float2*>(bim + 272 * k0 + off[(k0 >> 1) & 3]) = v[s].im;
            }
        }
        // the F1 -> F2 exchange stays inside a sub-block: named barrier over its 128 threads
        asm volatile("bar.sync %0, 128;" ::"r"(sb + 1) : "memory");
        // ------------------------------------------------------------------ F2: stride 16
        {
            const int k0 = tt >> 3, n0 = 2 * (tt & 7);
            int off2[4];
#pragma unroll
            for (int r = 0; r < 4; r++) off2[r] = 272 * k0 + ((n0 + 4 * ((r + (k0 >> 1)) & 3)) & 15);
            const float4* tw2 = reinterpret_cast<const float4*>(tw + 512) + (n0 >> 1);
#pragma unroll
            for (int n1 = 0; n1 < 16; n1++) {
                const int a = 16 * n1 + off2[(n1 >> 1) & 3];
                v[n1].re = *reinterpret_cast<const float2*>(bre + a);
                v[n1].im = *reinterpret_cast<const float2*>(bim + a);
            }
            r16<INV>(v);
#pragma unroll
            for (int s = 1; s < 16; s++) {
                const int k1 = r16_k(s);
                const float4 f = __ldg(tw2 + 8 * k1);
                cp w;
                w.re = make_float2(f.x, f.y);
                w.im = make_float2(f.z, f.w);
                v[s] = INV ? cmul_conj(v[s], w) : cmul(v[s], w);
            }
#pragma unroll
            for (int s = 0; s < 16; s++) {
                const int k1 = r16_k(s);
                const int a = 16 * k1 + off2[(k1 >> 1) & 3];
                *reinterpret_cast<float2*>(bre + a) = v[s].re;
                *reinterpret_cast<float2*>(bim + a) = v[s].im;
            }
        }
        __syncthreads();
        // ------------------------------------------------------------------ F3 of this row  ||  F0 of the next row
#pragma unroll
        for (int half = 0; half < 2; half++) {
            F16Raw raw;
            if (has_next) f16_load<SHIFT_IN>(raw, xn, c0_of(half));
            const int k0 = g_k0[half], k1 = g_k1[half];
            const int r = fp_rot(k0, k1);
            const int base = lsb * F16_B + 272 * k0 + 16 * k1;
            cp P[8];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int a = base + 4 * ((q + r) & 3);
                const float4 fr = *reinterpret_cast<const float4*>(sre + a);
                const float4 fi = *reinterpret_cast<const float4*>(sim + a);
                P[2 * q].re = make_float2(fr.x, fr.y); P[2 * q + 1].re = make_float2(fr.z, fr.w);
                P[2 * q].im = make_float2(fi.x, fi.y); P[2 * q + 1].im = make_float2(fi.z, fi.w);
            }
            __syncwarp();      // the quad has read its 4 x 16 words: F0 of the next row may overwrite them
            fft16_dif<INV>(P);
            // slot j holds k2 = bitrev4(j); k = lsb + 4*(k0 + 16*k1 + 256*k2)
            const size_t klow = (size_t)lsb + 4 * (size_t)(k0 + 16 * k1);
            if constexpr (MAG) {
                float* o = reinterpret_cast<float*>(out_) + (size_t)row * N + klow;
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    pk m2 = pfma(P[m].re, P[m].re, pmul(P[m].im, P[m].im));
                    const int ka = bitrev4(2 * m) ^ (SHIFT_OUT ? 8 : 0), kb = bitrev4(2 * m + 1) ^ (SHIFT_OUT ? 8 : 0);
                    o[1024 * ka] = sqrt_fast(m2.x) * scale;
                    o[1024 * kb] = sqrt_fast(m2.y) * scale;
                }
            } else {
                float2* o = reinterpret_cast<float2*>(out_) + (size_t)row * N + klow;
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    const int ka = bitrev4(2 * m) ^ (SHIFT_OUT ? 8 : 0), kb = bitrev4(2 * m + 1) ^ (SHIFT_OUT ? 8 : 0);
                    o[1024 * ka] = make_float2(P[m].re.x * scale, P[m].im.x * scale);
                    o[1024 * kb] = make_float2(P[m].re.y * scale, P[m].im.y * scale);
                }
            }
            if (has_next) f0_store(raw, half);
        }
        __syncthreads();
    }
}

namespace {
template <bool INV, bool SI, bool SO, bool MAG>
int f16_launch(const void* in, void* out, size_t rows, float scale, cudaStream_t st) {
    const size_t smem = (size_t)2 * 4 * F16_B * sizeof(float);
    auto kern = fftp16k_kernel<INV, SI, SO, MAG>;
    static PerDeviceOnce configured;   // per instantiation and device
    if (configured.need()) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured.mark();
    }
    const float* tw = fftp_twiddles();
    if (!tw) return -1001;
    size_t ctas = (size_t)sm_count();
    if (ctas > rows) ctas = rows;
    kern<<<(unsigned)ctas, F16_NT, smem, st>>>(reinterpret_cast<const float2*>(in), out, (long long)rows, scale, tw);
    BDSP_LAUNCHED();
    return 0;
}
}  // namespace

// rows of 16384 c32 points (FftRoute::Packed16k)
int fftp16k(const void* in, void* out, size_t rows, bool inverse, bool shift_in, bool shift_out, bool magnitude, float scale, cudaStream_t st) {
    return fftp_with_flags<true, true>(inverse, shift_in, shift_out, magnitude, [&](auto inv, auto si, auto so, auto mag) {
        return f16_launch<inv, si, so, mag>(in, out, rows, scale, st);
    });
}

}  // namespace bdsp
