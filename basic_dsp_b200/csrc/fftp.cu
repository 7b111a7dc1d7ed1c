// Packed-FP32x2 shared-memory FFT kernels for c32 (and real f32 input) sequences.
//
// fftp_kernel: one 128-thread group per 4096 points, same building blocks as the fused overlap-save kernel (ols4096.cuh):
//   F0  radix-R0 DIF over stride 4096 (global -> shared), twiddle W_n^{k0' c}          (n = 4096*R0, R0 in {2, 4})
//   F1  radix-16 DIF over stride 256, F2 radix-16 DIF over stride 16 (in place in shared memory)
//   F3  radix-16 DIF over 16 contiguous points in registers -> global, natural order
//       (output k = k0' + R0*(k0 + 16*k1 + 256*k2); lanes walk k0', k0 so that stores coalesce)
// Modes (template parameters):
//   plain     n = 4096 / 8192 / 16384, one sequence per CTA (R0 = 1, 2, 4)
//   NATQ = Q  16/Q sequences of 256*Q points per CTA (512, 1024, 2048): F1 becomes a radix-Q step inside every sequence
//   ROWS      last pass of a multi-pass transform: four adjacent 4096-point rows per CTA, transposing store
//   TQ = Q    last pass with 16/Q adjacent rows of 256*Q points per CTA (128 threads), transposing store
//   RIN       the input holds real scalars
//   FRAMES    the sequences are strided frames of one signal, with an optional window multiplied in on the first load
//   PSUM      (with FRAMES) Welch's power sum: |X|^2 added into a partial row per CTA instead of stored
// fftp_col16_kernel / fftp_col256_kernel: first pass(es) of the multi-pass transforms: 16- / 256-point (NH = 2: 32- / 512-point)
//   columns of 16 adjacent columns per CTA, inter-pass twiddle evaluated with sincospif on exact arguments.
// Launchers, one per route of fft_route.h: fftp_single (complex or real rows), fftp_frames (strided frames), fftp_frames_psum
//   (Welch power sums, welch_route), fftp_two_pass (2^15..2^20), fftp_three_pass
//   (2^21..2^24), fftp_rows_pass (packed last pass, also behind a generic column pass).
// Replaces rustfft for these lengths (vector/src/vector_types/time_freq/mod.rs:45-58) incl. the fused
// fft_shift (time_to_freq.rs:163), ifft's scale + ifft_shift (freq_to_time.rs:165-167) and magnitude.
#include <map>
#include <mutex>
#include <vector>

#include "fftp.cuh"

namespace bdsp {
using namespace ols16;

// ROWS = true (R0 = 4): the CTA transforms FOUR independent, adjacent 4096-point rows (no F0) and
// writes result k of row r to out[(r0 + r) + n1 * k]: the transposing last pass of a two-pass transform of
// n1 * 4096 points, with the four rows providing the contiguous 32 bytes of every store sector.
// TQ = Q in {2, 4} (with ROWS, R0 = 1): the CTA's 4096 points are 16/Q adjacent rows of 256*Q points (k0 = (16/Q)*q + row):
// the first stage is a radix-Q butterfly inside every row, the other two stages are unchanged; 128 threads and 35 KB of
// shared memory per CTA as for a plain 4096-point transform (which runs at the HBM roofline); the adjacent rows make
// the transposing stores fill 32-byte (Q = 4) or 64-byte (Q = 2) runs.
// RIN = true (forward, no ROWS): `x` holds REAL scalars (one float per point); the first stage loads two adjacent reals
// per column pair and the imaginary parts start as zero.
// SQ = P in {4, 8} (with NATQ = 1): the CTA's 4096 contiguous points are 256/P rows of 16*P points (64, 128): the first stage
// is empty, the second one is a radix-P step inside every row (instead of radix 16), the third one is unchanged.
// NATQ = Q in {1, 2, 4, 8} (R0 = 1, no ROWS): the CTA's 4096 contiguous points are 16/Q independent rows of 256*Q points
// (k0 = q + Q*row); the first stage is a radix-Q butterfly inside every row, results are stored in natural order.
// Batched 512 / 1024 / 2048-point transforms with the structure of the 4096-point kernel.
// FRAMES = true (forward, no ROWS, n <= 8192): the sequences are frames of one signal that start `hop` points apart (hop
// even): point p of the CTA's N points is read from x[(row * (N / n) + p / n) * hop + p % n], n the sequence length, and,
// when `win` is not null, multiplied by win[p % n] as it is loaded.  The product is rounded on its own (__fmul_rn), as the
// separate multiplier pass (fft.cu in_mul_rows_kernel) rounds it, so that the result is the one of that pass followed by the
// plain kernel.
// PSUM = true (with FRAMES): Welch's power sum.  `rows` counts the groups of N / n frames, of which only the first `frames`
// frames exist: a frame index >= frames loads nothing and transforms zeros, so the last group may be incomplete.  Instead of
// storing X, F3 adds |X|^2 (the MAG epilogue's pfma, without the sqrt) into the CTA's partial row out[blockIdx.x * N + k]:
// every slot has one owner thread, the CTA's first row stores and later rows add, and after the last row the CTA sums its
// N / n frames' slots into the first n (fixed order, no atomics).  No scale, no fft_shift: welch_final_kernel applies them.
#define FP_MINB256 2   // CTAs per SM for the 256-thread 8192-point kernel
template <int R0, bool INV, bool SHIFT_IN, bool SHIFT_OUT, bool MAG, bool ROWS, int TQ = 0, int NATQ = 0, bool RIN = false, int SQ = 0,
          bool FRAMES = false, bool PSUM = false>
__global__ void __launch_bounds__(128 * R0, R0 == 2 ? FP_MINB256 : 4 / R0)
fftp_kernel(const float2* __restrict__ x, void* __restrict__ out_, long long rows, float scale, const float* __restrict__ tw, int n1, int n2c,
            long long hop, const float* __restrict__ win, long long frames) {
    constexpr int NSB = R0;               // sub-blocks (4096-point transforms) owned by this CTA
    constexpr int NT = 128 * NSB;         // threads
    constexpr int N = 4096 * R0;
    constexpr int FP_B = FP_B_OF(NSB);
    extern __shared__ __align__(16) float smem[];
    float* sre = smem;
    float* sim = smem + NSB * FP_B;
    const int t = threadIdx.x;
    constexpr int NU = R0 > 1 ? 2048 / NT : 1;   // column pairs per thread in F0
    const long long row_step = gridDim.x;
    long long row = blockIdx.x;
    for (; row < rows; row += row_step) {
    // ROWS: `row` counts groups of NSB rows; groups_per_seq = n1 / NSB
    constexpr bool R1K = TQ > 0;
    constexpr int RPC = R1K ? 16 / TQ : NSB;      // rows per CTA (ROWS)
    constexpr int RLEN = R1K ? 256 * TQ : 4096;   // row length (ROWS)
    // ROWS: the sequence has n1 * n2c rows of RLEN points; row (k1, k2o) sits at tmp[(k1 * n2c + k2o) * RLEN] and its result
    // index kk goes to out[k1 + n1 * k2o + n1 * n2c * kk].  n2c = 1: last pass of a two-pass transform; n2c > 1: of a
    // three-pass transform (k2o = index of the middle pass).  A CTA takes RPC rows with consecutive k1.
    const int gpo = ROWS ? n1 / RPC : 1;
    const size_t per_seq = (size_t)gpo * (size_t)(ROWS ? n2c : 1);
    const size_t seq = ROWS ? (size_t)row / per_seq : (size_t)row;
    const int k2o = ROWS ? (int)(((size_t)row % per_seq) / (size_t)gpo) : 0;
    const int grp = ROWS ? (int)(((size_t)row % per_seq) % (size_t)gpo) : 0;
    const size_t seq_len = ROWS ? (size_t)RLEN * (size_t)n1 * (size_t)n2c : (size_t)N;
    const size_t rstride = ROWS ? (size_t)RLEN * (size_t)n2c : (size_t)RLEN;
    const float2* xr = x + seq * seq_len + (ROWS ? (size_t)k2o * RLEN + (size_t)grp * RPC * rstride : 0);   // NATQ: N = 4096 = one group of rows

    // two adjacent points starting at complex element pointer gp: {re0, im0, re1, im1}
    auto ldpair = [&](const float2* gp) -> float4 {
        if constexpr (FRAMES) {
            constexpr int FN = SQ ? 16 * SQ : NATQ ? 256 * NATQ : N;   // frame length
            const int p = (int)(gp - xr);
            const long long fr = (long long)seq * (N / FN) + p / FN;
            if constexpr (PSUM) { if (fr >= frames) return make_float4(0.f, 0.f, 0.f, 0.f); }
            const long long src = fr * hop + p % FN;
            float4 v;
            if constexpr (RIN) {
                const float2 r = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(x) + src));
                v = make_float4(r.x, 0.f, r.y, 0.f);
            } else {
                v = __ldg(reinterpret_cast<const float4*>(x + src));
            }
            if (win) {
                const float2 w = __ldg(reinterpret_cast<const float2*>(win + p % FN));
                v.x = __fmul_rn(v.x, w.x);
                v.z = __fmul_rn(v.z, w.y);
                if constexpr (!RIN) {
                    v.y = __fmul_rn(v.y, w.x);
                    v.w = __fmul_rn(v.w, w.y);
                }
            }
            return v;
        } else if constexpr (RIN) {
            const float2 r = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(x) + (gp - x)));
            return make_float4(r.x, 0.f, r.y, 0.f);
        } else {
            return __ldg(reinterpret_cast<const float4*>(gp));
        }
    };
    cp v[16];
    // ------------------------------------------------------------------ F0: radix-R0 over stride 4096
    if constexpr (R0 > 1 && !ROWS) {
        const float* tw0 = tw + 1024 + (R0 == 4 ? 8192 : 0);
#pragma unroll
        for (int u = 0; u < NU; u++) {
            const int pi = t + NT * u;     // column pair index, c = 2*pi
            const int c = 2 * pi;
            cp a[R0];
#pragma unroll
            for (int n3 = 0; n3 < R0; n3++) {
                const int src = SHIFT_IN ? ((n3 + R0 / 2) % R0) : n3;
                const float4 ab = ldpair(xr + c + 4096 * src);
                a[n3].re = make_float2(ab.x, ab.z);
                a[n3].im = make_float2(ab.y, ab.w);
            }
            if constexpr (R0 == 4) r4<INV>(a[0], a[1], a[2], a[3]);
            else { cp s = cadd(a[0], a[1]); cp d = csub(a[0], a[1]); a[0] = s; a[1] = d; }
            cp w1;
            w1.re = __ldg(reinterpret_cast<const float2*>(tw0 + c));
            w1.im = __ldg(reinterpret_cast<const float2*>(tw0 + 4096 + c));
            if (INV) w1.im = pneg(w1.im);
            a[1] = cmul(a[1], w1);
            if constexpr (R0 == 4) {
                cp w2 = cmul(w1, w1);
                a[2] = cmul(a[2], w2);
                a[3] = cmul(a[3], cmul(w2, w1));
            }
            const int prow = pi >> 7, g = (pi >> 3) & 15, j = 2 * (pi & 7);
            const int off = 272 * prow + 16 * g + ((j + 4 * fp_rot(prow, g)) & 15);
#pragma unroll
            for (int k = 0; k < R0; k++) {
                *reinterpret_cast<float2*>(sre + k * FP_B + off) = a[k].re;
                *reinterpret_cast<float2*>(sim + k * FP_B + off) = a[k].im;
            }
        }
        __syncthreads();
    }
    // ------------------------------------------------------------------ F1: stride 256 inside every sub-block
    const int sb = t >> 7, tt = t & 127;
    float* bre = sre + sb * FP_B;
    float* bim = sim + sb * FP_B;
    {
        const int c = 2 * tt;
        const int g = tt >> 3, j = 2 * (tt & 7);
        int off[4];   // row>>1 takes 8 values but only (row>>1)&3 matters: 4 rotations
#pragma unroll
        for (int r = 0; r < 4; r++) off[r] = 16 * g + ((j + 4 * (((g >> 1) + r) & 3)) & 15);
        if constexpr (R0 > 1 && !ROWS) {
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++) {
                v[n2].re = *reinterpret_cast<const float2*>(bre + 272 * n2 + off[(n2 >> 1) & 3]);
                v[n2].im = *reinterpret_cast<const float2*>(bim + 272 * n2 + off[(n2 >> 1) & 3]);
            }
        } else {
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++) {
                const int src = SHIFT_IN ? (n2 ^ 8) : n2;
                const float2* gp = NATQ ? xr + (n2 / (NATQ ? NATQ : 1)) * (256 * NATQ) + 256 * ((n2 % (NATQ ? NATQ : 1)) ^ (SHIFT_IN ? NATQ / 2 : 0)) +
                                              (NATQ == 1 && SQ == 0 && SHIFT_IN ? (c ^ 128) : c)
                                   : R1K ? xr + (n2 % RPC) * rstride + 256 * (n2 / RPC) + c : xr + (ROWS ? sb * rstride : 0) + c + 256 * src;
                const float4 ab = ldpair(gp);
                v[n2].re = make_float2(ab.x, ab.z);
                v[n2].im = make_float2(ab.y, ab.w);
            }
        }
        if constexpr (NATQ == 1) {
            // sixteen 256-point rows: the first stage is empty
#pragma unroll
            for (int k0 = 0; k0 < 16; k0++) {
                *reinterpret_cast<float2*>(bre + 272 * k0 + off[(k0 >> 1) & 3]) = v[k0].re;
                *reinterpret_cast<float2*>(bim + 272 * k0 + off[(k0 >> 1) & 3]) = v[k0].im;
            }
        } else if constexpr (NATQ > 1) {
            // radix Q inside each row (v[Q*row + q] -> v[Q*row + q']), then W_{256Q}^{c q'}
            constexpr int TWO = NATQ == 2 ? FP_TW_512 : NATQ == 4 ? FP_TW_1K : FP_TW_2K;
            cp w[8];
            w[1].re = *reinterpret_cast<const float2*>(tw + TWO + c);
            w[1].im = *reinterpret_cast<const float2*>(tw + TWO + 256 + c);
            if (INV) w[1].im = pneg(w[1].im);
            if constexpr (NATQ >= 4) { w[2] = cmul(w[1], w[1]); w[3] = cmul(w[2], w[1]); }
            if constexpr (NATQ == 8) { w[4] = cmul(w[2], w[2]); w[5] = cmul(w[4], w[1]); w[6] = cmul(w[4], w[2]); w[7] = cmul(w[4], w[3]); }
#pragma unroll
            for (int r = 0; r < 16 / NATQ; r++) {
                cp* u = v + NATQ * r;
                if constexpr (NATQ == 2) { const cp a = cadd(u[0], u[1]), b = csub(u[0], u[1]); u[0] = a; u[1] = b; }
                else if constexpr (NATQ == 4) r4<INV>(u[0], u[1], u[2], u[3]);
                else {
                    // 8-point DIF: a_j = x_j + x_{j+4}, b_j = (x_j - x_{j+4}) W8^j; X[2m] = DFT4(a)[m], X[2m+1] = DFT4(b)[m]
                    cp a0 = cadd(u[0], u[4]), a1 = cadd(u[1], u[5]), a2 = cadd(u[2], u[6]), a3 = cadd(u[3], u[7]);
                    cp b0 = csub(u[0], u[4]), b1 = mul_w16<2, INV>(csub(u[1], u[5])), b2 = mul_w16<4, INV>(csub(u[2], u[6])),
                       b3 = mul_w16<6, INV>(csub(u[3], u[7]));
                    r4<INV>(a0, a1, a2, a3);
                    r4<INV>(b0, b1, b2, b3);
                    u[0] = a0; u[2] = a1; u[4] = a2; u[6] = a3; u[1] = b0; u[3] = b1; u[5] = b2; u[7] = b3;
                }
#pragma unroll
                for (int q = 1; q < NATQ; q++) u[q] = cmul(u[q], w[q]);
            }
#pragma unroll
            for (int k0 = 0; k0 < 16; k0++) {
                *reinterpret_cast<float2*>(bre + 272 * k0 + off[(k0 >> 1) & 3]) = v[k0].re;
                *reinterpret_cast<float2*>(bim + 272 * k0 + off[(k0 >> 1) & 3]) = v[k0].im;
            }
        } else if constexpr (R1K) {
            // radix Q inside each row (v[row + RPC*q] -> v[row + RPC*q']), then W_{256Q}^{c q'}  (Q = 1: nothing to do)
            if constexpr (TQ > 1) {
                cp w1;
                constexpr int TWO = TQ == 2 ? FP_TW_512 : TQ == 4 ? FP_TW_1K : FP_TW_2K;
                w1.re = *reinterpret_cast<const float2*>(tw + TWO + c);
                w1.im = *reinterpret_cast<const float2*>(tw + TWO + 256 + c);
                if (INV) w1.im = pneg(w1.im);
                if constexpr (TQ == 8) {
                    cp w[8];
                    w[1] = w1; w[2] = cmul(w1, w1); w[3] = cmul(w[2], w1); w[4] = cmul(w[2], w[2]);
                    w[5] = cmul(w[4], w1); w[6] = cmul(w[4], w[2]); w[7] = cmul(w[4], w[3]);
#pragma unroll
                    for (int r = 0; r < 2; r++) {   // row r holds v[r + 2q]
                        cp a0 = cadd(v[r], v[r + 8]), a1 = cadd(v[r + 2], v[r + 10]), a2 = cadd(v[r + 4], v[r + 12]), a3 = cadd(v[r + 6], v[r + 14]);
                        cp b0 = csub(v[r], v[r + 8]), b1 = mul_w16<2, INV>(csub(v[r + 2], v[r + 10])),
                           b2 = mul_w16<4, INV>(csub(v[r + 4], v[r + 12])), b3 = mul_w16<6, INV>(csub(v[r + 6], v[r + 14]));
                        r4<INV>(a0, a1, a2, a3);
                        r4<INV>(b0, b1, b2, b3);
                        v[r] = a0; v[r + 4] = cmul(a1, w[2]); v[r + 8] = cmul(a2, w[4]); v[r + 12] = cmul(a3, w[6]);
                        v[r + 2] = cmul(b0, w[1]); v[r + 6] = cmul(b1, w[3]); v[r + 10] = cmul(b2, w[5]); v[r + 14] = cmul(b3, w[7]);
                    }
                } else if constexpr (TQ == 4) {
                    const cp w2 = cmul(w1, w1), w3 = cmul(w2, w1);
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        r4<INV>(v[r], v[r + 4], v[r + 8], v[r + 12]);
                        v[r + 4] = cmul(v[r + 4], w1);
                        v[r + 8] = cmul(v[r + 8], w2);
                        v[r + 12] = cmul(v[r + 12], w3);
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < 8; r++) {
                        const cp a = cadd(v[r], v[r + 8]), b = csub(v[r], v[r + 8]);
                        v[r] = a;
                        v[r + 8] = cmul(b, w1);
                    }
                }
            }
#pragma unroll
            for (int k0 = 0; k0 < 16; k0++) {
                *reinterpret_cast<float2*>(bre + 272 * k0 + off[(k0 >> 1) & 3]) = v[k0].re;
                *reinterpret_cast<float2*>(bim + 272 * k0 + off[(k0 >> 1) & 3]) = v[k0].im;
            }
        } else {
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
    }
    __syncthreads();
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
        if constexpr (SQ > 0) {
            // rows of 16*SQ points: g = SQ*rowsub + g'; radix SQ over g' (natural order), then W_{16 SQ}^{kg j}, j = n0, n0 + 1.
            // SHIFT_IN (rotation by half a row = SQ/2 steps of g'): the butterfly inputs are taken from g' ^ (SQ/2).
            const float4* tws = reinterpret_cast<const float4*>(tw + (SQ == 4 ? FP_TW_S4 : FP_TW_S8)) + (n0 >> 1);
#pragma unroll
            for (int r = 0; r < 16 / SQ; r++) {
                cp u[SQ];
#pragma unroll
                for (int q = 0; q < SQ; q++) u[q] = v[SQ * r + (SHIFT_IN ? (q ^ (SQ / 2)) : q)];
                if constexpr (SQ == 4) r4<INV>(u[0], u[1], u[2], u[3]);
                else {
                    cp a0 = cadd(u[0], u[4]), a1 = cadd(u[1], u[5]), a2 = cadd(u[2], u[6]), a3 = cadd(u[3], u[7]);
                    cp b0 = csub(u[0], u[4]), b1 = mul_w16<2, INV>(csub(u[1], u[5])), b2 = mul_w16<4, INV>(csub(u[2], u[6])),
                       b3 = mul_w16<6, INV>(csub(u[3], u[7]));
                    r4<INV>(a0, a1, a2, a3);
                    r4<INV>(b0, b1, b2, b3);
                    u[0] = a0; u[2] = a1; u[4] = a2; u[6] = a3; u[1] = b0; u[3] = b1; u[5] = b2; u[7] = b3;
                }
#pragma unroll
                for (int q = 0; q < SQ; q++) {
                    if (q > 0) {
                        const float4 f = __ldg(tws + 8 * q);
                        cp w;
                        w.re = make_float2(f.x, f.y);
                        w.im = make_float2(f.z, f.w);
                        u[q] = INV ? cmul_conj(u[q], w) : cmul(u[q], w);
                    }
                    v[SQ * r + q] = u[q];
                }
            }
#pragma unroll
            for (int n1 = 0; n1 < 16; n1++) {
                const int a = 16 * n1 + off2[(n1 >> 1) & 3];
                *reinterpret_cast<float2*>(bre + a) = v[n1].re;
                *reinterpret_cast<float2*>(bim + a) = v[n1].im;
            }
        } else {
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
    }
    __syncthreads();
    // ------------------------------------------------------------------ F3: 16 contiguous points -> global
#pragma unroll 1
    for (int half = 0; half < 2; half++) {
        const int gl = t + NT * half;                 // local group index: lsb + NSB*(k0 + 16*k1)
        // NATQ: lanes take the low 3 bits of k0 and the low 2 bits of k1 (quarter-warps still walk k0: conflict-free 128-bit
        // loads), so that one store instruction writes 4*Q-point runs (16 consecutive results for 1024-point rows)
        const int lsb = gl % NSB;
        // (Q = 2: lanes take q' = k0 bit 0 and all of k1, with the quarter-warp on (q', k1 bits 1-2) so that the eight 128-bit
        // loads still fall into eight different bank windows: 32 consecutive results per store instruction)
        // (SQ: lanes take all of k1 = SQ*rowsub + kg and k0 bit 0: runs of SQ results per row and store instruction)
        const int k0 = SQ ? (gl >> 4) : (NATQ == 2 || NATQ == 1) ? ((gl & 1) | (((gl >> 5) & 7) << 1))
                       : NATQ ? ((gl & 7) | (((gl >> 5) & 1) << 3)) : (gl / NSB) & 15;
        const int k1 = SQ ? (gl & 15) : (NATQ == 2 || NATQ == 1) ? (((gl >> 3) & 1) | (((gl >> 1) & 3) << 1) | (((gl >> 4) & 1) << 3))
                       : NATQ ? (((gl >> 3) & 3) | ((gl >> 6) << 2)) : gl / (16 * NSB);
        const int r = fp_rot(k0, k1);
        const int base = lsb * FP_B + 272 * k0 + 16 * k1;
        cp P[8];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int a = base + 4 * ((q + r) & 3);
            const float4 fr = *reinterpret_cast<const float4*>(sre + a);
            const float4 fi = *reinterpret_cast<const float4*>(sim + a);
            P[2 * q].re = make_float2(fr.x, fr.y); P[2 * q + 1].re = make_float2(fr.z, fr.w);
            P[2 * q].im = make_float2(fi.x, fi.y); P[2 * q + 1].im = make_float2(fi.z, fi.w);
        }
        fft16_dif<INV>(P);
        // slot j holds k2 = bitrev4(j); k = lsb + R0*(k0 + 16*k1 + 256*k2)
        // (ROWS: k = (NSB*grp + lsb) + n1*(k0 + 16*k1 + 256*k2))
        // (TQ: row = k0 % RPC, k = (RPC*grp + row) + n1*((k0 / RPC) + Q*(k1 + 16*k2)))
        const size_t kst = ROWS ? (size_t)n1 * (size_t)n2c : (size_t)R0;
        const size_t kbase = ROWS ? (size_t)n1 * (size_t)k2o : 0;
        // (NATQ: row = k0 / Q, k = row*256*Q + (k0 % Q) + Q*(k1 + 16*k2))
        // (SQ: row = k0*(16/SQ) + k1/SQ, k = row*16*SQ + (k1 % SQ) + SQ*k2)
        const size_t klow = SQ ? (size_t)((k0 * (16 / (SQ ? SQ : 1)) + k1 / (SQ ? SQ : 1)) * (16 * SQ) + (k1 % (SQ ? SQ : 1)))
                            : NATQ ? (size_t)((k0 / (NATQ ? NATQ : 1)) * (256 * NATQ) + (k0 % (NATQ ? NATQ : 1)) + NATQ * k1)
                            : R1K ? kbase + (size_t)(RPC * grp + (k0 % RPC)) + kst * (size_t)((k0 / RPC) + TQ * k1)
                                : kbase + (ROWS ? (size_t)(NSB * grp + lsb) : (size_t)lsb) + kst * (size_t)(k0 + 16 * k1);
        const size_t k2s = SQ ? (size_t)SQ : NATQ ? (size_t)(16 * NATQ) : R1K ? (size_t)(16 * TQ) * kst : (size_t)256 * kst;
        if constexpr (PSUM) {
            float* o = reinterpret_cast<float*>(out_) + (size_t)blockIdx.x * N + klow;
            const bool first = row == (long long)blockIdx.x;
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const pk m2 = pfma(P[m].re, P[m].re, pmul(P[m].im, P[m].im));
                float* a = o + k2s * bitrev4(2 * m);
                float* b = o + k2s * bitrev4(2 * m + 1);
                *a = first ? m2.x : *a + m2.x;
                *b = first ? m2.y : *b + m2.y;
            }
        } else if constexpr (MAG) {
            float* o = reinterpret_cast<float*>(out_) + seq * seq_len + klow;
#pragma unroll
            for (int m = 0; m < 8; m++) {
                pk m2 = pfma(P[m].re, P[m].re, pmul(P[m].im, P[m].im));
                const int ka = bitrev4(2 * m) ^ (SHIFT_OUT ? 8 : 0), kb = bitrev4(2 * m + 1) ^ (SHIFT_OUT ? 8 : 0);
                o[k2s * ka] = sqrtf(m2.x) * scale;
                o[k2s * kb] = sqrtf(m2.y) * scale;
            }
        } else {
            float2* o = reinterpret_cast<float2*>(out_) + seq * seq_len + klow;
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int ka = bitrev4(2 * m) ^ (SHIFT_OUT ? 8 : 0), kb = bitrev4(2 * m + 1) ^ (SHIFT_OUT ? 8 : 0);
                o[k2s * ka] = make_float2(P[m].re.x * scale, P[m].im.x * scale);
                o[k2s * kb] = make_float2(P[m].re.y * scale, P[m].im.y * scale);
            }
        }
    }
    if (row + row_step < rows) __syncthreads();   // the next row's F0 overwrites the shared memory F3 just read
    }  // rows
    if constexpr (PSUM) {
        constexpr int FN = SQ ? 16 * SQ : NATQ ? 256 * NATQ : N;
        if constexpr (N / FN > 1) {
            __syncthreads();   // the slots other threads of this CTA wrote
            float* o = reinterpret_cast<float*>(out_) + (size_t)blockIdx.x * N;
            for (int k = t; k < FN; k += NT) {
                float s = o[k];
#pragma unroll 4
                for (int j = 1; j < N / FN; j++) s += o[j * FN + k];
                o[k] = s;
            }
        }
    }
}


// ------------------------------------------------------------------------------------------
// two-pass transforms of n = N1 * 4096 points, N1 in {16, 256}  (n = 2^16, 2^20)
//   pass A (below):  tmp[k1*4096 + n2] = W_n^{n2*k1} * sum_{n1} x[n1*4096 + n2] * W_N1^{n1*k1}
//   pass B (fftp_kernel<ROWS>): X[k1 + N1*k2] = sum_{n2} tmp[k1*4096 + n2] * W_4096^{n2*k2}
// Both passes move every point exactly once in full 32-byte sectors: 16 B/point of DRAM traffic each.
// The inter-pass twiddle is evaluated with sincospif on an exactly representable argument (m/n with
// m < 2^22) for the base root(s) and raised to the <= 15th power with the A_a*B_b product scheme.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ cp unit_root_pair(unsigned m0, unsigned m1, float two_over_n, bool inv) {
    // {W_n^{m0}, W_n^{m1}} = cos(2 pi m/n) - i sin(2 pi m/n); conjugated for the inverse transform
    float s0, c0, s1, c1;
    sincospif((float)m0 * two_over_n, &s0, &c0);
    sincospif((float)m1 * two_over_n, &s1, &c1);
    cp w;
    w.re = make_float2(c0, c1);
    w.im = inv ? make_float2(s0, s1) : make_float2(-s0, -s1);
    return w;
}

// W_32^a, a = 0..15 (forward sign: cos - i sin)
__device__ __constant__ float FP_C32[16] = {1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                                            0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f, 0.19509032201612826785f,
                                            0.f, -0.19509032201612826785f, -0.38268343236508977173f, -0.55557023301960222474f,
                                            -0.70710678118654752440f, -0.83146961230254523708f, -0.92387953251128675613f, -0.98078528040323044913f};
__device__ __constant__ float FP_S32[16] = {0.f, 0.19509032201612826785f, 0.38268343236508977173f, 0.55557023301960222474f,
                                            0.70710678118654752440f, 0.83146961230254523708f, 0.92387953251128675613f, 0.98078528040323044913f,
                                            1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                                            0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f, 0.19509032201612826785f};

// NH = 2: 32-point columns as a radix-2 step in front of the 16-point transform (two sweeps over the inputs: the
// second one is served by L2): y_h[a] = (x[a] + (-1)^h x[a + 16]) W_32^{a h}, X[2k' + h] = DFT16(y_h)[k'].
// RIN: x holds real scalars (see fftp_kernel)
// two adjacent points {re0, im0, re1, im1} at complex element pointer gp.  MUL: a multiplier table is fused into the load,
// indexed by the points' positions gp - xseq (even) inside their sequence (FftOpts::in_mul kinds 1 and 2: real window
// table / complex spectrum); MUL = false compiles to the plain load.
template <bool RIN, bool MUL> __device__ __forceinline__ float4 col_ldpair(const float2* x, const float2* gp, const InMul& im, const float2* xseq) {
    float4 v;
    if constexpr (RIN) {
        const float2 r = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(x) + (gp - x)));
        v = make_float4(r.x, 0.f, r.y, 0.f);
    } else {
        v = __ldg(reinterpret_cast<const float4*>(gp));
    }
    if constexpr (MUL) {
        const long long g = (long long)(gp - xseq);
        if (im.kind == 2) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float2*>(im.p) + g));
            v = make_float4(v.x * w.x - v.y * w.y, v.x * w.y + v.y * w.x, v.z * w.z - v.w * w.w, v.z * w.w + v.w * w.z);
        } else {
            const float2 w = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(im.p) + g));
            v = make_float4(v.x * w.x, v.y * w.x, v.z * w.y, v.w * w.y);
        }
    }
    return v;
}

template <bool INV, bool SHIFT_IN, int NH, bool RIN = false, bool MUL = false>
__global__ void __launch_bounds__(128) fftp_col16_kernel(const float2* __restrict__ x, float2* __restrict__ tmp, int log2n2, InMul im) {
    // n = 16 * NH * N2 points per sequence, N2 = 2^log2n2 = row length of the second pass
    const unsigned N2 = 1u << log2n2, N = 16u * NH * N2;
    const unsigned pi = blockIdx.x * 128u + threadIdx.x;   // column pair over all sequences
    const size_t seq = pi >> (log2n2 - 1);
    const unsigned c = 2u * (pi & (N2 / 2 - 1));
    const float2* xq = x + seq * N;
    const float2* xs = xq + c;
    float2* o = tmp + seq * N + c;
    const float ton = 2.0f / (float)N;
#pragma unroll 1
    for (int h = 0; h < NH; h++) {
        cp v[16];
#pragma unroll
        for (int a = 0; a < 16; a++) {
            if constexpr (NH == 1) {
                const int src = SHIFT_IN ? (a ^ 8) : a;
                const float4 ab = col_ldpair<RIN, MUL>(x, xs + (size_t)N2 * src, im, xq);
                v[a].re = make_float2(ab.x, ab.z);
                v[a].im = make_float2(ab.y, ab.w);
            } else {
                // SHIFT_IN rotates the input by n/2 = 16 rows: the two halves swap
                const float4 lo = col_ldpair<RIN, MUL>(x, xs + (size_t)N2 * (a + (SHIFT_IN ? 16 : 0)), im, xq);
                const float4 hi = col_ldpair<RIN, MUL>(x, xs + (size_t)N2 * (a + (SHIFT_IN ? 0 : 16)), im, xq);
                cp l, g;
                l.re = make_float2(lo.x, lo.z); l.im = make_float2(lo.y, lo.w);
                g.re = make_float2(hi.x, hi.z); g.im = make_float2(hi.y, hi.w);
                if (h == 0) v[a] = cadd(l, g);
                else v[a] = cmulc(csub(l, g), splat(FP_C32[a]), splat(INV ? FP_S32[a] : -FP_S32[a]));
            }
        }
        r16<INV>(v);
        if constexpr (NH == 1) {
            apply_twiddles<true>(v, unit_root_pair(c, c + 1, ton, INV));
        } else {
            apply_twiddles<true>(v, unit_root_pair(2u * c, 2u * (c + 1), ton, INV));     // (W_n^{2 n2})^{k'}
            if (h == 1) {
                const cp wh = unit_root_pair(c, c + 1, ton, INV);                        // W_n^{n2 h}
#pragma unroll
                for (int s = 0; s < 16; s++) v[s] = cmul(v[s], wh);
            }
        }
#pragma unroll
        for (int s = 0; s < 16; s++)
            *reinterpret_cast<float4*>(o + (size_t)N2 * (NH * r16_k(s) + h)) = make_float4(v[s].re.x, v[s].im.x, v[s].re.y, v[s].im.y);
    }
}

// NH = 2: 512-point columns, radix-2 step in front of the 256-point transform (two sweeps, see fftp_col16_kernel):
// y_h[m] = (x[m] + (-1)^h x[m + 256]) W_512^{m h}, X[2k' + h] = DFT256(y_h)[k'].  Not usable in place.
template <bool INV, bool SHIFT_IN, int NH, bool RIN = false, bool MUL = false>
__global__ void __launch_bounds__(128, 5) fftp_col256_kernel(const float2* __restrict__ x, float2* __restrict__ tmp,
                                                             const float4* __restrict__ tws, int log2n2, InMul im) {
    // n = 256 * NH * N2 points per sequence, N2 = 2^log2n2 = row length of the second pass
    const unsigned N2 = 1u << log2n2;
    const unsigned N = 256u * NH * N2;
    __shared__ __align__(16) float sre[16 * 272];
    __shared__ __align__(16) float sim[16 * 272];
    const int t = threadIdx.x;
    const unsigned tiles = N2 >> 4;                    // 16 columns per CTA
    const size_t seq = blockIdx.x / tiles;
    const unsigned c0 = (blockIdx.x % tiles) * 16u;
    const int hi = t >> 3, j = 2 * (t & 7);
    const float ton = 2.0f / (float)N;
#pragma unroll 1
    for (int h = 0; h < NH; h++) {
    cp v[16];
    {   // stage 1: radix 16 over m = 16a + b, b = hi
        const float2* xq = x + seq * N;
        const float2* xs = xq + c0 + j + (size_t)hi * N2;
        cp wb;
        if constexpr (NH == 2) wb = unit_root_pair((unsigned)hi, (unsigned)hi, 2.0f / 512.0f, INV);   // W_512^b (both lanes)
#pragma unroll
        for (int a = 0; a < 16; a++) {
            if constexpr (NH == 1) {
                const int src = SHIFT_IN ? (a ^ 8) : a;
                const float4 ab = col_ldpair<RIN, MUL>(x, xs + (size_t)src * (16 * (size_t)N2), im, xq);
                v[a].re = make_float2(ab.x, ab.z);
                v[a].im = make_float2(ab.y, ab.w);
            } else {
                const size_t r0 = (size_t)a * (16 * (size_t)N2), half = (size_t)256 * N2;
                const float4 lo = col_ldpair<RIN, MUL>(x, xs + r0 + (SHIFT_IN ? half : 0), im, xq);
                const float4 hh = col_ldpair<RIN, MUL>(x, xs + r0 + (SHIFT_IN ? 0 : half), im, xq);
                cp l, g;
                l.re = make_float2(lo.x, lo.z); l.im = make_float2(lo.y, lo.w);
                g.re = make_float2(hh.x, hh.z); g.im = make_float2(hh.y, hh.w);
                if (h == 0) v[a] = cadd(l, g);
                else {   // W_512^{16a + b} = W_32^a W_512^b
                    const cp d = cmulc(csub(l, g), splat(FP_C32[a]), splat(INV ? FP_S32[a] : -FP_S32[a]));
                    v[a] = cmul(d, wb);
                }
            }
        }
        r16<INV>(v);
        const int off = 16 * hi + ((j + 4 * rot_of(hi)) & 15);
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int ka = r16_k(s);
            if (s > 0) {
                const float4 f = __ldg(tws + 16 * ka + hi);
                cp w;
                w.re = make_float2(f.x, f.y);
                w.im = make_float2(f.z, f.w);
                v[s] = INV ? cmul_conj(v[s], w) : cmul(v[s], w);
            }
            *reinterpret_cast<float2*>(sre + 272 * ka + off) = v[s].re;
            *reinterpret_cast<float2*>(sim + 272 * ka + off) = v[s].im;
        }
    }
    __syncthreads();
    {   // stage 2: radix 16 over b for ka = hi; k' = ka + 16*kb, output row k1 = NH*k' + h
        const int ka = hi;
#pragma unroll
        for (int b = 0; b < 16; b++) {
            const int a = 272 * ka + 16 * b + ((j + 4 * rot_of(b)) & 15);
            v[b].re = *reinterpret_cast<const float2*>(sre + a);
            v[b].im = *reinterpret_cast<const float2*>(sim + a);
        }
        r16<INV>(v);
        // W_n^{n2*k1} = W_n^{n2*(NH*ka + h)} * (W_n^{16*NH*n2})^{kb}
        const unsigned n2 = c0 + (unsigned)j;
        const unsigned kl = (unsigned)(NH * ka + h);
        const cp w0 = unit_root_pair(n2 * kl, (n2 + 1) * kl, ton, INV);
        const cp u = unit_root_pair(16u * NH * n2, 16u * NH * (n2 + 1), ton, INV);
        cp A[4], B[4];
        A[0] = w0;
        A[1] = cmul(w0, u);
        A[2] = cmul(A[1], u);
        A[3] = cmul(A[2], u);
        const cp u2 = cmul(u, u);
        B[1] = cmul(u2, u2);
        B[2] = cmul(B[1], B[1]);
        B[3] = cmul(B[2], B[1]);
        float2* o = tmp + seq * N + (size_t)kl * N2 + c0 + j;
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int kb = r16_k(s);
            const cp w = (kb >> 2) == 0 ? A[kb & 3] : cmul(A[kb & 3], B[kb >> 2]);
            const cp r = cmul(v[s], w);
            *reinterpret_cast<float4*>(o + (size_t)kb * (16 * NH * (size_t)N2)) = make_float4(r.re.x, r.im.x, r.re.y, r.im.y);
        }
    }
    if (NH > 1) __syncthreads();   // the next sweep overwrites the shared tile
    }
}

// ------------------------------------------------------------------------------------------
namespace {
std::mutex g_fp_mu;
std::map<int, float*> g_fp_tw;
}  // namespace

const float* fftp_twiddles() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) { set_last_error("cudaGetDevice failed"); return nullptr; }
    std::lock_guard<std::mutex> lk(g_fp_mu);
    auto it = g_fp_tw.find(d);
    if (it != g_fp_tw.end()) return it->second;
    std::vector<float> h(FP_TW_FLOATS, 0.f);
    const long double tau = 2.0L * 3.14159265358979323846264338327950288L;
    for (int c = 0; c < 256; c++) {
        h[c] = (float)cosl(-tau * c / 4096.0L);
        h[256 + c] = (float)sinl(-tau * c / 4096.0L);
    }
    for (int k = 0; k < 16; k++)
        for (int n = 0; n < 16; n++) {
            const long double a = -tau * (long double)((k * n) % 256) / 256.0L;
            h[512 + (8 * k + n / 2) * 4 + (n & 1)] = (float)cosl(a);
            h[512 + (8 * k + n / 2) * 4 + 2 + (n & 1)] = (float)sinl(a);
        }
    for (int i = 0; i < 2; i++)
        for (int c = 0; c < 4096; c++) {
            const long double a = -tau * (long double)c / (long double)(8192 << i);
            h[1024 + 8192 * i + c] = (float)cosl(a);
            h[1024 + 8192 * i + 4096 + c] = (float)sinl(a);
        }
    for (int c = 0; c < 256; c++) {
        h[FP_TW_1K + c] = (float)cosl(-tau * c / 1024.0L);
        h[FP_TW_1K + 256 + c] = (float)sinl(-tau * c / 1024.0L);
        h[FP_TW_512 + c] = (float)cosl(-tau * c / 512.0L);
        h[FP_TW_512 + 256 + c] = (float)sinl(-tau * c / 512.0L);
        h[FP_TW_2K + c] = (float)cosl(-tau * c / 2048.0L);
        h[FP_TW_2K + 256 + c] = (float)sinl(-tau * c / 2048.0L);
    }
    for (int P = 4; P <= 8; P += 4)
        for (int kg = 0; kg < P; kg++)
            for (int j = 0; j < 16; j++) {
                const long double a = -tau * (long double)((kg * j) % (16 * P)) / (long double)(16 * P);
                float* e = &h[(P == 4 ? FP_TW_S4 : FP_TW_S8) + (8 * kg + j / 2) * 4];
                e[j & 1] = (float)cosl(a);
                e[2 + (j & 1)] = (float)sinl(a);
            }
    for (int ka = 0; ka < 16; ka++)
        for (int b = 0; b < 16; b++) {
            const long double a = -tau * (long double)((ka * b) % 256) / 256.0L;
            float* e = &h[FP_TW_SPLAT + 4 * (16 * ka + b)];
            e[0] = e[1] = (float)cosl(a);
            e[2] = e[3] = (float)sinl(a);
        }
    float* dev = nullptr;
    if (cudaMalloc(&dev, FP_TW_FLOATS * sizeof(float)) != cudaSuccess ||
        cudaMemcpy(dev, h.data(), FP_TW_FLOATS * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
        if (dev) cudaFree(dev);
        cudaGetLastError();
        set_last_error("fftp: twiddle table allocation failed");
        return nullptr;
    }
    g_fp_tw[d] = dev;
    return dev;
}

namespace {

// grid: CTAs that loop over the rows (0: one CTA per row); frames: fftp_kernel<PSUM>'s frame count
template <int R0, bool INV, bool SI, bool SO, bool MAG, bool ROWS = false, int TQ = 0, int NATQ = 0, bool RIN = false, int SQ = 0,
          bool FRAMES = false, bool PSUM = false>
int fftp_launch(const void* in, void* out, size_t rows, float scale, cudaStream_t st, int n1 = 1, int n2c = 1, size_t hop = 0,
                const float* win = nullptr, size_t frames = 0, size_t grid = 0) {
    const size_t smem = (size_t)2 * R0 * FP_B_OF(R0) * sizeof(float);
    auto kern = fftp_kernel<R0, INV, SI, SO, MAG, ROWS, TQ, NATQ, RIN, SQ, FRAMES, PSUM>;
    static PerDeviceOnce configured;   // per instantiation and device
    if (configured.need()) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured.mark();
    }
    const float* tw = fftp_twiddles();
    if (!tw) return -1001;
    kern<<<(unsigned)(grid ? grid : rows), 128 * R0, smem, st>>>(reinterpret_cast<const float2*>(in), out, (long long)rows, scale, tw, n1,
                                                                 n2c, (long long)hop, win, (long long)frames);
    BDSP_CUDA_OK(cudaGetLastError());
    BDSP_LAUNCHED();
    return 0;
}

template <bool INV, bool SI, bool RIN = false>
int fftp_colpass(const void* in, void* tmp, int n1, int log2n2, size_t rows, cudaStream_t st, const InMul& im) {
    const float* tw = fftp_twiddles();
    if (!tw) return -1001;
    const float2* i2 = reinterpret_cast<const float2*>(in);
    float2* t2 = reinterpret_cast<float2*>(tmp);
    const float4* tws = reinterpret_cast<const float4*>(tw + FP_TW_SPLAT);
    const unsigned g16 = (unsigned)(rows * ((size_t)1 << (log2n2 - 8))), g256 = (unsigned)(rows * ((size_t)1 << (log2n2 - 4)));
    if (im.kind == 1 || im.kind == 2) {
        if (n1 == 16) fftp_col16_kernel<INV, SI, 1, RIN, true><<<g16, 128, 0, st>>>(i2, t2, log2n2, im);
        else if (n1 == 32) fftp_col16_kernel<INV, SI, 2, RIN, true><<<g16, 128, 0, st>>>(i2, t2, log2n2, im);
        else if (n1 == 256) fftp_col256_kernel<INV, SI, 1, RIN, true><<<g256, 128, 0, st>>>(i2, t2, tws, log2n2, im);
        else fftp_col256_kernel<INV, SI, 2, RIN, true><<<g256, 128, 0, st>>>(i2, t2, tws, log2n2, im);
    } else if (im.kind) {
        set_last_error("fftp_colpass: multiplier kind %d must be materialised as a table", im.kind);
        return -2;
    } else {
        if (n1 == 16) fftp_col16_kernel<INV, SI, 1, RIN><<<g16, 128, 0, st>>>(i2, t2, log2n2, im);
        else if (n1 == 32) fftp_col16_kernel<INV, SI, 2, RIN><<<g16, 128, 0, st>>>(i2, t2, log2n2, im);
        else if (n1 == 256) fftp_col256_kernel<INV, SI, 1, RIN><<<g256, 128, 0, st>>>(i2, t2, tws, log2n2, im);
        else fftp_col256_kernel<INV, SI, 2, RIN><<<g256, 128, 0, st>>>(i2, t2, tws, log2n2, im);
    }
    BDSP_CUDA_OK(cudaGetLastError());
    BDSP_LAUNCHED();
    return 0;
}

// first pass of the multi-pass transforms; real input comes forward and unrotated only
int fftp_first_colpass(const void* in, void* tmp, int n1, int log2n2, size_t rows, bool inverse, bool si, bool real_in, const InMul& im,
                       cudaStream_t st) {
    if (real_in) return fftp_colpass<false, false, true>(in, tmp, n1, log2n2, rows, st, im);
    if (inverse) return si ? fftp_colpass<true, true>(in, tmp, n1, log2n2, rows, st, im) : fftp_colpass<true, false>(in, tmp, n1, log2n2, rows, st, im);
    return si ? fftp_colpass<false, true>(in, tmp, n1, log2n2, rows, st, im) : fftp_colpass<false, false>(in, tmp, n1, log2n2, rows, st, im);
}
}  // namespace

// Last pass of a multi-pass transform, stored at k1 + n1 * k2 (+ n1 * n2c * k3): tq = 0: four adjacent 4096-point rows per
// 512-thread CTA; tq = Q: 16/Q adjacent rows of 256*Q points per 128-thread CTA.  Also the packed 1024-point pass (tq = 4)
// behind the generic column pass of FftRoute::Hybrid, which left tmp[k1 * 1024 + n2] (column transform and inter-pass
// twiddle applied).
int fftp_rows_pass(const void* tmp, void* out, int tq, size_t groups, bool inverse, bool so, bool magnitude, float sc, cudaStream_t st,
                   int n1, int n2c) {
    return fftp_with_flags<true, false>(inverse, false, so, magnitude, [&](auto inv, auto si, auto sho, auto mag) {
        switch (tq) {
        case 0: return fftp_launch<4, inv, si, sho, mag, true>(tmp, out, groups, sc, st, n1, n2c);
        case 1: return fftp_launch<1, inv, si, sho, mag, true, 1>(tmp, out, groups, sc, st, n1, n2c);
        case 2: return fftp_launch<1, inv, si, sho, mag, true, 2>(tmp, out, groups, sc, st, n1, n2c);
        case 4: return fftp_launch<1, inv, si, sho, mag, true, 4>(tmp, out, groups, sc, st, n1, n2c);
        default: return fftp_launch<1, inv, si, sho, mag, true, 8>(tmp, out, groups, sc, st, n1, n2c);
        }
    });
}

// single pass over rows of n = 64 .. 16384 points (FftRoute::Packed); RIN: forward transforms of real scalars (FftRoute::RealRows)
template <bool RIN>
int fftp_single(const void* in, void* out, size_t n, size_t groups, bool inverse, bool si, bool so, bool magnitude, double scale,
                cudaStream_t st) {
    const float sc = (float)scale;
    return fftp_with_flags<!RIN, !RIN>(inverse, si, so, magnitude, [&](auto inv, auto shi, auto sho, auto mag) {
        switch (n) {
        case 64: return fftp_launch<1, inv, shi, sho, mag, false, 0, 1, RIN, 4>(in, out, groups, sc, st);
        case 128: return fftp_launch<1, inv, shi, sho, mag, false, 0, 1, RIN, 8>(in, out, groups, sc, st);
        case 256: return fftp_launch<1, inv, shi, sho, mag, false, 0, 1, RIN>(in, out, groups, sc, st);
        case 512: return fftp_launch<1, inv, shi, sho, mag, false, 0, 2, RIN>(in, out, groups, sc, st);
        case 1024: return fftp_launch<1, inv, shi, sho, mag, false, 0, 4, RIN>(in, out, groups, sc, st);
        case 2048: return fftp_launch<1, inv, shi, sho, mag, false, 0, 8, RIN>(in, out, groups, sc, st);
        case 4096: return fftp_launch<1, inv, shi, sho, mag, false, 0, 0, RIN>(in, out, groups, sc, st);
        case 8192: return fftp_launch<2, inv, shi, sho, mag, false, 0, 0, RIN>(in, out, groups, sc, st);
        default: return fftp_launch<4, inv, shi, sho, mag, false, 0, 0, RIN>(in, out, groups, sc, st);
        }
    });
}
template int fftp_single<false>(const void*, void*, size_t, size_t, bool, bool, bool, bool, double, cudaStream_t);
template int fftp_single<true>(const void*, void*, size_t, size_t, bool, bool, bool, bool, double, cudaStream_t);

// forward single pass over frames of n = 64 .. 8192 points that start `hop` points apart (FftRoute::PackedFrames), with an
// optional table of n real multipliers (the window) on the first load; RIN: the frames hold real scalars
template <bool RIN>
int fftp_frames(const void* in, void* out, size_t n, size_t groups, size_t hop, const float* win, bool so, bool magnitude, double scale,
                cudaStream_t st) {
    const float sc = (float)scale;
    return fftp_with_flags<false, false>(false, false, so, magnitude, [&](auto inv, auto shi, auto sho, auto mag) {
        switch (n) {
        case 64: return fftp_launch<1, inv, shi, sho, mag, false, 0, 1, RIN, 4, true>(in, out, groups, sc, st, 1, 1, hop, win);
        case 128: return fftp_launch<1, inv, shi, sho, mag, false, 0, 1, RIN, 8, true>(in, out, groups, sc, st, 1, 1, hop, win);
        case 256: return fftp_launch<1, inv, shi, sho, mag, false, 0, 1, RIN, 0, true>(in, out, groups, sc, st, 1, 1, hop, win);
        case 512: return fftp_launch<1, inv, shi, sho, mag, false, 0, 2, RIN, 0, true>(in, out, groups, sc, st, 1, 1, hop, win);
        case 1024: return fftp_launch<1, inv, shi, sho, mag, false, 0, 4, RIN, 0, true>(in, out, groups, sc, st, 1, 1, hop, win);
        case 2048: return fftp_launch<1, inv, shi, sho, mag, false, 0, 8, RIN, 0, true>(in, out, groups, sc, st, 1, 1, hop, win);
        case 4096: return fftp_launch<1, inv, shi, sho, mag, false, 0, 0, RIN, 0, true>(in, out, groups, sc, st, 1, 1, hop, win);
        default: return fftp_launch<2, inv, shi, sho, mag, false, 0, 0, RIN, 0, true>(in, out, groups, sc, st, 1, 1, hop, win);
        }
    });
}
template int fftp_frames<false>(const void*, void*, size_t, size_t, size_t, const float*, bool, bool, double, cudaStream_t);
template int fftp_frames<true>(const void*, void*, size_t, size_t, size_t, const float*, bool, bool, double, cudaStream_t);

// Welch power sums over frames of n = 64 .. 8192 points that start `hop` points apart (welch_route): `groups` groups of N / n
// frames (N = 4096, or 8192), the last one possibly incomplete; `ctas` CTAs each leave the sums of their groups' |X|^2 in
// part[cta * N + k], k < n.  win: n real multipliers on the first load, or null; RIN: the frames hold real scalars
template <bool RIN>
int fftp_frames_psum(const void* in, float* part, size_t n, size_t groups, size_t ctas, size_t hop, size_t frames, const float* win,
                     cudaStream_t st) {
    switch (n) {
    case 64: return fftp_launch<1, false, false, false, false, false, 0, 1, RIN, 4, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 128: return fftp_launch<1, false, false, false, false, false, 0, 1, RIN, 8, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 256: return fftp_launch<1, false, false, false, false, false, 0, 1, RIN, 0, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 512: return fftp_launch<1, false, false, false, false, false, 0, 2, RIN, 0, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 1024: return fftp_launch<1, false, false, false, false, false, 0, 4, RIN, 0, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 2048: return fftp_launch<1, false, false, false, false, false, 0, 8, RIN, 0, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 4096: return fftp_launch<1, false, false, false, false, false, 0, 0, RIN, 0, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    case 8192: return fftp_launch<2, false, false, false, false, false, 0, 0, RIN, 0, true, true>(in, part, groups, 1.f, st, 1, 1, hop, win, frames, ctas);
    default: set_last_error("fftp_frames_psum: no kernel for %zu points", n); return -2;
    }
}
template int fftp_frames_psum<false>(const void*, float*, size_t, size_t, size_t, size_t, size_t, const float*, cudaStream_t);
template int fftp_frames_psum<true>(const void*, float*, size_t, size_t, size_t, size_t, size_t, const float*, cudaStream_t);

// two-pass transform for n = 2^15 .. 2^20 (FftRoute::TwoPass), n = p.n1 * 2^p.log2n2; tmp holds n*rows complex values
int fftp_two_pass(const void* in, void* out, void* tmp, const FftPlan& p, size_t rows, bool inverse, bool si, bool so, bool magnitude,
                  double scale, bool real_in, const InMul& im, cudaStream_t st) {
    // One launch pair over the whole batch.  Measured on B200 (64 x 2^20): 0.448 ms, against 0.571 / 0.596 / 1.18 ms for
    // chunks of sequences whose intermediate (8 bytes per point) is 64 / 32 / 8 MB and could stay in the 126 MB L2 between
    // the passes: launch rate and wave tails cost more than the saved DRAM traffic.
    const int rc = fftp_first_colpass(in, tmp, p.n1, p.log2n2, rows, inverse, si, real_in, im, st);
    if (rc) return rc;
    // The 4096-point last pass takes four rows per 512-thread CTA (one CTA per SM, full 32-byte store sectors).  Measured on
    // B200 (64 x 2^20): 0.453 ms, against 0.494 ms with two rows per 256-thread CTA (16-byte half sectors, two CTAs per SM).
    const int tq = p.log2n2 < 12 ? 1 << (p.log2n2 - 8) : 0;
    return fftp_rows_pass(tmp, out, tq, p.groups, inverse, so, magnitude, (float)scale, st, p.n1, 1);
}

// three-pass transform for n = 2^21 .. 2^24 (FftRoute::ThreePass):  n = nA * 256 * N3 with nA = p.n1 in {16, 32, 256}:
//   pass A: nA-point columns over stride n/nA (+ W_n twiddle), pass B: 256-point columns inside every block of 256*N3
//   points (exactly the first pass of the two-pass transform of that length, in place), pass C: rows of N3 = 256*Q points,
//   16/Q rows with consecutive k1 per CTA, stored at k1 + nA*k2 + nA*256*k3.
int fftp_three_pass(const void* in, void* out, void* tmp, const FftPlan& p, size_t n, size_t rows, bool inverse, bool si, bool so,
                    bool magnitude, double scale, bool real_in, const InMul& im, cudaStream_t st) {
    int l2 = 0;
    while (((size_t)p.n1 << l2) < n) l2++;                 // n / nA = 2^l2
    int rc = fftp_first_colpass(in, tmp, p.n1, l2, rows, inverse, si, real_in, im, st);
    if (rc) return rc;
    rc = fftp_first_colpass(tmp, tmp, 256, p.log2n3, rows * (size_t)p.n1, inverse, false, false, InMul(), st);
    if (rc) return rc;
    return fftp_rows_pass(tmp, out, 1 << (p.log2n3 - 8), p.groups, inverse, so, magnitude, (float)scale, st, p.n1, 256);
}

}  // namespace bdsp
