// Planar packed-FP32x2 building blocks of the fftp* kernels (fftp.cu, fftp16k.cu).
// Written for sm_100a: all butterfly arithmetic uses the packed FP32x2 instructions of Blackwell
// (FADD2 / FMUL2 / FFMA2 via __fadd2_rn / __fmul2_rn / __ffma2_rn), which halve the issue slots per
// flop; data are planar (re plane, im plane) so that one 64-bit register pair holds the same
// component of two adjacent points ("two columns per thread").
// (The file is named after round 1's planar 4096-point overlap-save kernel, for which these pieces were written.)
#pragma once
#include "common.cuh"

namespace bdsp {
namespace ols16 {

typedef float2 pk;
struct cp { pk re, im; };

__device__ __forceinline__ pk padd(pk a, pk b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ pk pneg(pk a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ pk psub(pk a, pk b) { return __fadd2_rn(a, pneg(b)); }
__device__ __forceinline__ pk pmul(pk a, pk b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ pk pfma(pk a, pk b, pk c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ pk splat(float v) { return make_float2(v, v); }
// sqrt with a maximum relative error of 2^-23 (MUFU.SQRT; the IEEE sqrtf costs ~10 instructions and a slow-path call):
// used by the fused magnitude epilogues, whose tolerance is the transform's (1e-5 * log2 N relative L2)
__device__ __forceinline__ float sqrt_fast(float v) { float r; asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
// {re0, im0, re1, im1} (two adjacent interleaved points) -> planar pairs {re0, re1}, {im0, im1}; the explicit 64-bit packs
// keep the compiler from materialising each pair twice (once per consumer)
__device__ __forceinline__ void planar_of(const float4& ab, pk& re, pk& im) {
    unsigned long long r, i;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(ab.x), "f"(ab.z));
    asm("mov.b64 %0, {%1, %2};" : "=l"(i) : "f"(ab.y), "f"(ab.w));
    re = *reinterpret_cast<pk*>(&r);
    im = *reinterpret_cast<pk*>(&i);
}

__device__ __forceinline__ cp cadd(cp a, cp b) { cp r; r.re = padd(a.re, b.re); r.im = padd(a.im, b.im); return r; }
__device__ __forceinline__ cp csub(cp a, cp b) { cp r; r.re = psub(a.re, b.re); r.im = psub(a.im, b.im); return r; }
// a * w
__device__ __forceinline__ cp cmul(cp a, cp w) {
    cp r;
    r.re = pfma(a.re, w.re, pneg(pmul(a.im, w.im)));
    r.im = pfma(a.re, w.im, pmul(a.im, w.re));
    return r;
}
// a * conj(w)
__device__ __forceinline__ cp cmul_conj(cp a, cp w) {
    cp r;
    r.re = pfma(a.re, w.re, pmul(a.im, w.im));
    r.im = pfma(a.im, w.re, pneg(pmul(a.re, w.im)));
    return r;
}
// a * (wr + i*wi) with per-lane constants
__device__ __forceinline__ cp cmulc(cp a, pk wr, pk wi) {
    cp r;
    r.re = pfma(a.re, wr, pneg(pmul(a.im, wi)));
    r.im = pfma(a.re, wi, pmul(a.im, wr));
    return r;
}

// radix-4 butterfly, results in natural order (a_k = sum_j a_j * exp(-+2 pi i j k / 4))
template <bool INV> __device__ __forceinline__ void r4(cp& a0, cp& a1, cp& a2, cp& a3) {
    cp s0 = cadd(a0, a2), d0 = csub(a0, a2), s1 = cadd(a1, a3), d1 = csub(a1, a3);
    a0 = cadd(s0, s1);
    a2 = csub(s0, s1);
    if (!INV) {  // a1 = d0 - i d1, a3 = d0 + i d1
        a1.re = padd(d0.re, d1.im); a1.im = psub(d0.im, d1.re);
        a3.re = psub(d0.re, d1.im); a3.im = padd(d0.im, d1.re);
    } else {     // a1 = d0 + i d1, a3 = d0 - i d1
        a1.re = psub(d0.re, d1.im); a1.im = padd(d0.im, d1.re);
        a3.re = padd(d0.re, d1.im); a3.im = psub(d0.im, d1.re);
    }
}

#define OLS_C1 0.92387953251128675613f
#define OLS_S1 0.38268343236508977173f
#define OLS_H 0.70710678118654752440f

// v *= exp(-+2 pi i m / 16)  (same constant in both lanes)
template <int MM, bool INV> __device__ __forceinline__ cp mul_w16(cp v) {
    constexpr int m = MM & 15;
    if constexpr (m == 0) return v;
    else if constexpr (m == 4) { cp r; if (!INV) { r.re = v.im; r.im = pneg(v.re); } else { r.re = pneg(v.im); r.im = v.re; } return r; }
    else if constexpr (m == 8) { cp r; r.re = pneg(v.re); r.im = pneg(v.im); return r; }
    else if constexpr (m == 12) { cp r; if (!INV) { r.re = pneg(v.im); r.im = v.re; } else { r.re = v.im; r.im = pneg(v.re); } return r; }
    else {
        // cos/sin(m*pi/8)
        constexpr float cs[16] = {1.f, OLS_C1, OLS_H, OLS_S1, 0.f, -OLS_S1, -OLS_H, -OLS_C1, -1.f, -OLS_C1, -OLS_H, -OLS_S1, 0.f, OLS_S1, OLS_H, OLS_C1};
        constexpr float sn[16] = {0.f, OLS_S1, OLS_H, OLS_C1, 1.f, OLS_C1, OLS_H, OLS_S1, 0.f, -OLS_S1, -OLS_H, -OLS_C1, -1.f, -OLS_C1, -OLS_H, -OLS_S1};
        const float wr = cs[m];
        const float wi = INV ? sn[m] : -sn[m];
        return cmulc(v, splat(wr), splat(wi));
    }
}

// 16-point transform of v[j] (j natural).  On return slot s holds frequency k(s) = (s >> 2) + 4 * (s & 3).
__device__ __forceinline__ constexpr int r16_k(int s) { return (s >> 2) + 4 * (s & 3); }

template <bool INV> __device__ __forceinline__ void r16(cp (&v)[16]) {
#pragma unroll
    for (int j0 = 0; j0 < 4; j0++) r4<INV>(v[j0], v[4 + j0], v[8 + j0], v[12 + j0]);
    // twiddle W16^{j0*k1} on slot 4*k1 + j0
    v[5] = mul_w16<1, INV>(v[5]);  v[6] = mul_w16<2, INV>(v[6]);   v[7] = mul_w16<3, INV>(v[7]);
    v[9] = mul_w16<2, INV>(v[9]);  v[10] = mul_w16<4, INV>(v[10]); v[11] = mul_w16<6, INV>(v[11]);
    v[13] = mul_w16<3, INV>(v[13]); v[14] = mul_w16<6, INV>(v[14]); v[15] = mul_w16<9, INV>(v[15]);
#pragma unroll
    for (int k1 = 0; k1 < 4; k1++) r4<INV>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
}

// multiply v[slot] by w1^{k(slot)} where k(slot) = SLOTMAP ? r16_k(slot) : slot
// (powers built as A_a * B_b, k = a + 4b: 14 complex products, depth <= 4)
template <bool SLOTMAP> __device__ __forceinline__ void apply_twiddles(cp (&v)[16], cp w1) {
    cp A[4], B[4];
    A[1] = w1;
    A[2] = cmul(w1, w1);
    A[3] = cmul(A[2], w1);
    B[1] = cmul(A[2], A[2]);
    B[2] = cmul(B[1], B[1]);
    B[3] = cmul(B[2], B[1]);
#pragma unroll
    for (int s = 1; s < 16; s++) {
        const int k = SLOTMAP ? r16_k(s) : s;
        const int a = k & 3, b = k >> 2;
        cp w;
        if (b == 0) w = A[a];
        else if (a == 0) w = B[b];
        else w = cmul(A[a], B[b]);
        v[s] = cmul(v[s], w);
    }
}

// swizzled shared-memory layout of a 16 x 256-point tile: point 16*g + j of row k0 lives at
// 272*k0 + 16*g + ((j + 4*rot_of(g)) & 15), which keeps the row- and column-wise accesses free of bank conflicts
__device__ __forceinline__ int rot_of(int g) { return (g >> 1) & 3; }

// ---- in-register 16-point transforms over 16 CONTIGUOUS points, packed over adjacent points ------
// P[m] = {a[2m], a[2m+1]}.  DIF, natural in -> bit-reversed out; INV selects exp(+i...).
template <bool INV> __device__ __forceinline__ void fft16_dif(cp (&P)[8]) {
    const float sg = INV ? -1.f : 1.f;   // sign applied to the imaginary parts of the forward roots
    // level 1, span 8: twiddle W16^{j}, j = 2m, 2m+1
    const pk t1r[4] = {make_float2(1.f, OLS_C1), make_float2(OLS_H, OLS_S1), make_float2(0.f, -OLS_S1), make_float2(-OLS_H, -OLS_C1)};
    const pk t1i[4] = {make_float2(0.f, -sg * OLS_S1), make_float2(-sg * OLS_H, -sg * OLS_C1), make_float2(-sg, -sg * OLS_C1), make_float2(-sg * OLS_H, -sg * OLS_S1)};
#pragma unroll
    for (int m = 0; m < 4; m++) {
        cp u = cadd(P[m], P[m + 4]);
        cp d = csub(P[m], P[m + 4]);
        P[m] = u;
        P[m + 4] = cmulc(d, t1r[m], t1i[m]);
    }
    // level 2, span 4: twiddle W8^{j}, j = 2m, 2m+1
    const pk t2r[2] = {make_float2(1.f, OLS_H), make_float2(0.f, -OLS_H)};
    const pk t2i[2] = {make_float2(0.f, -sg * OLS_H), make_float2(-sg, -sg * OLS_H)};
#pragma unroll
    for (int b = 0; b < 8; b += 4) {
#pragma unroll
        for (int m = 0; m < 2; m++) {
            cp u = cadd(P[b + m], P[b + m + 2]);
            cp d = csub(P[b + m], P[b + m + 2]);
            P[b + m] = u;
            P[b + m + 2] = cmulc(d, t2r[m], t2i[m]);
        }
    }
    // level 3, span 2 (twiddle {1, -+i} of the difference deferred into level 4) and level 4, span 1
#pragma unroll
    for (int b = 0; b < 8; b += 2) {
        cp u = cadd(P[b], P[b + 1]);
        cp d = csub(P[b], P[b + 1]);
        cp o;
        o.re = make_float2(u.re.x + u.re.y, u.re.x - u.re.y);
        o.im = make_float2(u.im.x + u.im.y, u.im.x - u.im.y);
        P[b] = o;
        if (!INV) {   // lane y carries the deferred -i: y' = (y.im, -y.re)
            o.re = make_float2(d.re.x + d.im.y, d.re.x - d.im.y);
            o.im = make_float2(d.im.x - d.re.y, d.im.x + d.re.y);
        } else {      // +i: y' = (-y.im, y.re)
            o.re = make_float2(d.re.x - d.im.y, d.re.x + d.im.y);
            o.im = make_float2(d.im.x + d.re.y, d.im.x - d.re.y);
        }
        P[b + 1] = o;
    }
}

// bit reversal of a 4-bit index (host + device)
__host__ __device__ __forceinline__ int bitrev4(int j) { return ((j & 1) << 3) | ((j & 2) << 1) | ((j & 4) >> 1) | ((j & 8) >> 3); }

}  // namespace ols16
}  // namespace bdsp
