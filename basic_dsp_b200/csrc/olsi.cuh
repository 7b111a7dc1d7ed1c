// Pieces shared by the fused overlap-save kernels on interleaved-complex FP32x2 arithmetic (ols4096i.cu, ols8192i.cu).
#pragma once
#include "cxmath.cuh"

namespace bdsp {
using namespace cx;

// two adjacent block inputs as one 128-bit read-only load
__device__ __forceinline__ float4 ld_x4(const float2* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// --- bulk asynchronous copies between global and shared memory, mbarrier completion (shared addresses as u32) ------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// one arrival that also announces `bytes` of copies completing on the barrier's current phase
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned done;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
// bytes: multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// orders this thread's earlier generic-proxy accesses to shared memory before later async-proxy (bulk copy) accesses
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// shared -> global bulk copy (same rules as bulk_g2s); returns once the copy has READ its shared-memory source, so the
// buffer may be reused or the CTA may exit
__device__ __forceinline__ void bulk_s2g_wait_read(void* dst, unsigned src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// stride-16 stage twiddles W256^{k c}, k = 1..15: six 128-bit table loads (k = 1, 2, 3, 4, 8, 12) and nine products.
// Fifteen loads per stage (4-5 L1 wavefronts each) were 16 % of the kernel's L1 data-pipe traffic, which is its saturated
// unit.
// v[s] *= W^{k(s)} (CONJ: conjugated), k(s) = SLOTMAP ? r16_k(s) : s, for the two columns held in v / u
// tw2[STRIDE * k]: float4 = W^{k c}, W^{k (c + 1)} of the thread's two columns
template <bool SLOTMAP, bool CONJ, int STRIDE>
__device__ __forceinline__ void oi_tw2(c2 (&v)[16], c2 (&u)[16], const float4* __restrict__ tw2) {
    c2 Av[4], Bv[4], Au[4], Bu[4];
#pragma unroll
    for (int i = 1; i < 4; i++) {
        const float4 fa = __ldg(tw2 + STRIDE * i), fb = __ldg(tw2 + STRIDE * 4 * i);
        Av[i] = make_float2(fa.x, CONJ ? -fa.y : fa.y); Au[i] = make_float2(fa.z, CONJ ? -fa.w : fa.w);
        Bv[i] = make_float2(fb.x, CONJ ? -fb.y : fb.y); Bu[i] = make_float2(fb.z, CONJ ? -fb.w : fb.w);
    }
#pragma unroll
    for (int s = 1; s < 16; s++) {
        const int k = SLOTMAP ? r16_k(s) : s;
        const int a = k & 3, b = k >> 2;
        const c2 wv = b == 0 ? Av[a] : a == 0 ? Bv[b] : mul(Av[a], Bv[b]);
        const c2 wu = b == 0 ? Au[a] : a == 0 ? Bu[b] : mul(Au[a], Bu[b]);
        v[s] = mul(v[s], wv);
        u[s] = mul(u[s], wu);
    }
}

// plan geometry shared by prepare and convolve (block length M): the delay d in {0, 1} samples that the plan folds
// into H makes the distance `shift` between a block position's input index and its output index even, so that with even
// block offsets every thread moves its two adjacent points with one 128-bit access on both sides.
// m_first: first block position whose circular-convolution value is valid; step: outputs per block.
static inline void olsi_geometry(size_t M, size_t L, int* d, int* shift, int* m_first, int* step) {
    const int cl = (int)(L - L / 2);
    *d = (cl - 1) & 1;
    *shift = cl - 1 + *d;
    int mf = (int)L - 1 + *d;
    if (mf & 1) mf++;
    *m_first = mf;
    *step = ((int)M - mf) & ~1;
}

// the M-point kernel takes N-point vectors and L taps: at most one wrap per strided load, 32-bit row indices
static inline bool olsi_applicable(size_t M, size_t N, size_t L) { return L >= 2 && L <= M / 2 - 2 && N >= M && N < (1ull << 30); }

// blocks per vector (L must be applicable: the step is only positive then)
static inline long long olsi_blocks(size_t M, size_t N, size_t L) {
    int d, shift, m_first, step;
    olsi_geometry(M, L, &d, &shift, &m_first, &step);
    return ((long long)N + step - 1) / step;
}

// twiddle table of the M-point kernel (M = 4096, 8192), built once per device and M (float2):
// [0, M/16) W_M^c; [M/16 + (M/256) k + c] W_{M/16}^{k c}, k < 16, c < M/256.  nullptr (last error set) on failure.
const float2* olsi_twiddles(int M);

}  // namespace bdsp
