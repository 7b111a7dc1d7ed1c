// Reductions of the reference's C facade (SURVEY 8f row 4): sum / sum_sq (statistics.rs:98-131,
// 440-560), dot_product (dot_products.rs:67-160), statistics / statistics_split (statistics.rs:179-440)
// and their `_prec` twins (precise_stats.rs: f32 data accumulated in f64, f64 data with Kahan summation).
//
// One pass over HBM: every thread keeps its partial record in registers (double accumulators; Kahan
// compensation for f64 `_prec`), blocks tree-reduce in shared memory, a second one-block kernel folds
// the per-block records.  Minimum / maximum keep the FIRST index of the extreme value (the reference's
// strict comparisons on one chunk); complex values are ordered by their norm computed in T.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <map>
#include <mutex>

#include "common.cuh"
#include "mathops.cuh"

namespace bdsp {
void* workspace(size_t bytes, int slot);

namespace {

struct Rec {
    double s[4], c[4];
    double mn[2], mx[2], mnn, mxn;
    unsigned long long mni, mxi, cnt;
};

__device__ __forceinline__ void rec_init(Rec& r, bool cplx) {
#pragma unroll
    for (int k = 0; k < 4; k++) { r.s[k] = 0.0; r.c[k] = 0.0; }
    r.mn[0] = CUDART_INF; r.mn[1] = cplx ? CUDART_INF : 0.0; r.mnn = CUDART_INF;
    r.mx[0] = cplx ? 0.0 : -CUDART_INF; r.mx[1] = 0.0; r.mxn = cplx ? 0.0 : -CUDART_INF;
    r.mni = r.mxi = r.cnt = 0;
}

template <bool PREC> __device__ __forceinline__ void kadd(double& s, double& c, double v) {
    if (PREC) {   // Kahan: c carries the rounding error of the running sum
        const double y = __dsub_rn(v, c);
        const double t = __dadd_rn(s, y);
        c = __dsub_rn(__dsub_rn(t, s), y);
        s = t;
    } else {
        s = __dadd_rn(s, v);
    }
}

template <bool PREC> __device__ __forceinline__ void rec_merge(Rec& a, const Rec& b) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
        kadd<PREC>(a.s[k], a.c[k], b.s[k]);
        if (PREC) kadd<PREC>(a.s[k], a.c[k], -b.c[k]);
    }
    if (b.cnt) {
        if (b.mnn < a.mnn || (b.mnn == a.mnn && b.mni < a.mni) || !a.cnt) { a.mn[0] = b.mn[0]; a.mn[1] = b.mn[1]; a.mnn = b.mnn; a.mni = b.mni; }
        if (b.mxn > a.mxn || (b.mxn == a.mxn && b.mxi < a.mxi) || !a.cnt) { a.mx[0] = b.mx[0]; a.mx[1] = b.mx[1]; a.mxn = b.mxn; a.mxi = b.mxi; }
    }
    a.cnt += b.cnt;
}

enum { R_SUMS = 0, R_DOT = 1, R_STATS = 2 };

// ordering key of complex values: the squared norm in double (exact products for f32 data).  The reference orders
// by norm() rounded to T; the two orders differ only between values whose norms round to the same T.
__device__ __forceinline__ double norm_key(double re, double im) { return fma(re, re, im * im); }

// one element: real (re; bre for the dot product) or complex (re, im; bre, bim)
template <typename T, int MODE, bool PREC>
__device__ __forceinline__ void rec_add(Rec& r, T tre, T tim, T tbre, T tbim, unsigned long long index, bool cplx) {
    if (!cplx) {
        const double v = (double)tre;
        if (MODE == R_DOT) { kadd<PREC>(r.s[0], r.c[0], __dmul_rn(v, (double)tbre)); return; }
        kadd<PREC>(r.s[0], r.c[0], v);
        kadd<PREC>(r.s[2], r.c[2], __dmul_rn(v, v));
        if (MODE == R_STATS) {
            if (v > r.mxn) { r.mxn = v; r.mx[0] = v; r.mxi = index; }
            if (v < r.mnn) { r.mnn = v; r.mn[0] = v; r.mni = index; }
            r.cnt++;
        }
    } else {
        const double re = (double)tre, im = (double)tim;
        if (MODE == R_DOT) {
            const double bre = (double)tbre, bim = (double)tbim;
            kadd<PREC>(r.s[0], r.c[0], __dsub_rn(__dmul_rn(re, bre), __dmul_rn(im, bim)));
            kadd<PREC>(r.s[1], r.c[1], __dadd_rn(__dmul_rn(re, bim), __dmul_rn(im, bre)));
            return;
        }
        kadd<PREC>(r.s[0], r.c[0], re);
        kadd<PREC>(r.s[1], r.c[1], im);
        kadd<PREC>(r.s[2], r.c[2], __dsub_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
        kadd<PREC>(r.s[3], r.c[3], __dadd_rn(__dmul_rn(re, im), __dmul_rn(im, re)));
        if (MODE == R_STATS) {
            const double nn = norm_key(re, im);
            if (nn > r.mxn) { r.mxn = nn; r.mx[0] = re; r.mx[1] = im; r.mxi = index; }
            if (nn < r.mnn) { r.mnn = nn; r.mn[0] = re; r.mn[1] = im; r.mni = index; }
            r.cnt++;
        }
    }
}
template <typename T, int MODE, bool PREC>
__device__ __forceinline__ void rec_add_at(Rec& r, const T* __restrict__ a, const T* __restrict__ b, long long j, unsigned long long index, bool cplx) {
    if (!cplx) rec_add<T, MODE, PREC>(r, a[j], (T)0, MODE == R_DOT ? b[j] : (T)0, (T)0, index, false);
    else rec_add<T, MODE, PREC>(r, a[2 * j], a[2 * j + 1], MODE == R_DOT ? b[2 * j] : (T)0, MODE == R_DOT ? b[2 * j + 1] : (T)0, index, true);
}

template <typename T> struct alignas(16) Pack { T v[16 / sizeof(T)]; };

constexpr int RT = 256;

template <bool PREC> __device__ __forceinline__ void block_fold(Rec& r, Rec* sh) {
    sh[threadIdx.x] = r;
    __syncthreads();
    for (int off = RT / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off) rec_merge<PREC>(sh[threadIdx.x], sh[threadIdx.x + off]);
        __syncthreads();
    }
}

// grid (blocks, parts): row `part` reduces elements j = part + parts * m
template <typename T, int MODE, bool PREC>
__global__ void __launch_bounds__(RT) reduce_kernel(const T* __restrict__ a, const T* __restrict__ b, long long elems, int cplx, Rec* __restrict__ partial) {
    extern __shared__ __align__(16) unsigned char shraw[];
    Rec* sh = reinterpret_cast<Rec*>(shraw);
    const int part = blockIdx.y, parts = gridDim.y;
    const long long count = elems > part ? (elems - part + parts - 1) / parts : 0;
    Rec r;
    rec_init(r, cplx != 0);
    const long long stride = (long long)gridDim.x * RT;
    const long long tid = (long long)blockIdx.x * RT + threadIdx.x;
    if (parts == 1) {
        // 16-byte loads: SC scalars = W elements per thread and step; indices stay increasing within a thread
        constexpr int SC = 16 / sizeof(T);
        const int W = cplx ? SC / 2 : SC;
        const long long nv = count / W;
        const Pack<T>* av = reinterpret_cast<const Pack<T>*>(a);
        const Pack<T>* bv = reinterpret_cast<const Pack<T>*>(b);
        if (MODE == R_STATS) {
            // Per element only the ordering key and a 32-bit code (step * W + slot) are kept for the extremes; values and
            // 64-bit indices are reconstructed after the loop.  Strict comparisons in increasing index order keep the
            // first occurrence.
            constexpr unsigned NONE = 0xffffffffu;
            unsigned mxc = NONE, mnc = NONE, it = 0;
            if (!cplx) {
                T mxk = -(T)CUDART_INF, mnk = (T)CUDART_INF;
                for (long long m = tid; m < nv; m += stride, it++) {
                    const Pack<T> pa = av[m];
#pragma unroll
                    for (int k = 0; k < SC; k++) {
                        const T x = pa.v[k];
                        const double v = (double)x;
                        kadd<PREC>(r.s[0], r.c[0], v);
                        kadd<PREC>(r.s[2], r.c[2], __dmul_rn(v, v));
                        const unsigned code = it * SC + k;
                        if (x > mxk) { mxk = x; mxc = code; }
                        if (x < mnk) { mnk = x; mnc = code; }
                    }
                    r.cnt += SC;
                }
                if (mxc != NONE) { r.mxn = r.mx[0] = (double)mxk; r.mxi = (unsigned long long)((tid + (long long)(mxc / SC) * stride) * SC + mxc % SC); }
                if (mnc != NONE) { r.mnn = r.mn[0] = (double)mnk; r.mni = (unsigned long long)((tid + (long long)(mnc / SC) * stride) * SC + mnc % SC); }
            } else {
                constexpr int WC = SC / 2 > 0 ? SC / 2 : 1;
                double mxk = 0.0, mnk = CUDART_INF;
                for (long long m = tid; m < nv; m += stride, it++) {
                    const Pack<T> pa = av[m];
#pragma unroll
                    for (int k = 0; k < WC; k++) {
                        const double re = (double)pa.v[2 * k], im = (double)pa.v[2 * k + 1];
                        kadd<PREC>(r.s[0], r.c[0], re);
                        kadd<PREC>(r.s[1], r.c[1], im);
                        kadd<PREC>(r.s[2], r.c[2], __dsub_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
                        kadd<PREC>(r.s[3], r.c[3], __dadd_rn(__dmul_rn(re, im), __dmul_rn(im, re)));
                        const double nn = norm_key(re, im);
                        const unsigned code = it * WC + k;
                        if (nn > mxk) { mxk = nn; mxc = code; }
                        if (nn < mnk) { mnk = nn; mnc = code; }
                    }
                    r.cnt += WC;
                }
                if (mxc != NONE) {
                    const long long j = (tid + (long long)(mxc / WC) * stride) * WC + mxc % WC;
                    r.mxn = mxk; r.mx[0] = (double)a[2 * j]; r.mx[1] = (double)a[2 * j + 1]; r.mxi = (unsigned long long)j;
                }
                if (mnc != NONE) {
                    const long long j = (tid + (long long)(mnc / WC) * stride) * WC + mnc % WC;
                    r.mnn = mnk; r.mn[0] = (double)a[2 * j]; r.mn[1] = (double)a[2 * j + 1]; r.mni = (unsigned long long)j;
                }
            }
        } else
        for (long long m = tid; m < nv; m += stride) {
            const Pack<T> pa = av[m];
            Pack<T> pb = pa;
            if (MODE == R_DOT) pb = bv[m];
            if (!cplx) {
#pragma unroll
                for (int k = 0; k < SC; k++) rec_add<T, MODE, PREC>(r, pa.v[k], (T)0, pb.v[k], (T)0, (unsigned long long)(m * SC + k), false);
            } else {
#pragma unroll
                for (int k = 0; k < SC / 2; k++)
                    rec_add<T, MODE, PREC>(r, pa.v[2 * k], pa.v[2 * k + 1], pb.v[2 * k], pb.v[2 * k + 1], (unsigned long long)(m * (SC / 2) + k), true);
            }
        }
        if (tid == 0)
            for (long long j = nv * W; j < count; j++) rec_add_at<T, MODE, PREC>(r, a, b, j, (unsigned long long)j, cplx != 0);
    } else {
        for (long long m = tid; m < count; m += stride)
            rec_add_at<T, MODE, PREC>(r, a, b, part + parts * m, (unsigned long long)m, cplx != 0);
    }
    block_fold<PREC>(r, sh);
    if (threadIdx.x == 0) partial[(long long)part * gridDim.x + blockIdx.x] = sh[0];
}

template <bool PREC>
__global__ void __launch_bounds__(RT) fold_kernel(const Rec* __restrict__ partial, int nblocks, int cplx, Rec* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char shraw[];
    Rec* sh = reinterpret_cast<Rec*>(shraw);
    const int part = blockIdx.x;
    Rec r;
    rec_init(r, cplx != 0);
    // block-contiguous assignment keeps the index order (thread t folds blocks [t*per, (t+1)*per))
    const int per = (nblocks + RT - 1) / RT;
    for (int k = 0; k < per; k++) {
        const int bidx = threadIdx.x * per + k;
        if (bidx < nblocks) rec_merge<PREC>(r, partial[(long long)part * nblocks + bidx]);
    }
    block_fold<PREC>(r, sh);
    if (threadIdx.x == 0) out[part] = sh[0];
}

template <typename T, int MODE, bool PREC>
int run_reduce(const void* a, const void* b, size_t elems, int cplx, int parts, Rec* host, cudaStream_t st) {
    long long blocks = ((long long)(elems / (size_t)parts) + RT * 8 - 1) / (RT * 8);
    const long long cap = (long long)sm_count() * 8 / parts + 1;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    Rec* dev = reinterpret_cast<Rec*>(workspace(sizeof(Rec) * (size_t)(blocks * parts + parts), 3));
    if (!dev) return -1001;
    Rec* dev_out = dev + blocks * parts;
    const size_t shm = sizeof(Rec) * RT;
    static PerDeviceOnce configured;   // per instantiation and device
    if (configured.need()) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(reduce_kernel<T, MODE, PREC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
        BDSP_CUDA_OK(cudaFuncSetAttribute(fold_kernel<PREC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
        configured.mark();
    }
    reduce_kernel<T, MODE, PREC><<<dim3((unsigned)blocks, (unsigned)parts), RT, shm, st>>>(reinterpret_cast<const T*>(a), reinterpret_cast<const T*>(b),
                                                                                        (long long)elems, cplx, dev);
    BDSP_LAUNCHED();
    fold_kernel<PREC><<<(unsigned)parts, RT, shm, st>>>(dev, (int)blocks, cplx, dev_out);
    BDSP_LAUNCHED();
    BDSP_CUDA_OK(cudaMemcpyAsync(host, dev_out, sizeof(Rec) * (size_t)parts, cudaMemcpyDeviceToHost, st));
    BDSP_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

template <typename T, int MODE>
int run_reduce_p(const void* a, const void* b, size_t elems, int cplx, int parts, int prec, Rec* host, cudaStream_t st) {
    // Kahan only where the reference uses it: f64 data with the `_prec` entry points
    if (prec && sizeof(T) == 8) return run_reduce<T, MODE, true>(a, b, elems, cplx, parts, host, st);
    return run_reduce<T, MODE, false>(a, b, elems, cplx, parts, host, st);
}

}  // namespace

template <typename T>
int reduce_sums(const void* data, size_t elems, int is_complex, int prec, double* out4, cudaStream_t st) {
    Rec r;
    int rc = run_reduce_p<T, R_SUMS>(data, nullptr, elems, is_complex, 1, prec, &r, st);
    if (rc) return rc;
    for (int k = 0; k < 4; k++) out4[k] = r.s[k];
    return 0;
}

template <typename T>
int reduce_dot(const void* a, const void* b, size_t elems, int is_complex, int prec, double* out2, cudaStream_t st) {
    Rec r;
    int rc = run_reduce_p<T, R_DOT>(a, b, elems, is_complex, 1, prec, &r, st);
    if (rc) return rc;
    out2[0] = r.s[0];
    out2[1] = r.s[1];
    return 0;
}

template <typename T>
int reduce_stats(const void* data, size_t elems, int is_complex, int parts, int prec, StatsRaw* out, cudaStream_t st) {
    if (parts < 1 || parts > 16) return 7;
    Rec r[16];
    int rc = run_reduce_p<T, R_STATS>(data, nullptr, elems, is_complex, parts, prec, r, st);
    if (rc) return rc;
    for (int p = 0; p < parts; p++) {
        out[p].sum[0] = r[p].s[0]; out[p].sum[1] = r[p].s[1];
        out[p].sumsq[0] = r[p].s[2]; out[p].sumsq[1] = r[p].s[3];
        out[p].min[0] = r[p].mn[0]; out[p].min[1] = r[p].mn[1];
        out[p].max[0] = r[p].mx[0]; out[p].max[1] = r[p].mx[1];
        out[p].min_index = r[p].mni; out[p].max_index = r[p].mxi; out[p].count = r[p].cnt;
    }
    return 0;
}

#define BDSP_INST(T)                                                                         \
    template int reduce_sums<T>(const void*, size_t, int, int, double*, cudaStream_t);       \
    template int reduce_dot<T>(const void*, const void*, size_t, int, int, double*, cudaStream_t); \
    template int reduce_stats<T>(const void*, size_t, int, int, int, StatsRaw*, cudaStream_t);
BDSP_INST(float)
BDSP_INST(double)
#undef BDSP_INST

}  // namespace bdsp
