// Single-launch 65536-point c32 transform on a 16-CTA thread-block cluster (BASELINE config C1: one 2^16-point vector,
// fft -> ifft): the transposition between the two passes of the four-step algorithm goes through distributed shared
// memory instead of through HBM and a second kernel launch.
//
// The two-kernel path (fftp_col256_kernel + fftp_kernel<TQ>) costs two launches of 16 CTAs per transform; for a single
// vector the time is launch latency and the dependent start-up of the second kernel, not bandwidth (0.3 us of HBM
// time in 6.8 us per kernel).  Here: n = 256 x 256, x[256 n1 + n2]:
//   step 1  CTA c owns columns n2 = 16c .. 16c+15: 256-point transforms over n1 (radix 16 x 16, one local exchange),
//           twiddle W_n^{n2 k1};
//   send    result k1 = ka + 16 kb belongs to the CTA that owns rows 16 kb .. 16 kb + 15: every thread stores one value
//           into each of the 16 CTAs' shared memory (128-byte runs per half-warp), then one cluster barrier;
//   step 3  CTA c owns rows k1 = 16c .. 16c+15: 256-point transforms over n2 (one local exchange), X[k1 + 256 k2] stored
//           as 128-byte runs; fft_shift / ifft_shift / 1/n folded into the index arithmetic.
// Replaces rustfft + swap_halves (time_to_freq.rs:136-165, freq_to_time.rs:138-168) for this length in the latency
// regime (few sequences); batches keep the packed two-pass kernels, which are the faster ones per byte.
#include <cooperative_groups.h>

#include "cxmath.cuh"
#include "fft.cuh"

namespace bdsp {
namespace cg = cooperative_groups;
using namespace cx;

namespace {

constexpr int FC_CL = 16;            // CTAs per cluster = columns / rows per CTA
constexpr int FC_T = 256;
constexpr int FC_RS = 257;           // row stride (float2) of the local exchange buffers: odd -> the row-fastest reads of the
                                     // last stage fall into 16 different 8-byte bank pairs
constexpr size_t FC_SMEM = (size_t)(16 * FC_RS + 16 * 256) * sizeof(float2);

__device__ __forceinline__ c2 root(unsigned m, float two_over_n, bool inv) {   // W_n^m (conjugated for the inverse)
    float s, c;
    sincospif((float)m * two_over_n, &s, &c);
    return make_float2(c, inv ? s : -s);
}

template <bool INV>
__global__ void __launch_bounds__(FC_T, 1)
fftc65536_kernel(const float2* __restrict__ x, float2* __restrict__ out, int shift_in, int shift_out, float scale) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* sa = reinterpret_cast<float2*>(smem_raw);          // local exchanges of step 1 and step 3: 16 x FC_RS
    float2* sb = sa + 16 * FC_RS;                               // rows received from the cluster: [row][n2], 16 x 256
    cg::cluster_group cluster = cg::this_cluster();
    const int c = (int)cluster.block_rank();
    const size_t seq = blockIdx.x / FC_CL;
    const float2* xs = x + seq * 65536;
    float2* os = out + seq * 65536;
    const int t = threadIdx.x;
    const int lo = t & 15, hi = t >> 4;
    cluster.barrier_arrive();   // residency handshake, completed just before the first remote store (hidden behind the loads)
    c2 v[16];
    // ---- step 1, stage 1: thread (col = lo, g = hi): radix 16 over a, n1 = 16 a + g ----
    {
        const float2* p = xs + (size_t)hi * 256 + 16 * c + lo;
#pragma unroll
        for (int a = 0; a < 16; a++) v[a] = __ldg(p + (size_t)(shift_in ? (a ^ 8) : a) * 4096);
        r16<INV>(v);                                             // slot s: ka = r16_k(s)
        apply_twiddles<true>(v, root((unsigned)hi, 2.0f / 256.0f, INV));   // W_256^{g ka}
#pragma unroll
        for (int s = 0; s < 16; s++) sa[r16_k(s) * FC_RS + hi * 16 + lo] = v[s];
    }
    __syncthreads();
    // ---- step 1, stage 2: thread (col = lo, ka = hi): radix 16 over g; k1 = ka + 16 kb; twiddle W_n^{n2 k1}; send ----
    {
#pragma unroll
        for (int g = 0; g < 16; g++) v[g] = sa[hi * FC_RS + g * 16 + lo];
        r16<INV>(v);                                             // slot s: kb = r16_k(s)
        const unsigned n2 = 16u * (unsigned)c + (unsigned)lo;
        apply_twiddles<true>(v, root(16u * n2, 2.0f / 65536.0f, INV));      // (W_n^{16 n2})^{kb}
        const c2 base = root(n2 * (unsigned)hi, 2.0f / 65536.0f, INV);      // W_n^{n2 ka}
        cluster.barrier_wait();   // every CTA of the cluster is resident before anyone writes into its shared memory
#pragma unroll
        for (int s = 0; s < 16; s++) {
            float2* dst = cluster.map_shared_rank(sb, r16_k(s));            // rows 16 kb .. 16 kb + 15 live in CTA kb
            dst[hi * 256 + n2] = mul(v[s], base);
        }
    }
    cluster.sync();   // all 16 x 256 values of this CTA's rows have arrived
    // ---- step 3, stage 1: thread (row = hi, j = lo): radix 16 over a, n2 = 16 a + j ----
    {
#pragma unroll
        for (int a = 0; a < 16; a++) v[a] = sb[hi * 256 + 16 * a + lo];
        r16<INV>(v);
        apply_twiddles<true>(v, root((unsigned)lo, 2.0f / 256.0f, INV));    // W_256^{j ka}
#pragma unroll
        for (int s = 0; s < 16; s++) sa[hi * FC_RS + r16_k(s) * 16 + lo] = v[s];
    }
    __syncthreads();
    // ---- step 3, stage 2: thread (row = lo, ka = hi): radix 16 over j; X[k1 + 256 k2], k2 = ka + 16 kb ----
    {
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = sa[lo * FC_RS + hi * 16 + j];
        r16<INV>(v);
        float2* o = os + 16 * c + lo;
#pragma unroll
        for (int s = 0; s < 16; s++) {
            int k2 = hi + 16 * r16_k(s);
            if (shift_out) k2 ^= 128;
            o[(size_t)k2 * 256] = cx::scale(v[s], scale);
        }
    }
}

cudaLaunchConfig_t fftc_config(size_t rows, cudaStream_t st, cudaLaunchAttribute* attr) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(FC_CL * rows), 1, 1);
    cfg.blockDim = dim3(FC_T, 1, 1);
    cfg.dynamicSmemBytes = FC_SMEM;
    cfg.stream = st;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = FC_CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

}  // namespace

// Whether a 16-CTA cluster of the kernel can be placed on the current device (configures the kernel on first use).  A
// device / driver that cannot place one takes the two-pass path.  Cached for device indices below 16.
bool fftc_cluster_ok() {
    static int state[16] = {};   // 0: unknown, 1: usable, -1: not usable
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return false; }
    if (dev < 16 && state[dev]) return state[dev] > 0;
    auto kf = fftc65536_kernel<false>;
    auto ki = fftc65536_kernel<true>;
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = fftc_config(1, nullptr, attr);
    bool ok = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FC_SMEM) == cudaSuccess &&
              cudaFuncSetAttribute(ki, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FC_SMEM) == cudaSuccess &&
              cudaFuncSetAttribute(kf, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
              cudaFuncSetAttribute(ki, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    int nclusters = 0;
    if (ok) ok = cudaOccupancyMaxActiveClusters(&nclusters, kf, &cfg) == cudaSuccess && nclusters >= 1;
    cudaGetLastError();   // a refusal here is not an error of the call: the two-pass path takes over
    if (dev < 16) state[dev] = ok ? 1 : -1;
    return ok;
}

// 1 .. 8 sequences of 65536 points, in != out (FftRoute::Cluster)
int fftc65536(const void* in, void* out, size_t rows, bool inverse, bool shift_in, bool shift_out, double scale, cudaStream_t st) {
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = fftc_config(rows, st, attr);
    auto kern = inverse ? fftc65536_kernel<true> : fftc65536_kernel<false>;
    BDSP_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, reinterpret_cast<const float2*>(in), reinterpret_cast<float2*>(out), (int)shift_in,
                                    (int)shift_out, (float)scale));
    BDSP_LAUNCHED();
    return 0;
}

}  // namespace bdsp
