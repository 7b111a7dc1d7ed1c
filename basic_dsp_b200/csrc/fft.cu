// FFT engine: plain unnormalised DFT of any length on device-resident interleaved complex data.
//
// Replaces the reference's call into rustfft (vector/src/vector_types/time_freq/mod.rs:32-63) and
// its clFFT offload (vector/src/gpu_support/ocl/mod.rs:335-349,395-413).
//
//   n = 2^k <= block limit : one CTA per (group of) sequence(s), whole sequence in shared memory
//                            -> one HBM read + one HBM write (fft_block_kernel)
//   n = 2^k larger         : 2 or 3 passes of shared-memory tiles (fft_tile_kernel); the twiddle
//                            between passes is fused into the store of the earlier pass and the
//                            transposition into the store of the last one
//   n = q * 2^k, q odd<=31 : one radix-q pass (dft_q_pass_kernel) + the power-of-two machinery
//   any other n            : Bluestein chirp-z on top of the power-of-two transform
//
// ifft_shift / scaling / real->complex are fused into the load of the first pass, fft_shift and
// magnitude into the store of the last one (FftOpts).
//
// fft_route (fft_route.h) is the one place that picks the path, packed kernels of fftp.cu / fftp16k.cu / fftc.cu
// included; fft_any calls it once per level and switches on the result.
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "fft.cuh"
#include "fft_core.cuh"
#include "fft_route.h"
#include "elementwise.cuh"

namespace bdsp {

// launchers of the packed routes (fftp.cu, fftp16k.cu, fftc.cu): 0 or a negative error
template <bool RIN>
int fftp_single(const void* in, void* out, size_t n, size_t groups, bool inverse, bool si, bool so, bool magnitude, double scale,
                cudaStream_t st);
template <bool RIN>
int fftp_frames(const void* in, void* out, size_t n, size_t groups, size_t hop, const float* win, bool so, bool magnitude, double scale,
                cudaStream_t st);
template <bool RIN>
int fftp_frames_psum(const void* in, float* part, size_t n, size_t groups, size_t ctas, size_t hop, size_t frames, const float* win,
                     cudaStream_t st);
int fftp_two_pass(const void* in, void* out, void* tmp, const FftPlan& p, size_t rows, bool inverse, bool si, bool so, bool magnitude,
                  double scale, bool real_in, const InMul& im, cudaStream_t st);
int fftp_three_pass(const void* in, void* out, void* tmp, const FftPlan& p, size_t n, size_t rows, bool inverse, bool si, bool so,
                    bool magnitude, double scale, bool real_in, const InMul& im, cudaStream_t st);
int fftp_rows_pass(const void* tmp, void* out, int tq, size_t groups, bool inverse, bool so, bool magnitude, float sc, cudaStream_t st,
                   int n1, int n2c);
int fftp16k(const void* in, void* out, size_t rows, bool inverse, bool shift_in, bool shift_out, bool magnitude, float scale, cudaStream_t st);
int fftc65536(const void* in, void* out, size_t rows, bool inverse, bool shift_in, bool shift_out, double scale, cudaStream_t st);
bool fftc_cluster_ok();

// ------------------------------------------------------------------------------------------
// per-device state: twiddle tables, workspaces
// ------------------------------------------------------------------------------------------
namespace {
struct DeviceState {
    float2* tw32 = nullptr;
    double2* tw64 = nullptr;
    int sms = 0;
};
std::mutex g_mu;
std::map<int, DeviceState> g_dev;

// nullptr (last error set) when the device cannot be queried or the tables cannot be allocated
DeviceState* dev_state() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) { set_last_error("cudaGetDevice failed"); return nullptr; }
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceState& s = g_dev[d];
    if (!s.tw32) {
        std::vector<float2> h32(BDSP_TW_LEN);
        std::vector<double2> h64(BDSP_TW_LEN);
        for (int i = 0; i < BDSP_TW_LEN; i++) {
            // exact octant symmetry is not needed: long double evaluation then rounding
            long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)i / (long double)BDSP_TW_LEN;
            long double c = cosl(a), sn = sinl(a);
            if (i == 0) { c = 1; sn = 0; }
            if (i == BDSP_TW_LEN / 4) { c = 0; sn = -1; }
            if (i == BDSP_TW_LEN / 2) { c = -1; sn = 0; }
            if (i == 3 * BDSP_TW_LEN / 4) { c = 0; sn = 1; }
            h64[i].x = (double)c; h64[i].y = (double)sn;
            h32[i].x = (float)c; h32[i].y = (float)sn;
        }
        float2* t32 = nullptr;
        double2* t64 = nullptr;
        int sms = 0;
        if (cudaMalloc(&t32, sizeof(float2) * BDSP_TW_LEN) != cudaSuccess || cudaMalloc(&t64, sizeof(double2) * BDSP_TW_LEN) != cudaSuccess ||
            cudaMemcpy(t32, h32.data(), sizeof(float2) * BDSP_TW_LEN, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(t64, h64.data(), sizeof(double2) * BDSP_TW_LEN, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, d) != cudaSuccess) {
            set_last_error("twiddle tables: %s", cudaGetErrorString(cudaGetLastError()));
            if (t32) cudaFree(t32);
            if (t64) cudaFree(t64);
            return nullptr;
        }
        s.tw64 = t64; s.sms = sms; s.tw32 = t32;
    }
    return &s;
}
}  // namespace

int sm_count() { DeviceState* s = dev_state(); return s ? s->sms : BDSP_SM_COUNT_DEFAULT; }

template <> const float2* twiddle_table<float>() { DeviceState* s = dev_state(); return s ? s->tw32 : nullptr; }
template <> const double2* twiddle_table<double>() { DeviceState* s = dev_state(); return s ? s->tw64 : nullptr; }

// Workspaces are kept per host THREAD and (device, stream): threads that did not bind a stream all run on the legacy
// default stream, where their multi-kernel operations may interleave, so scratch buffers are never shared between
// threads (the reference is safe for concurrent use of distinct vectors).  The calling thread binds its stream with
// workspace_bind_stream (capi: bdsp_set_stream).  Slots: 0..3 the transforms and reductions, 4..5 the full-length
// convolution (its buffers stay live across nested fft_exec calls, which use 0..2), 6 the frame buffers of the frame
// entry points: the gathered frames of FftRoute::FramePass and the inverse rows of ifft_frames_exec (live across the
// transform that fills or reads them, which may use 0..3), 7..8 welch_exec and csd_exec: 7 a chunk of frame spectra
// (csd_exec: the chunk spectra of x, then of y; filled by frame transforms, which may use 0..3 and 6), 8 the window sums
// and the partial rows (live across every chunk).
namespace {
thread_local cudaStream_t tl_ws_stream = nullptr;
constexpr int WS_SLOTS = 9;
struct WsSet { void* p[WS_SLOTS] = {}; size_t bytes[WS_SLOTS] = {}; };
struct WsMap {
    std::map<std::pair<int, cudaStream_t>, WsSet> m;
    ~WsMap() {   // thread exit: give the memory back (errors ignored: the context may already be gone at process exit)
        for (auto& kv : m)
            for (int i = 0; i < WS_SLOTS; i++) if (kv.second.p[i]) cudaFree(kv.second.p[i]);
    }
};
thread_local WsMap tl_ws;
}  // namespace

void workspace_bind_stream(cudaStream_t st) { tl_ws_stream = st; }

void workspace_release_stream(cudaStream_t st) {
    for (auto it = tl_ws.m.begin(); it != tl_ws.m.end();) {
        if (it->first.second == st) {
            for (int i = 0; i < WS_SLOTS; i++) if (it->second.p[i]) cudaFree(it->second.p[i]);
            it = tl_ws.m.erase(it);
        } else ++it;
    }
}

void* workspace(size_t bytes, int slot) {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) { set_last_error("cudaGetDevice failed"); return nullptr; }
    WsSet& s = tl_ws.m[std::make_pair(d, tl_ws_stream)];
    if (s.bytes[slot] < bytes) {
        if (s.p[slot]) {
            cudaStreamSynchronize(tl_ws_stream);
            cudaFree(s.p[slot]);
            s.p[slot] = nullptr; s.bytes[slot] = 0;
        }
        size_t want = bytes + bytes / 8;
        if (cudaMalloc(&s.p[slot], want) != cudaSuccess) {
            cudaGetLastError();
            if (cudaMalloc(&s.p[slot], bytes) != cudaSuccess) {
                cudaGetLastError();
                s.p[slot] = nullptr;
                set_last_error("workspace: out of device memory (%zu bytes)", bytes);
                return nullptr;
            }
            want = bytes;
        }
        s.bytes[slot] = want;
    }
    return s.p[slot];
}

template <> size_t fft_block_max_n<float>() { return FFT_BLOCK_MAX_C32; }
template <> size_t fft_block_max_n<double>() { return FFT_BLOCK_MAX_C64; }

// ------------------------------------------------------------------------------------------
// output addressing shared by all "last pass" kernels
// ------------------------------------------------------------------------------------------
struct OutMap {
    // result element k of inner sequence b goes to
    //   group = b / seq_group, r = b % seq_group, local = r + k*oes,
    //   address = group*group_stride + (local + rot) mod rot_n
    long long seq_group;
    long long oes;
    long long group_stride;
    long long rot;
    long long rot_n;
};

__device__ __forceinline__ long long out_addr(const OutMap& m, long long b, long long k) {
    long long g = b / m.seq_group, r = b - g * m.seq_group;
    long long local = r + k * m.oes + m.rot;
    if (local >= m.rot_n) local -= m.rot_n;
    return g * m.group_stride + local;
}

template <typename T> __device__ __forceinline__ T mag_of(T re, T im) { return sqrt(re * re + im * im); }
__device__ __forceinline__ int spad_host_dev(int n) { return n + (n >> 4) + 1; }

// ------------------------------------------------------------------------------------------
// single-CTA kernel: nfft sequences of n = 2^log2n points per CTA
// ------------------------------------------------------------------------------------------
#define BDSP_BLOCK_POINTS 1024
template <typename T, bool INV, bool REAL_IN, bool MAG>
__global__ void __launch_bounds__(1024, 1) fft_block_kernel(const void* __restrict__ in_, void* __restrict__ out_, int log2n, int nfft,
                                 long long batch, long long in_rot, T scale, OutMap om,
                                 const typename CpxOf<T>::type* __restrict__ tw, InMul im) {
    typedef typename CpxOf<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C* s = reinterpret_cast<C*>(smem_raw);
    const int n = 1 << log2n;
    const int total = n * nfft;
    const long long seq0 = (long long)blockIdx.x * nfft;
    {   // UN independent global loads are issued before the first use (the loop is latency-bound otherwise)
        constexpr int UN = 8;
        for (int base = threadIdx.x; base < total; base += blockDim.x * UN) {
            C v[UN];
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const int idx = base + u * blockDim.x;
                v[u] = mk<T>(0, 0);
                if (idx < total) {
                    const int f = idx >> log2n, p = idx & (n - 1);
                    const long long seq = seq0 + f;
                    if (seq < batch) {
                        const long long src = (p + in_rot) & (n - 1);
                        if (REAL_IN) v[u].x = reinterpret_cast<const T*>(in_)[seq * n + src];
                        else v[u] = reinterpret_cast<const C*>(in_)[seq * n + src];
                        if (im.kind) v[u] = in_mul_apply<T>(v[u], im.p, im.kind, im.arg, src, n);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const int idx = base + u * blockDim.x;
                if (idx < total) {
                    v[u].x *= scale; v[u].y *= scale;
                    s[spad(idx)] = v[u];
                }
            }
        }
    }
    __syncthreads();
    if constexpr (sizeof(T) == 8) {
        // f64: radix-8 stages, 8 points per thread (see fft_tile_kernel)
        int Ns = 1, rem = log2n;
        while (rem >= 3) { stockham_stage_strided<T, 8, INV, 1>(s, n, nfft, n, Ns, tw); Ns <<= 3; rem -= 3; }
        if (rem == 2) stockham_stage_strided<T, 4, INV, 2>(s, n, nfft, n, Ns, tw);
        else if (rem == 1) stockham_stage_strided<T, 2, INV, 4>(s, n, nfft, n, Ns, tw);
    } else {
        block_fft<T, INV>(s, log2n, nfft, tw);
    }
#pragma unroll 4
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        int f = idx >> log2n, k = idx & (n - 1);
        long long seq = seq0 + f;
        if (seq < batch) {
            C v = s[spad(idx)];
            long long a = out_addr(om, seq, k);
            if (MAG) reinterpret_cast<T*>(out_)[a] = mag_of(v.x, v.y);
            else reinterpret_cast<C*>(out_)[a] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// tile kernel for multi-pass transforms: CT lanes x m points per CTA
// ------------------------------------------------------------------------------------------
struct TileParams {
    const void* in;
    void* out;
    int log2m;
    int ct;                    // lanes per tile (power of two)
    long long lanes;           // lanes per o1 group
    long long o1_count;
    long long in_lane_stride, in_point_stride, in_o1_stride, in_batch_stride;
    long long out_lane_stride, out_point_stride, out_o1_stride, out_batch_stride;
    long long tw_n;            // 0: no twiddle; else multiply result (lane, k) by W_{tw_n}^{lane*k}
    long long in_rot, in_n;    // first pass: read element (g + in_rot) mod in_n of the sequence
    int real_input;
    int last;                  // last pass: out index goes through OutMap (batch = inner sequence)
    int magnitude;
    OutMap om;
    InMul im;                  // first pass only: multiplier fused into the load (index = element position in the sequence)
    int q = 1;                 // > 1 (first pass only): columns of q * m points; a radix-q DIF step over stride m runs in shared
                               // memory in front of the m-point transforms, result index K = ka + q * kb
};

template <typename T, bool INV>
__global__ void __launch_bounds__(sizeof(T) == 4 ? 1024 : 512, sizeof(T) == 8 ? 2 : 1) fft_tile_kernel(TileParams p, T scale, const typename CpxOf<T>::type* __restrict__ tw) {
    typedef typename CpxOf<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C* s = reinterpret_cast<C*>(smem_raw);
    const int m = 1 << p.log2m;
    const int ct = p.ct;
    const int Q = p.q;           // sub-columns per lane (1: plain power-of-two columns)
    const int sstride = m + 16;  // sequence stride in shared memory (keeps lane-major accesses conflict free)
    const long long tiles_per_o1 = p.lanes / ct;
    long long t = blockIdx.x;
    const long long tile = t % tiles_per_o1; t /= tiles_per_o1;
    const long long o1 = t % p.o1_count;
    const long long b = t / p.o1_count;
    const long long lane0 = tile * ct;
    const long long in_base = b * p.in_batch_stride + o1 * p.in_o1_stride;
    const int total = m * ct * Q;
    // ---- load ----  (UN independent global loads are issued before the first use: the loop is latency-bound otherwise)
    {
        constexpr int UN = 8;
        const bool contiguous = p.in_point_stride == 1;
        const int lct = __ffs(ct) - 1;
        const int in_ls = (int)p.in_lane_stride, in_ps = (int)p.in_point_stride;
        const long long in_seq0 = o1 * p.in_o1_stride + lane0 * p.in_lane_stride + p.in_rot;
        const long long in_b0 = b * p.in_batch_stride;
        for (int base = threadIdx.x; base < total; base += blockDim.x * UN) {
            C v[UN];
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const int idx = base + u * blockDim.x;
                if (idx < total) {
                    int l, pt;
                    if (contiguous) { l = idx >> p.log2m; pt = idx & (m - 1); }
                    else { pt = idx >> lct; l = idx & (ct - 1); }
                    // 32 x 32 -> 64-bit products (strides are below 2^31: sequences have fewer than 2^31 points)
                    long long g = in_seq0 + (long long)l * in_ls + (long long)pt * in_ps;
                    if (g >= p.in_n) g -= p.in_n;
                    if (p.real_input) { v[u].x = reinterpret_cast<const T*>(p.in)[in_b0 + g]; v[u].y = 0; }
                    else v[u] = reinterpret_cast<const C*>(p.in)[in_b0 + g];
                    if (p.im.kind) v[u] = in_mul_apply<T>(v[u], p.im.p, p.im.kind, p.im.arg, g, p.in_n);
                }
            }
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const int idx = base + u * blockDim.x;
                if (idx < total) {
                    int l, pt;
                    if (contiguous) { l = idx >> p.log2m; pt = idx & (m - 1); }
                    else { pt = idx >> lct; l = idx & (ct - 1); }
                    v[u].x *= scale; v[u].y *= scale;
                    // Q > 1: point pt = a * m + b of lane l goes to sequence l * Q + a, element b
                    s[spad(Q > 1 ? (l * Q + (pt >> p.log2m)) * sstride + (pt & (m - 1)) : l * sstride + pt)] = v[u];
                }
            }
        }
    }
    (void)in_base;
    __syncthreads();
    if (Q > 1) {
        // radix-Q DIF step over stride m inside every lane: z_ka[b] = (sum_a y[a m + b] W_Q^{a ka}) W_{Q m}^{b ka}
        // (time_freq/mod.rs:32-63: rustfft takes any length; this folds the odd factor of q * 2^k lengths into the first pass)
        C* wq = s + spad_host_dev((m + 16) * ct * Q) + ct * (33 + (((Q * m + 31) >> 5) | 1));
        if ((int)threadIdx.x < Q) wq[threadIdx.x] = unit_root<T>((unsigned long long)threadIdx.x, (unsigned long long)Q, INV ? 1 : -1);
        __syncthreads();
        for (int i = threadIdx.x; i < m * ct; i += blockDim.x) {
            const int l = i >> p.log2m, b = i & (m - 1);
            if (Q == 3) {   // registers only
                C* p0 = &s[spad((l * 3 + 0) * sstride + b)];
                C* p1 = &s[spad((l * 3 + 1) * sstride + b)];
                C* p2 = &s[spad((l * 3 + 2) * sstride + b)];
                const C y0 = *p0, y1 = *p1, y2 = *p2;
                const C w1 = unit_root<T>((unsigned long long)b, (unsigned long long)(3 * m), INV ? 1 : -1);
                const C t1 = cmul(y1, wq[1]), t2 = cmul(y2, wq[2]), u1 = cmul(y1, wq[2]), u2 = cmul(y2, wq[1]);
                *p0 = cadd(y0, cadd(y1, y2));
                *p1 = cmul(cadd(y0, cadd(t1, t2)), w1);
                *p2 = cmul(cadd(y0, cadd(u1, u2)), cmul(w1, w1));
                continue;
            }
            C y[31];
            for (int a = 0; a < Q; a++) y[a] = s[spad((l * Q + a) * sstride + b)];
            const C w1 = unit_root<T>((unsigned long long)b, (unsigned long long)(Q * m), INV ? 1 : -1);   // W_{Q m}^{b}
            C wk = mk<T>(1, 0);
            for (int ka = 0; ka < Q; ka++) {
                C acc = y[0];
                int e = 0;
                for (int a = 1; a < Q; a++) {
                    e += ka; if (e >= Q) e -= Q;
                    acc = cadd(acc, cmul(y[a], wq[e]));
                }
                s[spad((l * Q + ka) * sstride + b)] = cmul(acc, wk);
                wk = cmul(wk, w1);
            }
        }
        __syncthreads();
    }
    // ---- transform ----
    {
        const int n = m;
        int Ns = 1, rem = p.log2m;
        // same stage sequence as block_fft, but with the padded sequence stride
        if constexpr (sizeof(T) == 8) {
            // f64: radix-8 stages, 8 points per thread (half the registers of radix 16 -> twice the resident warps;
            // 2^9 = 8*8*8 needs the same three stages as 16*16*2)
            while (rem >= 3) { stockham_stage_strided<T, 8, INV, 1>(s, n, ct * Q, sstride, Ns, tw); Ns <<= 3; rem -= 3; }
            if (rem == 2) stockham_stage_strided<T, 4, INV, 2>(s, n, ct * Q, sstride, Ns, tw);
            else if (rem == 1) stockham_stage_strided<T, 2, INV, 4>(s, n, ct * Q, sstride, Ns, tw);
        } else {
            while (rem >= 4) { stockham_stage_strided<T, 16, INV, 1>(s, n, ct * Q, sstride, Ns, tw); Ns <<= 4; rem -= 4; }
            if (rem == 3) stockham_stage_strided<T, 8, INV, 2>(s, n, ct * Q, sstride, Ns, tw);
            else if (rem == 2) stockham_stage_strided<T, 4, INV, 4>(s, n, ct * Q, sstride, Ns, tw);
            else if (rem == 1) stockham_stage_strided<T, 2, INV, 8>(s, n, ct * Q, sstride, Ns, tw);
        }
    }
    // ---- twiddle + store ----
    // W_{tw_n}^{lane*k} = A[l][k & 31] * B[l][k >> 5] with A[l][a] = W^{lane*a}, B[l][b] = W^{lane*32*b}:
    // ct*(32 + m/32) exactly reduced roots per tile (sincospi) instead of one per element.
    // rows are padded to an odd length: consecutive lanes (rows) must fall into different banks
    C* twA = s + spad_host_dev((m + 16) * ct * Q);
    C* twB = twA + ct * 33;
    const int nb = (Q * m + 31) >> 5;
    const int nbs = nb | 1;
    if (p.tw_n) {
        for (int i = threadIdx.x; i < ct * (32 + nb); i += blockDim.x) {
            const bool isB = i >= ct * 32;
            const int ii = isB ? i - ct * 32 : i;
            const int l = isB ? ii / nb : ii >> 5;
            const int e = isB ? ii - l * nb : ii & 31;
            const unsigned long long lane = (unsigned long long)(lane0 + l);
            const unsigned long long mul = isB ? 32ull * (unsigned long long)e : (unsigned long long)e;
            // lane < tw_n <= 2^40 and mul < 2^15: reduce lane*mul without overflow
            const unsigned long long num = ((lane % (unsigned long long)p.tw_n) * mul) % (unsigned long long)p.tw_n;
            const C w = unit_root<T>(num, (unsigned long long)p.tw_n, INV ? 1 : -1);
            if (isB) twB[l * nbs + e] = w; else twA[l * 33 + e] = w;
        }
        __syncthreads();
    }
    const bool lane_major = (p.out_lane_stride <= p.out_point_stride);
    const int lct = __ffs(ct) - 1;
    const int out_ls = (int)p.out_lane_stride, out_ps = (int)p.out_point_stride;
    const long long out_seq0 = o1 * p.out_o1_stride + lane0 * p.out_lane_stride;
#pragma unroll 4
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        int l, k;
        if (lane_major) { k = idx >> lct; l = idx & (ct - 1); }
        else { l = idx >> p.log2m; k = idx & (m - 1); }
        // Q > 1 (always lane-major): result K = ka + Q * kb of the column sits in sequence l * Q + ka, element kb
        C v = Q > 1 ? s[spad((l * Q + k % Q) * sstride + k / Q)] : s[spad(l * sstride + k)];
        if (p.tw_n) {
            const C w = cmul(twA[l * 33 + (k & 31)], twB[l * nbs + (k >> 5)]);
            v = cmul(v, w);
        }
        long long local = out_seq0 + (long long)l * out_ls + (long long)k * out_ps;
        if (p.last) {
            long long a = out_addr(p.om, b, local);
            if (p.magnitude) reinterpret_cast<T*>(p.out)[a] = mag_of(v.x, v.y);
            else reinterpret_cast<C*>(p.out)[a] = v;
        } else {
            reinterpret_cast<C*>(p.out)[b * p.out_batch_stride + local] = v;
        }
    }
}

#include "fft64t.cuh"   // namespace bdsp::f64t

// ------------------------------------------------------------------------------------------
// radix-q pass for n = q * P, q odd and small:  y[k1*P + n2] = W_n^{n2 k1} sum_{n1} x[n1*P + n2] W_q^{n1 k1}
// ------------------------------------------------------------------------------------------
// Q > 0: compile-time radix (registers, unrolled); Q == 0: any odd q <= 31 (arrays in local memory).
// The q-th roots of unity are evaluated once per block into shared memory.
template <typename T, bool INV, int Q>
__global__ void dft_q_pass_kernel(const void* __restrict__ in_, typename CpxOf<T>::type* __restrict__ out, int q_rt,
                                  long long P, long long batch, long long in_rot, int real_input, T scale, InMul im) {
    typedef typename CpxOf<T>::type C;
    constexpr int QM = Q > 0 ? Q : 31;
    const int q = Q > 0 ? Q : q_rt;
    __shared__ C wq[31];
    const int sign = INV ? 1 : -1;
    if ((int)threadIdx.x < q) wq[threadIdx.x] = unit_root<T>((unsigned long long)threadIdx.x, (unsigned long long)q, sign);
    __syncthreads();
    const long long n = (long long)q * P;
    long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= P * batch) return;
    const long long b = gid / P, n2 = gid - b * P;
    C xin[QM];
#pragma unroll
    for (int n1 = 0; n1 < QM; n1++) {
        if (n1 < q) {
            long long g = (long long)n1 * P + n2 + in_rot;
            if (g >= n) g -= n;
            C v;
            if (real_input) { v.x = reinterpret_cast<const T*>(in_)[b * n + g]; v.y = 0; }
            else v = reinterpret_cast<const C*>(in_)[b * n + g];
            if (im.kind) v = in_mul_apply<T>(v, im.p, im.kind, im.arg, g, n);
            xin[n1] = v;
        }
    }
    const C w1 = unit_root<T>((unsigned long long)n2, (unsigned long long)n, sign);   // W_n^{n2}
    C wk = mk<T>(1, 0);                                                                // W_n^{n2*k1}
#pragma unroll
    for (int k1 = 0; k1 < QM; k1++) {
        if (k1 < q) {
            C acc = xin[0];
            int e = 0;
#pragma unroll
            for (int n1 = 1; n1 < QM; n1++) {
                if (n1 < q) {
                    e += k1; if (e >= q) e -= q;          // (n1*k1) mod q
                    acc = cadd(acc, cmul(xin[n1], wq[e]));
                }
            }
            acc = cmul(acc, wk);
            acc.x *= scale; acc.y *= scale;
            out[b * n + (long long)k1 * P + n2] = acc;
            wk = cmul(wk, w1);
        }
    }
}

// out[b*n + ((k1 + q*k2 + rot) mod n)] = z[(b*q + k1)*P + k2]: the index interleave that follows the q
// row transforms of a q*2^k transform.  A separate, fully coalesced pass: folding it into the strided
// stores of the last tile pass made every 32-byte sector be written q times (read-modify-write in DRAM).
template <typename T>
__global__ void interleave_q_kernel(const typename CpxOf<T>::type* __restrict__ z, void* __restrict__ out_, int q, long long P,
                                    long long batch, long long rot, int magnitude) {
    typedef typename CpxOf<T>::type C;
    const long long n = (long long)q * P;
    long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= P * batch) return;
    const long long b = gid / P, k2 = gid - b * P;
    for (int k1 = 0; k1 < q; k1++) {
        const C v = z[(b * q + k1) * P + k2];
        long long k = k1 + (long long)q * k2 + rot;
        if (k >= n) k -= n;
        if (magnitude) reinterpret_cast<T*>(out_)[b * n + k] = mag_of(v.x, v.y);
        else reinterpret_cast<C*>(out_)[b * n + k] = v;
    }
}

// ------------------------------------------------------------------------------------------
// Bluestein helpers:  X[k] = conj(c[k]) * sum_n (x[n] conj(c[n])) c[k-n],  c[n] = exp(+-i pi n^2 / N)
// ------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ typename CpxOf<T>::type chirp(long long i, long long n, int sign) {
    // exp(sign * i*pi*i^2/n); i^2 mod 2n computed exactly
    unsigned long long m = (unsigned long long)i % (unsigned long long)(2 * n);
    unsigned long long sq = (m * m) % (unsigned long long)(2 * n);  // m < 2^32 guaranteed by the host
    return unit_root<T>(sq, (unsigned long long)(2 * n), sign);
}

template <typename T, bool INV>
__global__ void bluestein_pre_kernel(const void* __restrict__ in_, typename CpxOf<T>::type* __restrict__ a,
                                     long long n, long long M, long long batch, long long in_rot, int real_input, T scale, InMul im) {
    typedef typename CpxOf<T>::type C;
    long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= M * batch) return;
    long long b = gid / M, i = gid - b * M;
    C v = mk<T>(0, 0);
    if (i < n) {
        long long g = i + in_rot; if (g >= n) g -= n;
        if (real_input) v.x = reinterpret_cast<const T*>(in_)[b * n + g];
        else v = reinterpret_cast<const C*>(in_)[b * n + g];
        if (im.kind) v = in_mul_apply<T>(v, im.p, im.kind, im.arg, g, n);
        v.x *= scale; v.y *= scale;
        v = cmul(v, chirp<T>(i, n, INV ? 1 : -1));
    }
    a[gid] = v;
}

template <typename T, bool INV>
__global__ void bluestein_filter_kernel(typename CpxOf<T>::type* __restrict__ bfilt, long long n, long long M) {
    typedef typename CpxOf<T>::type C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    C v = mk<T>(0, 0);
    if (i < n) v = chirp<T>(i, n, INV ? -1 : 1);
    else if (i > M - n) v = chirp<T>(M - i, n, INV ? -1 : 1);
    bfilt[i] = v;
}

template <typename T, bool INV>
__global__ void bluestein_post_kernel(const typename CpxOf<T>::type* __restrict__ c, void* __restrict__ out_,
                                      long long n, long long M, long long batch, OutMap om, int magnitude) {
    typedef typename CpxOf<T>::type C;
    long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n * batch) return;
    long long b = gid / n, k = gid - b * n;
    C v = cmul(c[b * M + k], chirp<T>(k, n, INV ? 1 : -1));
    long long a = out_addr(om, b, k);
    if (magnitude) reinterpret_cast<T*>(out_)[a] = mag_of(v.x, v.y);
    else reinterpret_cast<C*>(out_)[a] = v;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
namespace {

template <typename K> int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) BDSP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

template <typename T, bool INV>
int launch_block(const void* in, void* out, size_t n, size_t batch, bool real_in, bool mag, long long in_rot,
                 T scale, const OutMap& om, cudaStream_t st, const InMul& im = InMul()) {
    typedef typename CpxOf<T>::type C;
    const int log2n = ilog2(n);
    // points per CTA for short sequences (BDSP_BLOCK_POINTS): smaller CTAs overlap their load / compute / store phases better
    int nfft = (int)(BDSP_BLOCK_POINTS / n);
    if (nfft < 1) nfft = 1;
    if ((size_t)nfft > batch) nfft = (int)batch;
    int threads = block_fft_threads((int)n, nfft);
    if (sizeof(T) == 8) { threads = ((int)n * nfft / 8 + 31) / 32 * 32; if (threads < 32) threads = 32; }
    const size_t smem = spad_host(n * nfft) * sizeof(C);
    const long long grid = ((long long)batch + nfft - 1) / nfft;
    const C* tw = twiddle_table<T>();
    if (!tw) return -1001;
#define BDSP_LAUNCH_BLOCK(RI, MG)                                                                   \
    do {                                                                                            \
        int rc = set_smem(fft_block_kernel<T, INV, RI, MG>, smem);                                  \
        if (rc) return rc;                                                                          \
        fft_block_kernel<T, INV, RI, MG><<<(unsigned)grid, threads, smem, st>>>(                    \
            in, out, log2n, nfft, (long long)batch, in_rot, scale, om, tw, im);                     \
    } while (0)
    if (real_in && mag) BDSP_LAUNCH_BLOCK(true, true);
    else if (real_in) BDSP_LAUNCH_BLOCK(true, false);
    else if (mag) BDSP_LAUNCH_BLOCK(false, true);
    else BDSP_LAUNCH_BLOCK(false, false);
#undef BDSP_LAUNCH_BLOCK
    BDSP_LAUNCHED();
    return 0;
}

template <typename T, bool INV>
int launch_tile(const TileParams& p, long long batch, T scale, cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    if constexpr (sizeof(T) == 8) {
        // c64: compile-time specialised passes for m = 64 .. 512 (fft64t.cuh); anything else runs the generic tile kernel
        const double2* twt = twiddle_table<double>();
        if (!twt) return -1001;
        const int rc = f64t::launch<INV>(p, batch, (double)scale, twt, st);
        if (rc <= 0) { if (!rc) BDSP_LAUNCHED(); return rc; }
    }
    const int m = 1 << p.log2m;
    const size_t smem = (spad_host((size_t)(m + 16) * p.ct * p.q) + (size_t)p.ct * (33 + (((p.q * m + 31) >> 5) | 1)) + (p.q > 1 ? 32 : 0)) * sizeof(C);
    int threads = block_fft_threads(m, p.ct * p.q);
    if (sizeof(T) == 8) { threads = (m * p.ct * p.q / 8 + 31) / 32 * 32; if (threads < 32) threads = 32; }
    if (threads > (sizeof(T) == 4 ? 1024 : 512)) { set_last_error("fft tile: %d threads", threads); return -2; }
    const long long grid = batch * p.o1_count * (p.lanes / p.ct);
    int rc = set_smem(fft_tile_kernel<T, INV>, smem);
    if (rc) return rc;
    const typename CpxOf<T>::type* twt = twiddle_table<T>();
    if (!twt) return -1001;
    fft_tile_kernel<T, INV><<<(unsigned)grid, threads, smem, st>>>(p, scale, twt);
    BDSP_LAUNCHED();
    return 0;
}

template <typename T> int tile_log2m_max() { return sizeof(T) == 4 ? 10 : 9; }
// lanes per tile: 128 contiguous bytes per row segment (f32: 16, f64: 8) -> 72 KB tiles, 3 CTAs per SM
// lanes per f64 tile: 4 (64-byte row segments, twice the CTAs) measured mixed on B200: C5a 8.83 -> 8.51 ms, 2^18 0.80 -> 0.73 ms,
// but 2^14 0.82 -> 0.88 and 2^20 1.20 -> 1.31 ms per 2^25 points; 8 stays the default
#define BDSP_TILE_LANES_F64 8
template <typename T> long long tile_lanes() { return sizeof(T) == 8 ? BDSP_TILE_LANES_F64 : 8; }

// power-of-two transform of `batch` sequences with the generic kernels: route C64Rows, Block, Hybrid or Tiles
template <typename T, bool INV>
int fft_pow2(const FftPlan& plan, const void* in, void* out, size_t n, size_t batch, bool real_in, bool mag, long long in_rot, T scale,
             const OutMap& om, void* work, cudaStream_t st, const InMul& im = InMul()) {
    if constexpr (sizeof(T) == 8) {
        if (plan.route == FftRoute::C64Rows) {
            // the 8-points-per-thread row kernel of fft64t.cuh
            const double2* twt = twiddle_table<double>();
            if (!twt) return -1001;
            const int rc = f64t::launch_rows<INV>(in, out, n, batch, real_in, mag, in_rot, (double)scale, om, im, twt, st);
            if (!rc) BDSP_LAUNCHED();
            return rc;
        }
    }
    if (plan.route == FftRoute::Block) return launch_block<T, INV>(in, out, n, batch, real_in, mag, in_rot, scale, om, st, im);
    const int L = ilog2(n);
    const int mx = tile_log2m_max<T>();
    if (plan.route == FftRoute::Hybrid) {
        // generic column pass (any input form: real, rotated, scaled) followed by the packed four-rows-per-CTA 1024-point
        // pass of fftp.cu
        TileParams p;
        p.in = in; p.out = work; p.log2m = L - 10;
        // short columns: more lanes per tile so that a CTA still holds >= 2048 points
        p.lanes = 1024; p.ct = (int)tile_lanes<T>(); p.o1_count = 1;
        while (p.ct < 64 && ((long long)p.ct << p.log2m) < 2048) p.ct *= 2;
        p.in_lane_stride = 1; p.in_point_stride = 1024; p.in_o1_stride = 0; p.in_batch_stride = (long long)n;
        p.out_lane_stride = 1; p.out_point_stride = 1024; p.out_o1_stride = 0; p.out_batch_stride = (long long)n;
        p.tw_n = (long long)n; p.in_rot = in_rot; p.in_n = (long long)n; p.real_input = real_in; p.last = 0; p.magnitude = 0;
        p.om = om;
        p.im = im;
        const int rc = launch_tile<T, INV>(p, (long long)batch, scale, st);
        if (rc) return rc;
        return fftp_rows_pass(work, out, 4, plan.groups, INV, om.rot != 0, mag, 1.0f, st, plan.n1, 1);
    }
    // (A three-pass variant of this hybrid - two generic column passes + the packed 1024-point pass - was measured
    // slower than three generic passes for 2^21 (2.03 vs 1.73 ms per 2^26 points): short columns make the generic
    // kernel's per-tile twiddle tables dominate.)
    int npass = (L + mx - 1) / mx;
    if (npass > 3) { set_last_error("fft: length 2^%d too large for this build", L); return -2; }
    int l[3] = {0, 0, 0};
    for (int i = 0; i < npass; i++) l[i] = L / npass + (i < L % npass ? 1 : 0);
    const long long n1 = 1ll << l[0], n2 = 1ll << l[1], n3 = npass == 3 ? (1ll << l[2]) : 1;
    typedef typename CpxOf<T>::type C;
    C* tmp = reinterpret_cast<C*>(work);
    TileParams p;
    // pass A: columns of length n1, stride n/n1, lanes contiguous
    p.in = in; p.out = tmp; p.log2m = l[0];
    p.lanes = (long long)n / n1; p.ct = (int)(p.lanes < tile_lanes<T>() ? p.lanes : tile_lanes<T>()); p.o1_count = 1;
    p.in_lane_stride = 1; p.in_point_stride = (long long)n / n1; p.in_o1_stride = 0; p.in_batch_stride = (long long)n;
    p.out_lane_stride = 1; p.out_point_stride = (long long)n / n1; p.out_o1_stride = 0; p.out_batch_stride = (long long)n;
    p.tw_n = (long long)n; p.in_rot = in_rot; p.in_n = (long long)n; p.real_input = real_in; p.last = 0; p.magnitude = 0;
    p.om = om;
    p.im = im;
    int rc = launch_tile<T, INV>(p, (long long)batch, scale, st);
    if (rc) return rc;
    p.im = InMul();
    if (npass == 3) {
        // pass B: inside every row k1: columns of length n2, stride n3, in place
        p.in = tmp; p.out = tmp; p.log2m = l[1];
        p.lanes = n3; p.ct = (int)(n3 < tile_lanes<T>() ? n3 : tile_lanes<T>()); p.o1_count = n1;
        p.in_lane_stride = 1; p.in_point_stride = n3; p.in_o1_stride = n2 * n3;
        p.out_lane_stride = 1; p.out_point_stride = n3; p.out_o1_stride = n2 * n3;
        p.tw_n = n2 * n3; p.in_rot = 0; p.real_input = 0;
        rc = launch_tile<T, INV>(p, (long long)batch, (T)1, st);
        if (rc) return rc;
    }
    // last pass: rows of length nl (contiguous), lanes = k1 (stride n/n1), transposing store
    const long long nl = npass == 3 ? n3 : n2;
    p.in = tmp; p.out = out; p.log2m = npass == 3 ? l[2] : l[1];
    p.lanes = n1; p.ct = (int)(n1 < tile_lanes<T>() ? n1 : tile_lanes<T>());
    p.o1_count = npass == 3 ? n2 : 1;
    p.in_lane_stride = (long long)n / n1; p.in_point_stride = 1; p.in_o1_stride = npass == 3 ? nl : 0;
    p.out_lane_stride = 1; p.out_point_stride = npass == 3 ? n1 * n2 : n1; p.out_o1_stride = npass == 3 ? n1 : 0;
    p.tw_n = 0; p.in_rot = 0; p.real_input = 0; p.last = 1; p.magnitude = mag;
    return launch_tile<T, INV>(p, (long long)batch, (T)1, st);
}

// n = q * 2^k (q odd <= 31) too long for one CTA: n = N1 * N2 * N3 with N1 = q * 2^a, three passes of tiles
//   A: columns of N1 points over stride n / N1 (radix-q step + 2^a-point transforms in shared memory), twiddle W_n^{l K1}
//   B: inside every row K1: columns of N2 points over stride N3, in place, twiddle W_{N2 N3}^{l k2}
//   C: rows of N3 points, lanes = K1, transposing store X[K1 + N1 (k2 + N2 k3)]
// 96 bytes per point (c64) instead of the 160 of "radix-q pre-pass + three passes + interleave pass".
// Geometry from the route (FftRoute::QThreePass): N1 = plan.n1 = q * 2^a <= ~1024 points per column, N2 = 2^plan.log2n2
// (1: short enough for no middle pass), N3 = 2^plan.log2n3.
template <typename T, bool INV>
int fft_q_three_pass(const FftPlan& plan, const void* in, void* out, size_t n, size_t batch, bool real_in, long long in_rot, T scale,
                     const OutMap& om, void* work, cudaStream_t st, const InMul& im) {
    typedef typename CpxOf<T>::type C;
    const size_t q = plan.q;
    const int a = ilog2((size_t)plan.n1 / q), b = plan.log2n2, c = plan.log2n3;
    const bool two = b == 0;
    const long long N1 = plan.n1, N2 = 1ll << b, N3 = 1ll << c;
    const long long ct1 = 4;                           // lanes of the first pass: 64-byte (c64) row segments, q * 2^a * 4 points per tile
    C* tmp = reinterpret_cast<C*>(work);
    TileParams p;
    p.in = in; p.out = tmp; p.log2m = a; p.q = (int)q;
    p.lanes = (long long)n / N1; p.ct = (int)ct1; p.o1_count = 1;
    p.in_lane_stride = 1; p.in_point_stride = (long long)n / N1; p.in_o1_stride = 0; p.in_batch_stride = (long long)n;
    p.out_lane_stride = 1; p.out_point_stride = (long long)n / N1; p.out_o1_stride = 0; p.out_batch_stride = (long long)n;
    p.tw_n = (long long)n; p.in_rot = in_rot; p.in_n = (long long)n; p.real_input = real_in; p.last = 0; p.magnitude = 0;
    p.om = om;
    p.im = im;
    int rc = launch_tile<T, INV>(p, (long long)batch, scale, st);
    if (rc) return rc;
    p.q = 1; p.im = InMul();
    if (!two) {
        p.in = tmp; p.out = tmp; p.log2m = b;
        p.lanes = N3; p.ct = (int)(N3 < tile_lanes<T>() ? N3 : tile_lanes<T>()); p.o1_count = N1;
        p.in_lane_stride = 1; p.in_point_stride = N3; p.in_o1_stride = N2 * N3;
        p.out_lane_stride = 1; p.out_point_stride = N3; p.out_o1_stride = N2 * N3;
        p.tw_n = N2 * N3; p.in_rot = 0; p.real_input = 0;
        rc = launch_tile<T, INV>(p, (long long)batch, (T)1, st);
        if (rc) return rc;
    }
    p.in = tmp; p.out = out; p.log2m = c;
    p.lanes = N1; p.ct = (int)tile_lanes<T>();
    // short rows: more lanes per tile so that a CTA still holds >= 2048 points
    while (p.ct < 64 && ((long long)p.ct << c) < 2048 && N1 % (2 * p.ct) == 0) p.ct *= 2;
    if (N1 % p.ct) return -2;
    p.o1_count = two ? 1 : N2;
    p.in_lane_stride = (long long)n / N1; p.in_point_stride = 1; p.in_o1_stride = two ? 0 : N3;
    p.out_lane_stride = 1; p.out_point_stride = two ? N1 : N1 * N2; p.out_o1_stride = two ? 0 : N1;
    p.tw_n = 0; p.in_rot = 0; p.real_input = 0; p.last = 1; p.magnitude = 0;
    return launch_tile<T, INV>(p, (long long)batch, (T)1, st);
}

struct BluesteinKey {
    size_t n; int inv; int is64; int dev;
    bool operator<(const BluesteinKey& o) const {
        if (n != o.n) return n < o.n;
        if (inv != o.inv) return inv < o.inv;
        if (is64 != o.is64) return is64 < o.is64;
        return dev < o.dev;
    }
};
// Cached chirp-filter spectra.  Entries are reference counted (a caller keeps its entry alive while its kernels are
// queued; the deleter synchronises the device before freeing), published only after the stream that computed them has
// been synchronised (any stream of the device may consume them), and evicted least-recently-used first once the cache
// holds more than BLUESTEIN_CACHE_BYTES.
struct BluesteinFilter {
    void* spec = nullptr; size_t bytes = 0; int dev = 0;
    ~BluesteinFilter() {
        if (!spec) return;
        int cur = 0;
        cudaGetDevice(&cur);
        if (cur != dev) cudaSetDevice(dev);
        cudaDeviceSynchronize();
        cudaFree(spec);
        if (cur != dev) cudaSetDevice(cur);
    }
};
struct BluesteinEntry { std::shared_ptr<BluesteinFilter> f; unsigned long long used = 0; };
constexpr size_t BLUESTEIN_CACHE_BYTES = 1ull << 30;
std::map<BluesteinKey, BluesteinEntry> g_bluestein;
unsigned long long g_bluestein_clock = 0;

template <typename T, bool INV>
int fft_any(const void* in, void* out, size_t n, size_t batch, const FftOpts& o, void* work, size_t work_bytes,
            cudaStream_t st);

// route of a plain transform that the caller runs on the generic kernels (fft_pow2) directly
template <typename T>
FftPlan generic_route(const void* in, void* out, size_t n, size_t batch, bool inverse, bool mag, const void* work) {
    return fft_route({sizeof(T) == 8, n, batch, inverse, false, mag, 0, 0, 0, reinterpret_cast<uintptr_t>(in), reinterpret_cast<uintptr_t>(out),
                      reinterpret_cast<uintptr_t>(work), false, true});
}

// spectrum of the chirp filter for length n (M = padded length), from the cache or computed on `st`
template <typename T, bool INV>
int bluestein_filter(size_t n, size_t M, void* w0, cudaStream_t st, std::shared_ptr<BluesteinFilter>* out) {
    typedef typename CpxOf<T>::type C;
    int d = 0;
    BDSP_CUDA_OK(cudaGetDevice(&d));
    const BluesteinKey key{n, INV ? 1 : 0, sizeof(T) == 8 ? 1 : 0, d};
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_bluestein.find(key);
        if (it != g_bluestein.end()) { it->second.used = ++g_bluestein_clock; *out = it->second.f; return 0; }
    }
    auto f = std::make_shared<BluesteinFilter>();
    f->dev = d; f->bytes = M * sizeof(C);
    BDSP_CUDA_OK(cudaMalloc(&f->spec, f->bytes));
    bluestein_filter_kernel<T, INV><<<(unsigned)((M + 255) / 256), 256, 0, st>>>(reinterpret_cast<C*>(f->spec), (long long)n, (long long)M);
    BDSP_LAUNCHED();
    OutMap plain; plain.seq_group = 1; plain.oes = 1; plain.group_stride = (long long)M; plain.rot = 0; plain.rot_n = (long long)M;
    int rc = fft_pow2<T, false>(generic_route<T>(f->spec, f->spec, M, 1, false, false, w0), f->spec, f->spec, M, 1, false, false, 0, (T)1,
                                plain, w0, st);
    if (rc) return rc;
    BDSP_CUDA_OK(cudaStreamSynchronize(st));
    std::vector<std::shared_ptr<BluesteinFilter>> evicted;   // destroyed (device sync + free) outside the lock
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_bluestein.find(key);
        if (it != g_bluestein.end()) {   // another thread computed the same filter meanwhile: use theirs, drop ours
            it->second.used = ++g_bluestein_clock;
            evicted.push_back(f);
            f = it->second.f;
        } else {
            size_t total = f->bytes;
            for (auto& kv : g_bluestein) total += kv.second.f->bytes;
            while (total > BLUESTEIN_CACHE_BYTES && !g_bluestein.empty()) {
                auto lru = g_bluestein.begin();
                for (auto jt = g_bluestein.begin(); jt != g_bluestein.end(); ++jt)
                    if (jt->second.used < lru->second.used) lru = jt;
                total -= lru->second.f->bytes;
                evicted.push_back(lru->second.f);
                g_bluestein.erase(lru);
            }
            BluesteinEntry e; e.f = f; e.used = ++g_bluestein_clock;
            g_bluestein[key] = e;
        }
    }
    *out = f;
    return 0;
}

// table of the built-in window `kind` (InMul kind 3 -> kind 1) for the kernels that take tables only
template <typename T>
__global__ void window_table_kernel(T* __restrict__ tab, long long n, int kind) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tab[i] = window_value_dev<T>(kind, i < (n + 1) / 2 ? i : n - 1 - i, n);
}

// out[b][g] = in[b][g] * multiplier[g]: the separate pass for transforms whose kernels take no first-load multiplier
// (packed single-pass c32 rows).  Real rows stay real under a real table and become complex under a complex one.
template <typename T>
__global__ void in_mul_rows_kernel(const void* __restrict__ in_, void* __restrict__ out_, long long n, long long total, int real_input, InMul im) {
    typedef typename CpxOf<T>::type C;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long g = i % n;
    C v = real_input ? mk<T>(reinterpret_cast<const T*>(in_)[i], (T)0) : reinterpret_cast<const C*>(in_)[i];
    v = in_mul_apply<T>(v, im.p, im.kind, im.arg, g, n);
    if (real_input && im.kind != 2) reinterpret_cast<T*>(out_)[i] = v.x;
    else reinterpret_cast<C*>(out_)[i] = v;
}

// out[f][p] = in[f * hop + p]: frames of a strided input laid back to back (FftRoute::FramePass), E = real or complex point
template <typename E>
__global__ void gather_frames_kernel(const E* __restrict__ in, E* __restrict__ out, long long n, long long hop, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long f = i / n;
    out[i] = in[f * hop + (i - f * n)];
}

// out[t] = sum_f w[p] y[f][p] / sum_f w[p]^2, p = t - f * hop, over the frames f that cover point t in ascending order:
// the least-squares overlap-add of bdsp_ifft_frames_* (win == nullptr: w = 1, the mean of the covering frames).  The sums
// start from the first frame's terms, so a point that one frame covers without a window is that frame's value bit for bit.
// Neighbouring threads read neighbouring points of every frame, each frame value once; no atomics, so every call writes
// the same bytes.
template <typename T, bool REAL_OUT>
__global__ void overlap_add_kernel(const typename CpxOf<T>::type* __restrict__ y, const T* __restrict__ win, void* __restrict__ out,
                                   long long n, long long hop, long long frames, long long len) {
    typedef typename CpxOf<T>::type C;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= len) return;
    long long f = t < n ? 0 : (t - n) / hop + 1;
    const long long f_hi = min(t / hop, frames - 1);
    long long p = t - f * hop;
    C v = y[f * n + p];
    T w = win ? win[p] : (T)1;
    C num = mk<T>(w * v.x, w * v.y);
    T den = w * w;
    for (++f, p -= hop; f <= f_hi; ++f, p -= hop) {
        v = y[f * n + p];
        w = win ? win[p] : (T)1;
        num.x += w * v.x;
        num.y += w * v.y;
        den += w * w;
    }
    if (REAL_OUT) reinterpret_cast<T*>(out)[t] = num.x / den;
    else reinterpret_cast<C*>(out)[t] = mk<T>(num.x / den, num.y / den);
}

// sums[0] = sum w, sums[1] = sum w^2 over the n entries of a window table, in double: one block, a fixed order
template <typename T>
__global__ void __launch_bounds__(1024) window_sums_kernel(const T* __restrict__ w, long long n, double* __restrict__ sums) {
    __shared__ double s1[1024], s2[1024];
    double a = 0, b = 0;
    for (long long i = threadIdx.x; i < n; i += 1024) {
        const double v = (double)w[i];
        a += v;
        b += v * v;
    }
    s1[threadIdx.x] = a;
    s2[threadIdx.x] = b;
    for (int h = 512; h > 0; h >>= 1) {
        __syncthreads();
        if ((int)threadIdx.x < h) {
            s1[threadIdx.x] += s1[threadIdx.x + h];
            s2[threadIdx.x] += s2[threadIdx.x + h];
        }
    }
    if (threadIdx.x == 0) { sums[0] = s1[0]; sums[1] = s2[0]; }
}

// part[i] (+)= sum |spec[j]|^2 over j = i, i + slabs * n, ... < frames * n: slab s = i / n of the partial rows takes the
// frames s, s + slabs, ... of the chunk, bin i % n.  |X|^2 is rounded in T, the sum kept in double; the first chunk stores.
template <typename T>
__global__ void welch_accumulate_kernel(const typename CpxOf<T>::type* __restrict__ spec, double* __restrict__ part, long long n,
                                        long long frames, long long slabs, int first) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= slabs * n || i >= frames * n) return;
    double s = first ? 0.0 : part[i];
#pragma unroll 4
    for (long long j = i; j < frames * n; j += slabs * n) {
        const typename CpxOf<T>::type v = spec[j];
        s += (double)add_rn(mul_rn(v.x, v.x), mul_rn(v.y, v.y));
    }
    part[i] = s;
}

// Output j of bdsp_welch_*: bin k = j (shift: (j + n - n/2) mod n), the sum of part[r * stride + k] over the `rows` partial
// rows in double (32 bins x 8 lanes per block: lane y takes rows y, y + 8, ..., the lanes are added in order), times
// 1 / (frames * fs * sum w^2), or 1 / (frames * (sum w)^2) with `power`; onesided: bins 0 .. n/2, doubled but for 0 and the
// Nyquist bin of an even n.  sums: the window sums of window_sums_kernel, null without a window (both n).
template <typename T, typename P>
__global__ void __launch_bounds__(256) welch_final_kernel(const P* __restrict__ part, long long rows, long long stride, const double* __restrict__ sums,
                                                          T* __restrict__ out, long long n, long long nout, int shift, int onesided, int power,
                                                          double fs, long long frames) {
    __shared__ double lane[8][33];
    const long long j = (long long)blockIdx.x * 32 + threadIdx.x;
    const long long k = shift ? (j + n - n / 2) % n : j;
    double s = 0;
    if (j < nout) {
#pragma unroll 4
        for (long long r = threadIdx.y; r < rows; r += 8) s += (double)part[r * stride + k];
    }
    lane[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y != 0 || j >= nout) return;
    for (int y = 1; y < 8; y++) s += lane[y][threadIdx.x];
    const double sw = sums ? sums[0] : (double)n, sw2 = sums ? sums[1] : (double)n;
    double v = s / ((double)frames * (power ? sw * sw : fs * sw2));
    if (onesided && k != 0 && 2 * k != n) v *= 2;
    out[j] = (T)v;
}

// part[c * rows + i] (+)= the sums over the frames s, s + slabs, ... < frames of the chunk at bin k (rows = slabs * nout,
// slab s = i / nout, k = i % nout): c = 0, 1 Re and Im of conj(X[k]) Y[k]; with COH c = 2, 3 |X[k]|^2 and |Y[k]|^2 (formed
// as welch_accumulate_kernel forms |X|^2).  Every product and sum of a frame's term is rounded in T on its own, so that
// csd(x, x) has an imaginary part of exactly 0 and csd(y, x) = conj(csd(x, y)) byte for byte; the sums over frames are
// kept in double.  The first chunk stores.
template <typename T, bool COH>
__global__ void csd_accumulate_kernel(const typename CpxOf<T>::type* __restrict__ xs, const typename CpxOf<T>::type* __restrict__ ys,
                                      double* __restrict__ part, long long n, long long nout, long long frames, long long slabs, int first) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long rows = slabs * nout, s = i / nout;
    if (i >= rows || s >= frames) return;
    double re = 0, im = 0, xx = 0, yy = 0;
    if (!first) {
        re = part[i];
        im = part[rows + i];
        if (COH) { xx = part[2 * rows + i]; yy = part[3 * rows + i]; }
    }
#pragma unroll 4
    for (long long j = s * n + (i - s * nout); j < frames * n; j += slabs * n) {
        const typename CpxOf<T>::type a = xs[j], b = ys[j];
        re += (double)add_rn(mul_rn(a.x, b.x), mul_rn(a.y, b.y));
        im += (double)sub_rn(mul_rn(a.x, b.y), mul_rn(a.y, b.x));
        if (COH) {
            xx += (double)add_rn(mul_rn(a.x, a.x), mul_rn(a.y, a.y));
            yy += (double)add_rn(mul_rn(b.x, b.x), mul_rn(b.y, b.y));
        }
    }
    part[i] = re;
    part[rows + i] = im;
    if (COH) { part[2 * rows + i] = xx; part[3 * rows + i] = yy; }
}

// Output j of bdsp_csd_* / bdsp_coherence_*: bin k = j (shift: (j + n - n/2) mod n); each sum of csd_accumulate_kernel
// added over the `rows` partial rows of nout bins in welch_final_kernel's order.  csd: the complex value scaled and folded
// as welch_final_kernel does; COH: |Sxy|^2 / (Sxx Syy) in double, NaN where x or y has no power.
template <typename T, bool COH>
__global__ void __launch_bounds__(256) csd_final_kernel(const double* __restrict__ part, long long rows, const double* __restrict__ sums,
                                                        void* __restrict__ out, long long n, long long nout, int shift, int onesided, int power,
                                                        double fs, long long frames) {
    constexpr int K = COH ? 4 : 2;
    __shared__ double lane[K][8][33];
    const long long j = (long long)blockIdx.x * 32 + threadIdx.x;
    const long long k = shift ? (j + n - n / 2) % n : j, comp = rows * nout;
    double s[K] = {};
    if (j < nout) {
#pragma unroll 4
        for (long long r = threadIdx.y; r < rows; r += 8)
            for (int c = 0; c < K; c++) s[c] += part[c * comp + r * nout + k];
    }
    for (int c = 0; c < K; c++) lane[c][threadIdx.y][threadIdx.x] = s[c];
    __syncthreads();
    if (threadIdx.y != 0 || j >= nout) return;
    for (int y = 1; y < 8; y++)
        for (int c = 0; c < K; c++) s[c] += lane[c][y][threadIdx.x];
    if (COH) {
        static_cast<T*>(out)[j] = (T)(add_rn(mul_rn(s[0], s[0]), mul_rn(s[1], s[1])) / mul_rn(s[2], s[3]));
        return;
    }
    const double sw = sums ? sums[0] : (double)n, sw2 = sums ? sums[1] : (double)n;
    const double den = (double)frames * (power ? sw * sw : fs * sw2);
    double re = s[0] / den, im = s[1] / den;
    if (onesided && k != 0 && 2 * k != n) { re *= 2; im *= 2; }
    static_cast<typename CpxOf<T>::type*>(out)[j] = mk<T>((T)re, (T)im);
}

template <typename T, bool INV>
int fft_any(const void* in, void* out, size_t n, size_t batch, const FftOpts& o, void* work, size_t work_bytes,
            cudaStream_t st) {
    typedef typename CpxOf<T>::type C;
    OutMap om;
    om.seq_group = 1; om.oes = 1; om.group_stride = (long long)n; om.rot = (long long)(o.out_rot % n); om.rot_n = (long long)n;
    const long long in_rot = (long long)(o.in_rot % n);
    const T scale = (T)o.scale;
    InMul im = o.in_mul;
    if (im.kind == 3) {
        // transform kernels take multiplier tables: one small kernel writes the window (n scalars, once per call)
        BDSP_WS(tab, T*, n * sizeof(T), 3);
        window_table_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tab, (long long)n, im.arg);
        BDSP_LAUNCHED();
        im.p = tab; im.kind = 1;
    }
    // the multi-pass power-of-two transforms need a scratch buffer: the caller's or the pass workspace
    void* w = work;
    if (is_pow2(n) && n > fft_block_max_n<T>()) {
        const size_t need = n * batch * sizeof(C);
        if (!w || work_bytes < need) { w = workspace(need, 0); if (!w) return -1001; }
    }
    const bool si = in_rot != 0, so = om.rot != 0, mag = o.magnitude != 0, real_in = o.real_input != 0;
    const FftPlan plan = fft_route({sizeof(T) == 8, n, batch, INV, real_in, mag, im.kind, (size_t)in_rot, (size_t)om.rot, reinterpret_cast<uintptr_t>(in),
                                    reinterpret_cast<uintptr_t>(out), reinterpret_cast<uintptr_t>(w), sizeof(T) == 4 && n == 65536 && fftc_cluster_ok(),
                                    false, o.in_stride});
    switch (plan.route) {
    case FftRoute::FramePass: {
        // the frames back to back in a slot that no route of the rows uses, then those rows exactly as fft_exec takes them
        const long long tot = (long long)(n * batch), hop = (long long)o.in_stride;
        const unsigned grid = (unsigned)((tot + 255) / 256);
        BDSP_WS(fr, void*, n * batch * (real_in ? sizeof(T) : sizeof(C)), 6);
        if (real_in) gather_frames_kernel<T><<<grid, 256, 0, st>>>(static_cast<const T*>(in), static_cast<T*>(fr), (long long)n, hop, tot);
        else gather_frames_kernel<C><<<grid, 256, 0, st>>>(static_cast<const C*>(in), static_cast<C*>(fr), (long long)n, hop, tot);
        BDSP_LAUNCHED();
        FftOpts o2 = o;
        o2.in_stride = n;
        o2.in_mul = im;   // the window table is already written
        return fft_any<T, INV>(fr, out, n, batch, o2, work, work_bytes, st);
    }
    case FftRoute::PackedFrames: {
        const float* win = static_cast<const float*>(im.kind ? im.p : nullptr);   // kind 1: n real scalars
        if (real_in) return fftp_frames<true>(in, out, n, plan.groups, o.in_stride, win, so, mag, o.scale, st);
        return fftp_frames<false>(in, out, n, plan.groups, o.in_stride, win, so, mag, o.scale, st);
    }
    case FftRoute::MulPass: {
        const bool to_complex = real_in && im.kind == 2;
        const bool real_rows = real_in && !to_complex;
        BDSP_WS(mx, void*, n * batch * (real_rows ? sizeof(T) : sizeof(C)), 2);
        const long long tot = (long long)(n * batch);
        in_mul_rows_kernel<T><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(in, mx, (long long)n, tot, o.real_input, im);
        BDSP_LAUNCHED();
        FftOpts o2 = o;
        o2.in_mul = InMul();
        if (to_complex) o2.real_input = 0;
        return fft_any<T, INV>(mx, out, n, batch, o2, work, work_bytes, st);
    }
    case FftRoute::Complexify: {
        BDSP_WS(cx, C*, n * batch * sizeof(C), 1);
        const int rc = ew_zero_interleave<T>(in, cx, n * batch, 2, 1, st);
        if (rc) return rc;
        FftOpts oc = o;
        oc.real_input = 0;
        oc.in_mul = im;
        return fft_any<T, INV>(cx, out, n, batch, oc, work, work_bytes, st);
    }
    case FftRoute::RealRows: return fftp_single<true>(in, out, n, plan.groups, false, false, so, mag, o.scale, st);
    case FftRoute::Packed: return fftp_single<false>(in, out, n, plan.groups, INV, si, so, mag, o.scale, st);
    case FftRoute::Packed16k: return fftp16k(in, out, batch, INV, si, so, mag, (float)o.scale, st);
    case FftRoute::Cluster: return fftc65536(in, out, batch, INV, si, so, o.scale, st);
    case FftRoute::TwoPass: return fftp_two_pass(in, out, w, plan, batch, INV, si, so, mag, o.scale, real_in, im, st);
    case FftRoute::ThreePass: return fftp_three_pass(in, out, w, plan, n, batch, INV, si, so, mag, o.scale, real_in, im, st);
    case FftRoute::C64Rows:
    case FftRoute::Block:
    case FftRoute::Hybrid:
    case FftRoute::Tiles: return fft_pow2<T, INV>(plan, in, out, n, batch, real_in, mag, in_rot, scale, om, w, st, im);
    case FftRoute::QThreePass: {
        // f64, long q * 2^k: three passes with the radix-q step inside the first one (C5a: 3 * 2^26)
        const size_t need = n * batch * sizeof(C);
        if (!w || work_bytes < need || w == in || w == out) { w = workspace(need, 0); if (!w) return -1001; }
        return fft_q_three_pass<T, INV>(plan, in, out, n, batch, real_in, in_rot, scale, om, w, st, im);
    }
    case FftRoute::QRowsInterleave:
    case FftRoute::QRows: {
        const size_t P = plan.P, q = plan.q, need = n * batch * sizeof(C);
        BDSP_WS(w1, C*, need, 1);
        const long long tot = (long long)(P * batch);
        const unsigned qgrid = (unsigned)((tot + 255) / 256);
        if (q == 3) dft_q_pass_kernel<T, INV, 3><<<qgrid, 256, 0, st>>>(in, w1, 3, (long long)P, (long long)batch, in_rot, o.real_input, scale, im);
        else if (q == 5) dft_q_pass_kernel<T, INV, 5><<<qgrid, 256, 0, st>>>(in, w1, 5, (long long)P, (long long)batch, in_rot, o.real_input, scale, im);
        else if (q == 7) dft_q_pass_kernel<T, INV, 7><<<qgrid, 256, 0, st>>>(in, w1, 7, (long long)P, (long long)batch, in_rot, o.real_input, scale, im);
        else dft_q_pass_kernel<T, INV, 0><<<qgrid, 256, 0, st>>>(in, w1, (int)q, (long long)P, (long long)batch, in_rot, o.real_input, scale, im);
        BDSP_LAUNCHED();
        if (plan.route == FftRoute::QRows) {
            // generic rows that store interleaved: result k1 + q*k2 of row (b, k1)
            OutMap om2;
            om2.seq_group = (long long)q; om2.oes = (long long)q; om2.group_stride = (long long)n;
            om2.rot = om.rot; om2.rot_n = (long long)n;
            return fft_pow2<T, INV>(generic_route<T>(w1, out, P, batch * q, INV, mag, nullptr), w1, out, P, batch * q, false, mag, 0, (T)1,
                                    om2, nullptr, st);
        }
        // row transforms into a second buffer (natural order), then one interleave pass
        void* w0 = P > fft_block_max_n<T>() ? workspace(need, 0) : nullptr;
        if (P > fft_block_max_n<T>() && !w0) return -1001;
        BDSP_WS(w2, C*, need, 2);
        FftOpts po;   // plain transform of the q*batch rows: takes the packed passes where they exist
        po.inverse = INV;
        const int rc = fft_any<T, INV>(w1, w2, P, batch * q, po, w0, w0 ? need : 0, st);
        if (rc) return rc;
        interleave_q_kernel<T><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(w2, out, (int)q, (long long)P, (long long)batch, om.rot, o.magnitude);
        BDSP_LAUNCHED();
        return 0;
    }
    case FftRoute::Bluestein: break;
    }
    // Bluestein
    if (n >= (1ull << 31)) { set_last_error("fft: length %zu not supported", n); return -2; }
    const size_t M = next_pow2(2 * n - 1);
    BDSP_WS(a, C*, M * batch * sizeof(C), 1);
    OutMap plain; plain.seq_group = 1; plain.oes = 1; plain.group_stride = (long long)M; plain.rot = 0; plain.rot_n = (long long)M;
    void* w0 = M > fft_block_max_n<T>() ? workspace(M * (batch > 1 ? batch : 1) * sizeof(C), 0) : nullptr;
    if (M > fft_block_max_n<T>() && !w0) return -1001;
    std::shared_ptr<BluesteinFilter> filt;
    {
        const int rcf = bluestein_filter<T, INV>(n, M, w0, st, &filt);
        if (rcf) return rcf;
    }
    const C* bspec = reinterpret_cast<const C*>(filt->spec);
    const long long totM = (long long)(M * batch);
    bluestein_pre_kernel<T, INV><<<(unsigned)((totM + 255) / 256), 256, 0, st>>>(in, a, (long long)n, (long long)M, (long long)batch,
                                                                                 in_rot, o.real_input, scale, im);
    BDSP_LAUNCHED();
    // the two length-M transforms of the chirp-z convolution take the packed passes where they exist: in place with the
    // pass workspace for M > 16384, ping-pong between two buffers for the single-pass sizes (those kernels are out of place)
    FftOpts fo;
    const size_t w0_bytes = w0 ? M * (batch > 1 ? batch : 1) * sizeof(C) : 0;
    int rc;
    const bool pingpong = !w0 && sizeof(T) == 4 && M >= 256 && M * batch >= (1u << 16);
    C* b2 = a;
    if (pingpong) { b2 = reinterpret_cast<C*>(workspace(M * batch * sizeof(C), 2)); if (!b2) return -1001; }
    if (w0) rc = fft_any<T, false>(a, a, M, batch, fo, w0, w0_bytes, st);
    else if (pingpong) rc = fft_any<T, false>(a, b2, M, batch, fo, nullptr, 0, st);
    else rc = fft_pow2<T, false>(generic_route<T>(a, a, M, batch, false, false, w0), a, a, M, batch, false, false, 0, (T)1, plain, w0, st);
    if (rc) return rc;
    // the product with the chirp filter's spectrum (and the 1/M of the inverse) rides on the inverse transform's first
    // load where that transform takes a multiplier; the packed single-pass c32 kernels keep the separate pass
    fo.inverse = 1;
    InMul fm; fm.p = bspec; fm.kind = 2;
    const bool fused_filter = !(sizeof(T) == 4 && M >= 64 && M <= 16384);
    if (!fused_filter) {
        rc = ew_spectrum_mul_rows<T>(b2, bspec, M, batch, 1.0 / (double)M, st);
        if (rc) return rc;
    } else {
        fo.in_mul = fm; fo.scale = 1.0 / (double)M;
    }
    if (w0) rc = fft_any<T, true>(a, a, M, batch, fo, w0, w0_bytes, st);
    else if (pingpong) rc = fft_any<T, true>(b2, a, M, batch, fo, nullptr, 0, st);
    else rc = fft_pow2<T, true>(generic_route<T>(a, a, M, batch, true, false, w0), a, a, M, batch, false, false, 0,
                                fused_filter ? (T)(1.0 / (double)M) : (T)1, plain, w0, st, fused_filter ? fm : InMul());
    if (rc) return rc;
    const long long totn = (long long)(n * batch);
    bluestein_post_kernel<T, INV><<<(unsigned)((totn + 255) / 256), 256, 0, st>>>(a, out, (long long)n, (long long)M, (long long)batch, om, o.magnitude);
    BDSP_LAUNCHED();
    return 0;
}

}  // namespace

template <typename T>
int fft_exec(const void* in, void* out, size_t n, size_t batch, const FftOpts& opts, void* work, size_t work_bytes,
             cudaStream_t stream) {
    if (n == 0 || batch == 0) return 0;
    if (opts.inverse) return fft_any<T, true>(in, out, n, batch, opts, work, work_bytes, stream);
    return fft_any<T, false>(in, out, n, batch, opts, work, work_bytes, stream);
}

template int fft_exec<float>(const void*, void*, size_t, size_t, const FftOpts&, void*, size_t, cudaStream_t);
template int fft_exec<double>(const void*, void*, size_t, size_t, const FftOpts&, void*, size_t, cudaStream_t);

template <typename T>
int ifft_frames_exec(const void* in, void* out, size_t n, size_t hop, size_t frames, const FftOpts& opts, bool real_out,
                     cudaStream_t stream) {
    typedef typename CpxOf<T>::type C;
    if (n == 0 || frames == 0) return 0;
    // the inverse rows into a slot that no route of the rows uses; it stays live across their transform (slots 0..3)
    BDSP_WS(y, C*, n * frames * sizeof(C), 6);
    FftOpts rows = opts;
    rows.in_mul = InMul();
    const int rc = fft_exec<T>(in, y, n, frames, rows, nullptr, 0, stream);
    if (rc) return rc;
    const T* win = nullptr;
    if (opts.in_mul.kind == 3) {
        BDSP_WS(tab, T*, n * sizeof(T), 3);
        window_table_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(tab, (long long)n, opts.in_mul.arg);
        BDSP_LAUNCHED();
        win = tab;
    }
    const long long len = (long long)((frames - 1) * hop + n);
    const unsigned grid = (unsigned)((len + 255) / 256);
    if (real_out) overlap_add_kernel<T, true><<<grid, 256, 0, stream>>>(y, win, out, (long long)n, (long long)hop, (long long)frames, len);
    else overlap_add_kernel<T, false><<<grid, 256, 0, stream>>>(y, win, out, (long long)n, (long long)hop, (long long)frames, len);
    BDSP_LAUNCHED();
    return 0;
}

template int ifft_frames_exec<float>(const void*, void*, size_t, size_t, size_t, const FftOpts&, bool, cudaStream_t);
template int ifft_frames_exec<double>(const void*, void*, size_t, size_t, size_t, const FftOpts&, bool, cudaStream_t);

// The window table of opts (built-in window, kind 3) in slot 3, the multiplier of the frame transforms of welch_exec and
// csd_exec, and with `sums` its sums (window_sums_kernel); *win stays null without a window
template <typename T>
int spectrum_window(const FftOpts& opts, size_t n, double* sums, const T** win, cudaStream_t stream) {
    if (opts.in_mul.kind != 3) return 0;
    BDSP_WS(tab, T*, n * sizeof(T), 3);
    window_table_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(tab, (long long)n, opts.in_mul.arg);
    BDSP_LAUNCHED();
    if (sums) {
        window_sums_kernel<T><<<1, 1024, 0, stream>>>(tab, (long long)n, sums);
        BDSP_LAUNCHED();
    }
    *win = tab;
    return 0;
}

template <typename T>
int welch_exec(const void* in, T* out, size_t n, size_t hop, size_t frames, const FftOpts& opts, bool onesided, bool power_spectrum, double fs,
               cudaStream_t stream) {
    typedef typename CpxOf<T>::type C;
    if (n == 0 || frames == 0) return 0;
    const bool real_in = opts.real_input != 0;
    const size_t esz = real_in ? sizeof(T) : sizeof(C);
    const WelchPlan plan = welch_route(sizeof(T) == 8, n, hop, frames, real_in, reinterpret_cast<uintptr_t>(in));
    // the partial rows: fused, `ctas` rows of N floats (N = 4096 * R0); otherwise `slabs` rows of n doubles, about 2^18
    // accumulating threads (each with four loads in flight) whatever n is.  Chunks of at most WELCH_CHUNK_POINTS spectrum
    // points bound the memory.
    constexpr size_t WELCH_CHUNK_POINTS = (size_t)1 << 24, WELCH_ACC_THREADS = (size_t)1 << 18;
    const size_t N = n < 4096 ? 4096 : n;
    const size_t chunk = n >= WELCH_CHUNK_POINTS ? 1 : (WELCH_CHUNK_POINTS / n < frames ? WELCH_CHUNK_POINTS / n : frames);
    const size_t slabs = (WELCH_ACC_THREADS + n - 1) / n < chunk ? (WELCH_ACC_THREADS + n - 1) / n : chunk;
    const size_t part_bytes = plan.fused ? plan.ctas * N * sizeof(float) : slabs * n * sizeof(double);
    BDSP_WS(ws, char*, 2 * sizeof(double) + part_bytes, 8);
    double* sums = reinterpret_cast<double*>(ws);
    void* part = ws + 2 * sizeof(double);
    const T* win = nullptr;
    if (const int rc = spectrum_window<T>(opts, n, sums, &win, stream)) return rc;
    const size_t nout = onesided ? n / 2 + 1 : n;
    const dim3 block(32, 8);
    const unsigned grid = (unsigned)((nout + 31) / 32);
    const int shift = opts.out_rot != 0;
    if constexpr (sizeof(T) == 4) {   // welch_route fuses c32 only
        if (plan.fused) {
            const int rc = real_in ? fftp_frames_psum<true>(in, static_cast<float*>(part), n, plan.groups, plan.ctas, hop, frames, win, stream)
                                   : fftp_frames_psum<false>(in, static_cast<float*>(part), n, plan.groups, plan.ctas, hop, frames, win, stream);
            if (rc) return rc;
            welch_final_kernel<T, float><<<grid, block, 0, stream>>>(static_cast<const float*>(part), (long long)plan.ctas, (long long)N,
                                                                     win ? sums : nullptr, out, (long long)n, (long long)nout, shift, onesided,
                                                                     power_spectrum, fs, (long long)frames);
            BDSP_LAUNCHED();
            return 0;
        }
    }
    // every chunk: the frame transform (fft_exec's routes for strided frames, the window table as its multiplier) into
    // slot 7, then |X|^2 added into the partial rows
    BDSP_WS(spec, C*, chunk * n * sizeof(C), 7);
    FftOpts o;
    o.real_input = opts.real_input;
    o.in_stride = hop;
    if (win) { o.in_mul.p = win; o.in_mul.kind = 1; }
    for (size_t f0 = 0; f0 < frames; f0 += chunk) {
        const size_t cf = frames - f0 < chunk ? frames - f0 : chunk;
        const int rc = fft_exec<T>(static_cast<const char*>(in) + f0 * hop * esz, spec, n, cf, o, nullptr, 0, stream);
        if (rc) return rc;
        const long long threads = (long long)(slabs * n);
        welch_accumulate_kernel<T><<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(spec, static_cast<double*>(part), (long long)n,
                                                                                        (long long)cf, (long long)slabs, f0 == 0);
        BDSP_LAUNCHED();
    }
    welch_final_kernel<T, double><<<grid, block, 0, stream>>>(static_cast<const double*>(part), (long long)slabs, (long long)n, win ? sums : nullptr,
                                                              out, (long long)n, (long long)nout, shift, onesided, power_spectrum, fs, (long long)frames);
    BDSP_LAUNCHED();
    return 0;
}

template int welch_exec<float>(const void*, float*, size_t, size_t, size_t, const FftOpts&, bool, bool, double, cudaStream_t);
template int welch_exec<double>(const void*, double*, size_t, size_t, size_t, const FftOpts&, bool, bool, double, cudaStream_t);

template <typename T>
int csd_exec(const void* x, const void* y, void* out, size_t n, size_t hop, size_t frames, const FftOpts& opts, bool onesided,
             bool power_spectrum, double fs, bool coherence, cudaStream_t stream) {
    typedef typename CpxOf<T>::type C;
    if (n == 0 || frames == 0) return 0;
    const size_t esz = opts.real_input ? sizeof(T) : sizeof(C);
    const CsdPlan plan = csd_plan(sizeof(T) == 8, n, frames);
    // slot 8: the window sums, then 2 (coherence: 4) sums of `slabs` partial rows of the nout output bins
    const size_t nout = onesided ? n / 2 + 1 : n, rows = plan.slabs * nout;
    BDSP_WS(ws, double*, (2 + (coherence ? 4 : 2) * rows) * sizeof(double), 8);
    double* sums = ws;
    const T* win = nullptr;
    if (const int rc = spectrum_window<T>(opts, n, coherence ? nullptr : sums, &win, stream)) return rc;
    // every chunk: the frame transforms of x and of y (fft_exec's routes for strided frames, the window table as their
    // multiplier) into the two halves of slot 7, then the cross sums added into the partial rows
    BDSP_WS(xs, C*, 2 * plan.chunk * n * sizeof(C), 7);
    C* ys = xs + plan.chunk * n;
    FftOpts o;
    o.real_input = opts.real_input;
    o.in_stride = hop;
    if (win) { o.in_mul.p = win; o.in_mul.kind = 1; }
    const unsigned acc_grid = (unsigned)((rows + 255) / 256);
    for (size_t f0 = 0; f0 < frames; f0 += plan.chunk) {
        const size_t cf = frames - f0 < plan.chunk ? frames - f0 : plan.chunk;
        int rc = fft_exec<T>(static_cast<const char*>(x) + f0 * hop * esz, xs, n, cf, o, nullptr, 0, stream);
        if (rc) return rc;
        rc = fft_exec<T>(static_cast<const char*>(y) + f0 * hop * esz, ys, n, cf, o, nullptr, 0, stream);
        if (rc) return rc;
        if (coherence) csd_accumulate_kernel<T, true><<<acc_grid, 256, 0, stream>>>(xs, ys, ws + 2, (long long)n, (long long)nout, (long long)cf,
                                                                                    (long long)plan.slabs, f0 == 0);
        else csd_accumulate_kernel<T, false><<<acc_grid, 256, 0, stream>>>(xs, ys, ws + 2, (long long)n, (long long)nout, (long long)cf,
                                                                          (long long)plan.slabs, f0 == 0);
        BDSP_LAUNCHED();
    }
    const dim3 block(32, 8);
    const unsigned grid = (unsigned)((nout + 31) / 32);
    const int shift = opts.out_rot != 0;
    if (coherence) csd_final_kernel<T, true><<<grid, block, 0, stream>>>(ws + 2, (long long)plan.slabs, nullptr, out, (long long)n, (long long)nout,
                                                                         shift, onesided, 0, 0.0, (long long)frames);
    else csd_final_kernel<T, false><<<grid, block, 0, stream>>>(ws + 2, (long long)plan.slabs, win ? sums : nullptr, out, (long long)n,
                                                                (long long)nout, shift, onesided, power_spectrum, fs, (long long)frames);
    BDSP_LAUNCHED();
    return 0;
}

template int csd_exec<float>(const void*, const void*, void*, size_t, size_t, size_t, const FftOpts&, bool, bool, double, bool, cudaStream_t);
template int csd_exec<double>(const void*, const void*, void*, size_t, size_t, size_t, const FftOpts&, bool, bool, double, bool, cudaStream_t);

}  // namespace bdsp
