// c64 tile passes of the multi-pass transforms (included by fft.cu after TileParams / OutMap).
//
// Same contract as fft_tile_kernel (one CTA = CT lanes x m points of one pass, strides and twiddle modulus in
// TileParams), specialised at compile time for m = 64 .. 512 and written for the instruction budget of f64 on B200:
// the generic kernel spends ~260 instructions per point (run-time index arithmetic, four shared-memory round trips,
// per-tile root tables: profiles/r2_c5a_tile_generic_ncu.txt) and runs at 21-35 % DRAM utilisation.  Here
//   * a thread owns the 8 points  j + i * m/8  (i < 8) of one lane: they are the inputs of its first radix-8 butterfly,
//     loaded straight from global memory, AND the outputs of its last one, stored straight to global memory -
//     two shared-memory exchanges per pass instead of four, no staging;
//   * lanes are the fastest thread index: a warp touches (32 / CT) x 8 row segments of CT * 16 bytes on both sides,
//     for column passes (lane stride 1) and for the transposing row pass alike;
//   * the pass twiddle W_tw^{lane k} costs one exactly reduced sincospi per thread (k = j) and one per lane (k = m/8);
//     the other seven are a product chain;
//   * Q = 3: columns of 3 m points - a radix-3 decimation-in-frequency step (global -> shared) in front of three
//     m-point transforms, results K = ka + 3 kb (time_freq/mod.rs:32-63: rustfft plans any length; BASELINE C5a).
#pragma once

#define F64T_MIN_CTAS 4
#define F64T_Q3_LCT 2   // lanes (log2) per tile of the radix-3 first pass: 3 x 256 x 4 points, 384 threads
#define F64T_Q3_MIN_CTAS 2
#define F64T_POINTS_LOG2 11
namespace f64t {

__device__ __forceinline__ double2 conj_if(double2 w, bool c) { return c ? make_double2(w.x, -w.y) : w; }

// W_den^x (forward sign, INV: conjugate) for x < 2^53: x mod den through the reciprocal estimate, then sincospi
template <bool INV>
__device__ __forceinline__ double2 root_of(unsigned long long x, long long den, double inv_den) {
    const long long q = (long long)((double)x * inv_den);
    long long r = (long long)x - q * den;
    if (r < 0) r += den;
    else if (r >= den) r -= den;
    double s, c;
    sincospi(2.0 * (double)r / (double)den, &s, &c);
    return make_double2(c, INV ? s : -s);
}

// v[r] *= w1^r, r = 1 .. R-1 (product tree of depth <= 3)
template <int R>
__device__ __forceinline__ void twiddle_powers(double2* v, int stride, double2 w1) {
    if (R >= 2) v[stride] = cmul(v[stride], w1);
    if (R >= 4) {
        const double2 w2 = cmul(w1, w1), w3 = cmul(w2, w1);
        v[2 * stride] = cmul(v[2 * stride], w2);
        v[3 * stride] = cmul(v[3 * stride], w3);
        if (R >= 8) {
            const double2 w4 = cmul(w2, w2);
            v[4 * stride] = cmul(v[4 * stride], w4);
            v[5 * stride] = cmul(v[5 * stride], cmul(w4, w1));
            v[6 * stride] = cmul(v[6 * stride], cmul(w3, w3));
            v[7 * stride] = cmul(v[7 * stride], cmul(w4, w3));
        }
    }
}

template <int LOG2M, int LCT, int Q> struct Geo {
    static constexpr int M = 1 << LOG2M, CT = 1 << LCT, J = M / 8;
    static constexpr int NT = J * CT * Q;
    static constexpr int UNITS = M * CT + (LCT < 3 ? M * CT / 8 : 0);   // padded complex words per sub-sequence region
    static constexpr size_t SMEM = ((size_t)UNITS * Q + CT) * sizeof(double2);
};

template <int LOG2M, int LCT, int Q, bool INV>
__global__ void __launch_bounds__(Geo<LOG2M, LCT, Q>::NT, Q == 1 ? (F64T_MIN_CTAS * 256) / Geo<LOG2M, LCT, Q>::NT : F64T_Q3_MIN_CTAS)
f64_tile_kernel(TileParams p, double scale, const double2* __restrict__ tw, const double2* __restrict__ w3tab) {
    typedef Geo<LOG2M, LCT, Q> G;
    constexpr int M = G::M, CT = G::CT, J = G::J, NT = G::NT;
    constexpr int R3 = LOG2M == 6 ? 1 : M / 64;   // radix of the third stage (m = 8 * 8 * R3; 1: two stages)
    constexpr int U3 = LOG2M == 6 ? 1 : 8 / R3;   // third-stage butterflies per thread
    constexpr int TWL = 16384;                    // master table W_16384^i
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* sbase = reinterpret_cast<double2*>(smem_raw);
    double2* sstep = sbase + G::UNITS * Q;        // per-lane step root W_tw^{lane * stepk}
    const int tid = threadIdx.x;
    const int l = tid & (CT - 1);
    const int jq = tid >> LCT;
    const int ka = Q > 1 ? jq >> (LOG2M - 3) : 0;
    const int j = jq & (J - 1);
    double2* s = sbase + ka * G::UNITS;
    // word of sequence element idx of this thread's lane: lanes fastest; one lane-group of padding per 8 elements keeps the
    // stride-8 writes of the first stage on distinct banks when a 128-byte phase spans several j (CT < 8)
    auto at = [&](int idx) -> double2& {
        const int u = (idx << LCT) + l;
        return s[LCT < 3 ? u + ((u >> (3 + LCT)) << LCT) : u];
    };
    const long long tile = blockIdx.x, o1 = blockIdx.y, b = blockIdx.z;
    const long long lane = tile * CT + l;
    const long long inb = b * p.in_batch_stride + o1 * p.in_o1_stride;
    const double inv_tw = p.tw_n ? 1.0 / (double)p.tw_n : 0.0;
    constexpr int stepk = Q * J;                  // distance of a thread's consecutive results in the column
    double2 v[8];

    if (Q == 1) {
        // positions inside a sequence fit 32 bits (sequences have fewer than 2^31 points)
        const int n_in = (int)p.in_n;
        const int g0 = (int)lane * (int)p.in_lane_stride + j * (int)p.in_point_stride + (int)p.in_rot;
        const int gs = J * (int)p.in_point_stride;
        if (p.real_input) {
            const double* in = reinterpret_cast<const double*>(p.in) + inb;
#pragma unroll
            for (int r = 0; r < 8; r++) {
                int g = g0 + r * gs;
                if (g >= n_in) g -= n_in;
                v[r] = make_double2(in[g], 0.0);
                if (p.im.kind) v[r] = in_mul_apply<double>(v[r], p.im.p, p.im.kind, p.im.arg, g, p.in_n);
            }
        } else {
            const double2* in = reinterpret_cast<const double2*>(p.in) + inb;
#pragma unroll
            for (int r = 0; r < 8; r++) {
                int g = g0 + r * gs;
                if (g >= n_in) g -= n_in;
                v[r] = in[g];
                if (p.im.kind) v[r] = in_mul_apply<double>(v[r], p.im.p, p.im.kind, p.im.arg, g, p.in_n);
            }
        }
        if (p.tw_n && jq == 0) sstep[l] = root_of<INV>((unsigned long long)lane * stepk, p.tw_n, inv_tw);
    } else {
        // ---- radix-3 step over stride m: z_ka[b] = (sum_a y[a m + b] W_3^{a ka}) W_{3m}^{b ka} ----
        constexpr int NB = M * CT;                    // butterflies per CTA
        constexpr int IT = (NB + NT - 1) / NT;
        double2 y[IT][3];
#pragma unroll
        for (int it = 0; it < IT; it++) {
            const int bi = tid + it * NT;
            if (bi < NB) {
                const int l3 = bi & (CT - 1), b3 = bi >> LCT;
                const int n_in = (int)p.in_n;   // positions inside a sequence fit 32 bits
                const int g0 = (int)(tile * CT + l3) * (int)p.in_lane_stride + b3 * (int)p.in_point_stride + (int)p.in_rot;
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    int g = g0 + a * M * (int)p.in_point_stride;
                    if (g >= n_in) g -= n_in;
                    if (p.real_input) y[it][a] = make_double2(reinterpret_cast<const double*>(p.in)[inb + g], 0.0);
                    else y[it][a] = reinterpret_cast<const double2*>(p.in)[inb + g];
                    if (p.im.kind) y[it][a] = in_mul_apply<double>(y[it][a], p.im.p, p.im.kind, p.im.arg, g, p.in_n);
                }
            }
        }
        if (p.tw_n && tid < CT) sstep[tid] = root_of<INV>((unsigned long long)(tile * CT + tid) * stepk, p.tw_n, inv_tw);   // read after later barriers
        const double sn = INV ? 0.86602540378443864676 : -0.86602540378443864676;   // Im W_3
#pragma unroll
        for (int it = 0; it < IT; it++) {
            const int bi = tid + it * NT;
            if (bi < NB) {
                const int l3 = bi & (CT - 1), b3 = bi >> LCT;
                const double2 y0 = y[it][0], t = cadd(y[it][1], y[it][2]), d = csub(y[it][1], y[it][2]);
                const double2 m0 = make_double2(y0.x - 0.5 * t.x, y0.y - 0.5 * t.y);
                const double2 id = make_double2(-sn * d.y, sn * d.x);          // i * Im(W_3) * (y1 - y2)
                const double2 w1 = conj_if(__ldg(&w3tab[b3]), INV);     // W_{3m}^b from the per-device table (forward sign)
                const int u = (b3 << LCT) + l3;
                const int word = LCT < 3 ? u + ((u >> (3 + LCT)) << LCT) : u;
                sbase[word] = cadd(y0, t);
                sbase[G::UNITS + word] = cmul(cadd(m0, id), w1);
                sbase[2 * G::UNITS + word] = cmul(csub(m0, id), cmul(w1, w1));
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = at(j + r * J);
        __syncthreads();
    }

    // ---- stage 1: radix 8 over stride m/8, no twiddles; results to 8 j + r ----
    RegFFT<double, 8, INV>::run(v);
#pragma unroll
    for (int r = 0; r < 8; r++) at(8 * j + r) = v[r];
    __syncthreads();
    // ---- stage 2: Ns = 8, radix 8 ----
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = at(j + r * J);
    {
        const int k = j & 7;
        twiddle_powers<8>(v, 1, conj_if(__ldg(&tw[k * (TWL / 64)]), INV));
    }
    RegFFT<double, 8, INV>::run(v);
    if constexpr (LOG2M > 6) {
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 8; r++) at((j >> 3) * 64 + (j & 7) + 8 * r) = v[r];
        __syncthreads();
        // ---- stage 3: Ns = 64, radix R3; butterfly u of the thread: jb = j + u J, element r at jb + 64 r = j + (u + r U3) J ----
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = at(j + i * J);
#pragma unroll
        for (int u = 0; u < U3; u++) {
            const int k = j + u * J;
            twiddle_powers<R3>(v + u, U3, conj_if(__ldg(&tw[k * (TWL / M)]), INV));
            double2 x[R3];
#pragma unroll
            for (int r = 0; r < R3; r++) x[r] = v[u + r * U3];
            RegFFT<double, R3, INV>::run(x);
#pragma unroll
            for (int r = 0; r < R3; r++) v[u + r * U3] = x[r];
        }
    }
    // ---- pass twiddle W_tw^{lane K}, K = kfirst + i * stepk, and store ----
    const int kfirst = Q > 1 ? ka + Q * j : j;
    if (p.tw_n) {
        double2 c = root_of<INV>((unsigned long long)lane * kfirst, p.tw_n, inv_tw);
        c.x *= scale; c.y *= scale;
        const double2 st = sstep[l];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            v[i] = cmul(v[i], c);
            if (i < 7) c = cmul(c, st);
        }
    } else if (scale != 1.0) {
#pragma unroll
        for (int i = 0; i < 8; i++) { v[i].x *= scale; v[i].y *= scale; }
    }
    const long long local0 = o1 * p.out_o1_stride + lane * p.out_lane_stride + (long long)kfirst * p.out_point_stride;
    const long long ls = (long long)stepk * p.out_point_stride;
    if (p.last) {
        const long long grp = p.om.seq_group == 1 ? b : b / p.om.seq_group;
        const long long rb = b - grp * p.om.seq_group;
        const long long base = grp * p.om.group_stride;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            long long loc = rb + (local0 + i * ls) * p.om.oes + p.om.rot;
            if (loc >= p.om.rot_n) loc -= p.om.rot_n;
            if (p.magnitude) reinterpret_cast<double*>(p.out)[base + loc] = sqrt(v[i].x * v[i].x + v[i].y * v[i].y);
            else reinterpret_cast<double2*>(p.out)[base + loc] = v[i];
        }
    } else {
        double2* out = reinterpret_cast<double2*>(p.out) + b * p.out_batch_stride;
        const int l0 = (int)local0, lsi = (int)ls;
#pragma unroll
        for (int i = 0; i < 8; i++) out[l0 + i * lsi] = v[i];
    }
}

template <int LOG2M, int LCT, int Q, bool INV>
int launch_one(const TileParams& p, long long batch, double scale, const double2* tw, cudaStream_t st) {
    typedef Geo<LOG2M, LCT, Q> G;
    auto kernel = f64_tile_kernel<LOG2M, LCT, Q, INV>;
    static bool configured[16] = {};
    int dev = 0;
    BDSP_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 16 && !configured[dev]) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM));
        BDSP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured[dev] = true;
    } else if (dev >= 16) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM));
    }
    const double2* w3tab = nullptr;
    if (Q == 3) {
        // W_{3m}^b, b < m (forward sign), evaluated once per device on the host in long double
        static double2* tabs[16] = {};
        static std::mutex mu;
        std::lock_guard<std::mutex> lk(mu);
        if (dev >= 16) return 1;
        if (!tabs[dev]) {
            std::vector<double2> h(G::M);
            const long double tau = 2.0L * 3.14159265358979323846264338327950288L;
            for (int b = 0; b < G::M; b++) {
                h[b].x = (double)cosl(tau * (long double)b / (long double)(3 * G::M));
                h[b].y = (double)-sinl(tau * (long double)b / (long double)(3 * G::M));
            }
            double2* d = nullptr;
            BDSP_CUDA_OK(cudaMalloc(&d, sizeof(double2) * G::M));
            BDSP_CUDA_OK(cudaMemcpy(d, h.data(), sizeof(double2) * G::M, cudaMemcpyHostToDevice));
            tabs[dev] = d;
        }
        w3tab = tabs[dev];
    }
    const dim3 grid((unsigned)(p.lanes >> LCT), (unsigned)p.o1_count, (unsigned)batch);
    kernel<<<grid, G::NT, G::SMEM, st>>>(p, scale, tw, w3tab);
    return 0;
}

// 1: not covered by these kernels (the caller falls back to fft_tile_kernel), 0: launched, < 0: error
template <bool INV>
int launch(const TileParams& p, long long batch, double scale, const double2* tw, cudaStream_t st) {
    if (batch > 65535 || p.o1_count > 65535 || p.in_n >= (1ll << 30)) return 1;   // (32-bit positions inside a sequence)
    if (p.q == 3) {
        if (p.log2m == 8 && p.lanes % (1 << F64T_Q3_LCT) == 0) return launch_one<8, F64T_Q3_LCT, 3, INV>(p, batch, scale, tw, st);
        return 1;
    }
    if (p.q != 1) return 1;
    constexpr int PL = F64T_POINTS_LOG2;          // points per CTA
    switch (p.log2m) {
        case 6: if (p.lanes % (1 << (PL - 6)) == 0) return launch_one<6, PL - 6, 1, INV>(p, batch, scale, tw, st); break;
        case 7: if (p.lanes % (1 << (PL - 7)) == 0) return launch_one<7, PL - 7, 1, INV>(p, batch, scale, tw, st); break;
        case 8: if (p.lanes % (1 << (PL - 8)) == 0) return launch_one<8, PL - 8, 1, INV>(p, batch, scale, tw, st); break;
        case 9:
            // 512-point passes: 8 lanes (128-byte segments, 4096 points, 512 threads) where the lane count allows - measured on
            // B200 (C5a): 5.56 ms against 5.72 ms with 4 lanes; 32-byte segments (2 lanes): 7.2 ms
            if (p.lanes % (2 << (PL - 9)) == 0) return launch_one<9, PL - 8, 1, INV>(p, batch, scale, tw, st);
            if (p.lanes % (1 << (PL - 9)) == 0) return launch_one<9, PL - 9, 1, INV>(p, batch, scale, tw, st);
            break;
        default: break;
    }
    return 1;
}

// ------------------------------------------------------------------------------------------
// single-pass rows of n = 1024 / 2048 / 4096 c64 points: one row per CTA, n/8 threads, radix 8 x 8 x 8 x (n/512), the
// same ownership as above (a thread loads the 8 inputs of its first butterfly and stores the 8 outputs of its last one),
// three shared-memory exchanges.  The generic fft_block_kernel ran these rows at 45-49 % of the 32 B/point bound.
// ------------------------------------------------------------------------------------------
template <int LOG2N, bool INV>
__global__ void __launch_bounds__((1 << LOG2N) / 8, 1024 / ((1 << LOG2N) / 8))
f64_row_kernel(const void* __restrict__ in_, void* __restrict__ out_, long long in_rot, int real_input, double scale, OutMap om, int magnitude,
               InMul im, const double2* __restrict__ tw) {
    constexpr int N = 1 << LOG2N, J = N / 8;
    constexpr int R4 = N / 512, U4 = 8 / R4;
    constexpr int TWL = 16384;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* s = reinterpret_cast<double2*>(smem_raw);
    auto at = [&](int idx) -> double2& { return s[idx + (idx >> 3)]; };
    const int j = threadIdx.x;
    const long long b = blockIdx.x;
    double2 v[8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const long long g = (j + r * J + in_rot) & (N - 1);
        if (real_input) v[r] = make_double2(reinterpret_cast<const double*>(in_)[b * N + g], 0.0);
        else v[r] = reinterpret_cast<const double2*>(in_)[b * N + g];
        if (im.kind) v[r] = in_mul_apply<double>(v[r], im.p, im.kind, im.arg, g, N);
    }
    RegFFT<double, 8, INV>::run(v);
#pragma unroll
    for (int r = 0; r < 8; r++) at(8 * j + r) = v[r];
    __syncthreads();
#pragma unroll
    for (int st = 1; st < 3; st++) {                                   // Ns = 8, 64
        const int Ns = 1 << (3 * st);
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = at(j + J * r);
        const int k = j & (Ns - 1);
        twiddle_powers<8>(v, 1, conj_if(__ldg(&tw[k * (TWL / (8 * Ns))]), INV));
        RegFFT<double, 8, INV>::run(v);
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 8; r++) at((j - k) * 8 + k + Ns * r) = v[r];
        __syncthreads();
    }
    // last stage: Ns = 512, radix R4; butterfly u of the thread: index j + u J, element r at j + (u + r U4) J
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = at(j + i * J);
#pragma unroll
    for (int u = 0; u < U4; u++) {
        const int k = j + u * J;
        twiddle_powers<R4>(v + u, U4, conj_if(__ldg(&tw[k * (TWL / N)]), INV));
        double2 x[R4];
#pragma unroll
        for (int r = 0; r < R4; r++) x[r] = v[u + r * U4];
        RegFFT<double, R4, INV>::run(x);
#pragma unroll
        for (int r = 0; r < R4; r++) v[u + r * U4] = x[r];
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const long long a = out_addr(om, b, j + i * J);
        const double2 y = make_double2(v[i].x * scale, v[i].y * scale);
        if (magnitude) reinterpret_cast<double*>(out_)[a] = sqrt(y.x * y.x + y.y * y.y);
        else reinterpret_cast<double2*>(out_)[a] = y;
    }
}

template <int LOG2N, bool INV>
int launch_row(const void* in, void* out, size_t batch, bool real_in, bool mag, long long in_rot, double scale, const OutMap& om,
               const InMul& im, const double2* tw, cudaStream_t st) {
    constexpr int N = 1 << LOG2N;
    const size_t smem = (size_t)(N + N / 8) * sizeof(double2);
    auto kernel = f64_row_kernel<LOG2N, INV>;
    static bool configured[16] = {};
    int dev = 0;
    BDSP_CUDA_OK(cudaGetDevice(&dev));
    if (dev >= 16 || !configured[dev]) {
        BDSP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        BDSP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        if (dev < 16) configured[dev] = true;
    }
    kernel<<<(unsigned)batch, N / 8, smem, st>>>(in, out, in_rot, real_in ? 1 : 0, scale, om, mag ? 1 : 0, im, tw);
    return 0;
}

// n = 1024 / 2048 / 4096, batch < 2^31 (FftRoute::C64Rows); 0: launched, < 0: error.  The scale is applied to the input by
// the generic kernel and to the output here (the transform is linear).
template <bool INV>
int launch_rows(const void* in, void* out, size_t n, size_t batch, bool real_in, bool mag, long long in_rot, double scale, const OutMap& om,
                const InMul& im, const double2* tw, cudaStream_t st) {
    if (n == 1024) return launch_row<10, INV>(in, out, batch, real_in, mag, in_rot, scale, om, im, tw, st);
    if (n == 2048) return launch_row<11, INV>(in, out, batch, real_in, mag, in_rot, scale, om, im, tw, st);
    return launch_row<12, INV>(in, out, batch, real_in, mag, in_rot, scale, om, im, tw, st);
}

}  // namespace f64t
