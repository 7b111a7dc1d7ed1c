// Common helpers for the basic_dsp_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#define BDSP_SM_COUNT_DEFAULT 148

namespace bdsp {

// --- last error (thread local), reported through bdsp_last_error() ------------------------
void set_last_error(const char* fmt, ...);
const char* get_last_error();
void count_launch();
unsigned long long launch_count();

#define BDSP_CUDA_OK(expr)                                                                  \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            bdsp::set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,              \
                                 cudaGetErrorString(_e));                                   \
            return -1000 - (int)_e;                                                         \
        }                                                                                   \
    } while (0)

// one kernel launch was just issued: count it and surface launch-configuration errors
#define BDSP_LAUNCHED()                                                                     \
    do {                                                                                    \
        bdsp::count_launch();                                                               \
        BDSP_CUDA_OK(cudaGetLastError());                                                   \
    } while (0)

// workspace(): nullptr (and last error set) when the allocation fails
#define BDSP_WS(ptr, T_, bytes, slot)                                                       \
    T_ ptr = reinterpret_cast<T_>(bdsp::workspace((bytes), (slot)));                        \
    if (!ptr) return -1001

// --- complex scalar types ------------------------------------------------------------------
template <typename T> struct CpxOf;
template <> struct CpxOf<float> { typedef float2 type; };
template <> struct CpxOf<double> { typedef double2 type; };

template <typename T> __host__ __device__ __forceinline__ typename CpxOf<T>::type mk(T re, T im) {
    typename CpxOf<T>::type r;
    r.x = re;
    r.y = im;
    return r;
}

template <typename C> __device__ __forceinline__ C cadd(C a, C b) { C r; r.x = a.x + b.x; r.y = a.y + b.y; return r; }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { C r; r.x = a.x - b.x; r.y = a.y - b.y; return r; }
// complex product; FMA contraction allowed (transform kernels, tolerance is rel-L2)
template <typename C> __device__ __forceinline__ C cmul(C a, C b) {
    C r;
    r.x = a.x * b.x - a.y * b.y;
    r.y = a.x * b.y + a.y * b.x;
    return r;
}
template <typename C> __device__ __forceinline__ C cconj(C a) { a.y = -a.y; return a; }

// --- the reference's CPU arithmetic: every product, sum, difference and quotient rounded on its own (no FMA contraction),
// so that elementwise results follow the reference operation by operation --------------------------------------------
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }

// num-complex Mul (ac-bd, ad+bc) in that arithmetic (simd_extensions/fallback.rs:195-203)
template <typename C> __device__ __forceinline__ C cmul_nofma(C a, C b) {
    C r;
    r.x = sub_rn(mul_rn(a.x, b.x), mul_rn(a.y, b.y));
    r.y = add_rn(mul_rn(a.x, b.y), mul_rn(a.y, b.x));
    return r;
}
// num-complex Div (a * conj(b)) / |b|^2 in that arithmetic
template <typename C> __device__ __forceinline__ C cdiv_nofma(C a, C b) {
    const auto ns = add_rn(mul_rn(b.x, b.x), mul_rn(b.y, b.y));
    const auto re = add_rn(mul_rn(a.x, b.x), mul_rn(a.y, b.y));
    const auto im = sub_rn(mul_rn(a.y, b.x), mul_rn(a.x, b.y));
    C r;
    r.x = div_rn(re, ns);
    r.y = div_rn(im, ns);
    return r;
}

__device__ __forceinline__ void sincospi_t(float x, float* s, float* c) { sincospif(x, s, c); }
__device__ __forceinline__ void sincospi_t(double x, double* s, double* c) { sincospi(x, s, c); }

// kernel attributes (dynamic shared memory size, carve-out) belong to the function IN ONE DEVICE'S context: launchers
// configure once per device, not once per process (a process may drive several devices through bdsp_set_device)
struct PerDeviceOnce {
    bool done[64] = {};
    int dev = 0;
    bool need() { if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { dev = -1; return true; } return !done[dev]; }
    void mark() { if (dev >= 0) done[dev] = true; }
};

// --- programmatic dependent launch (sm_90+): a kernel launched with launch_pdl() may become resident while the previous
// kernel of the stream is still draining; pdl_wait() (griddepcontrol.wait) blocks until that kernel has completed and its
// memory is visible, and must precede the first global access.  pdl_trigger() lets the NEXT kernel start its launch early.
// Hides the 2-3 us launch latency between the short kernels of single-vector operation chains.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// --- multiplier fused into the first load of a transform (FftOpts::in_mul) ------------------
// kind 0: none; 1: table of n real scalars T; 2: table of n complex values; 3: built-in window `arg` (0 triangular,
// 1 Hamming, 2 Blackman-Harris, else rectangular) of length n (window_functions.rs:25-129, symmetric evaluation of
// vector_types/mod.rs:528-598), which fft_exec writes into a table (4 B/point, one small kernel) before the transform.  The index is the element's position in its sequence.
struct InMul {
    const void* p = nullptr;
    int kind = 0;
    int arg = 0;
};
template <typename T> __device__ __forceinline__ T window_value_dev(int kind, long long n, long long length) {
    const T one = (T)1, two = (T)2, pi = (T)3.14159265358979323846;
    const T nn = (T)n, ln = (T)length;
    if (kind == 0) return one - fabs((nn - (ln - one) / two) / (ln / two));
    if (kind == 1) { const T alpha = (T)0.54; return alpha - (one - alpha) * cos(two * pi * nn / (ln - one)); }
    if (kind == 2)
        return (T)0.35875 - (T)0.48829 * cos(two * pi * nn / (ln - one)) + (T)0.14128 * cos((T)4 * pi * nn / (ln - one)) -
               (T)0.01168 * cos((T)6 * pi * nn / (ln - one));
    return one;
}
// v * multiplier[g], g = position inside a sequence of n elements
template <typename T>
__device__ __forceinline__ typename CpxOf<T>::type in_mul_apply(typename CpxOf<T>::type v, const void* p, int kind, int arg, long long g, long long n) {
    typedef typename CpxOf<T>::type C;
    if (kind == 1) { const T w = reinterpret_cast<const T*>(p)[g]; v.x *= w; v.y *= w; }
    else if (kind == 2) v = cmul(v, reinterpret_cast<const C*>(p)[g]);
    (void)arg; (void)n;   // kind 3 (built-in window) is materialised as a kind-1 table by fft_exec: no cos() in transform kernels
    return v;
}

// exp(sign * 2*pi*i * num/den), argument reduced exactly in integers first
template <typename T>
__device__ __forceinline__ typename CpxOf<T>::type unit_root(unsigned long long num, unsigned long long den, int sign) {
    num %= den;
    T s, c;
    sincospi_t((T)(2.0 * (double)num / (double)den), &s, &c);
    return mk<T>(c, sign < 0 ? -s : s);
}

int sm_count();

// grid-stride kernels: blocks of 256 threads for `items` work items, one item per thread up to 16 blocks per SM
constexpr int GRID_STRIDE_THREADS = 256;
inline unsigned grid_stride_blocks(long long items) {
    long long g = (items + GRID_STRIDE_THREADS - 1) / GRID_STRIDE_THREADS;
    const long long cap = (long long)sm_count() * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}
// launches a grid-stride kernel over `items` work items on `st` and counts the launch
template <typename... KArgs, typename... Args>
inline int launch_grid_stride(void (*kernel)(KArgs...), long long items, cudaStream_t st, Args... args) {
    kernel<<<grid_stride_blocks(items), GRID_STRIDE_THREADS, 0, st>>>(args...);
    BDSP_LAUNCHED();
    return 0;
}

static inline int ilog2(size_t v) {
    int l = 0;
    while ((1ull << (l + 1)) <= v) l++;
    return l;
}
static inline bool is_pow2(size_t v) { return v && !(v & (v - 1)); }
static inline size_t next_pow2(size_t v) {
    size_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace bdsp
