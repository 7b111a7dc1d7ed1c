// Convolution entry points (device pointers), see conv.cu.
#pragma once
#include "common.cuh"

namespace bdsp {

// Overlap-save plan of one impulse response (the reference recomputes this spectrum inside every
// convolve_signal call, convolution.rs:333-339,419-425).  Immutable after ols_plan_create, so any number of
// threads / streams of the creating device may convolve with it concurrently.  Destruction synchronises the device.
struct OlsPlan {
    int is64 = 0, device = 0, h_is_real = 0;
    size_t L = 0;
    // primary block: M points; Hs = FFT_M(pad(h))/M in natural order (M complex) followed, for the fused c32 kernels
    // (M = 4096 / 8192), by the same spectrum in the kernel's layout (2*M floats), bound to a texture object
    size_t M = 0;
    void* Hs = nullptr;
    cudaTextureObject_t htex = 0;
    // c32, 2 <= L <= 2046: second fused block length (8192) next to M = 4096; chosen per call from the amount of work
    size_t M2 = 0;
    void* Hs2 = nullptr;
    cudaTextureObject_t htex2 = 0;
};
// h: L complex (or real) taps on the device.  complex_signal: the vectors that will be convolved are complex.
template <typename T> OlsPlan* ols_plan_create(const void* h, size_t L, int h_is_real, bool complex_signal, cudaStream_t st);
void ols_plan_destroy(OlsPlan* p);

// true where convolve() runs overlap-save blocks and so needs a plan of h
template <typename T> bool conv_needs_plan(size_t L, int h_is_real);
// y <- centred circular convolution y[i] = sum_{k<L} x[(i + cl - 1 - k) mod N] h[k], cl = L - L/2, of every one of
// `batch` vectors of N points (x != y) with the L taps h (device).  Chooses the direct FIR, an overlap-save kernel or
// the full-length FFT path.  `plan` is required when conv_needs_plan<T>(L, h_is_real), otherwise ignored: the plan of
// these taps, made for complex signals when x_is_real is 0 and for real ones otherwise.  h must stay valid until the
// call's kernels have run.
template <typename T>
int convolve(const void* x, void* y, size_t N, size_t batch, int x_is_real, const void* h, size_t L, int h_is_real,
             const OlsPlan* plan, cudaStream_t st);

}  // namespace bdsp
