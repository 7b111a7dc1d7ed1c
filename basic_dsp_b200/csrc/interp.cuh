// Interpolation entry points (device pointers), see interp.cu.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace bdsp {

// tab_dev: [2][F][2L+3] tap tables (interior, edge) built by the host, see capi.cu interp_tap_tables()
template <typename T>
int interp_poly(const void* x, void* y, const T* tab_dev, size_t N, size_t new_points, int F, int L, int is_complex,
                cudaStream_t st);
// non-integer factor, built-in impulse responses only (kind 0 = Sinc, else RaisedCosine(rolloff))
template <typename T>
int interp_frac(const void* x, void* y, size_t N, size_t new_points, double factor, double delay, int L, int kind,
                double rolloff, int is_complex, cudaStream_t st);
template <typename T>
int interp_lin(const void* x, void* y, size_t n, size_t dest_len, double factor, double delay, cudaStream_t st);

}  // namespace bdsp
