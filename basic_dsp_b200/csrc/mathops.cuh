// Elementwise math family + reductions of the reference's C facade (see mathops.cu / reduce.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace bdsp {

enum MathOp {
    M_SIN, M_COS, M_TAN, M_ASIN, M_ACOS, M_ATAN, M_SINH, M_COSH, M_TANH, M_ASINH, M_ACOSH, M_ATANH,
    M_SQRT, M_SQUARE, M_LN, M_EXP, M_ABS, M_POWF, M_LOG, M_EXPF, M_WRAP
};

// in place; elems = scalars (real) or points (complex)
template <typename T> int math_unary(int op, void* data, size_t elems, int is_complex, double arg, cudaStream_t st);
template <typename T> int math_unwrap(void* data, size_t n, double divisor, cudaStream_t st);
template <typename T> int math_diff(const void* in, void* out, size_t n_out_scalars, int step, int with_start, cudaStream_t st);
size_t math_cumsum_workspace(size_t points, int lanes, size_t elem_size);
template <typename T> int math_cumsum(const void* in, void* out, void* work, size_t points, int lanes, cudaStream_t st);
// op: EW_ADD, EW_SUB, EW_MUL or EW_DIV (elementwise.cuh); operand element i % w_points
template <typename T> int math_binary_smaller(int op, void* data, const void* w, size_t points, size_t w_points, int is_complex, cudaStream_t st);
template <typename T> int math_split_merge(void* whole, void* const* parts, int nparts, size_t elems, int esz, int merge, cudaStream_t st);
template <typename T> int math_compose(const void* a, const void* b, void* out, size_t points, int polar, cudaStream_t st);
template <typename T> int math_hermite(const void* x, void* y, size_t n, size_t dest_len, size_t start, double factor, double delay, cudaStream_t st);

// ---- reductions (reduce.cu) ----------------------------------------------------------------------------
// Statistics<T> / Statistics<Complex<T>> of the reference (statistics.rs:11-31), #[repr(C)]
template <typename V> struct StatsOut {
    V sum; size_t count; V average; V rms; V min; size_t min_index; V max; size_t max_index;
};
struct Cpx32 { float re, im; };
struct Cpx64 { double re, im; };

// sums[0..1] = sum (re, im), sums[2..3] = sum of squares; accumulated in double (f32 input) or with
// compensated (Kahan / two-sum) double arithmetic (`prec` and f64 input); results in double
template <typename T> int reduce_sums(const void* data, size_t elems, int is_complex, int prec, double* host_out4, cudaStream_t st);
// sum(a[i] * b[i]) (complex product without conjugation); result (re, im) in double
template <typename T> int reduce_dot(const void* a, const void* b, size_t elems, int is_complex, int prec, double* host_out2, cudaStream_t st);
// statistics of `parts` interleaved sub-sequences (element j -> part j % parts, index j / parts); parts <= 16
// out: per part {sum re, sum im, sumsq re, sumsq im, min re, min im, max re, max im} + indices + counts
struct StatsRaw { double sum[2], sumsq[2], min[2], max[2]; unsigned long long min_index, max_index, count; };
template <typename T> int reduce_stats(const void* data, size_t elems, int is_complex, int parts, int prec, StatsRaw* host_out, cudaStream_t st);

}  // namespace bdsp
