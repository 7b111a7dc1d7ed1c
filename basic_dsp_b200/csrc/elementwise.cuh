// Elementwise entry points (device pointers), see elementwise.cu.
#pragma once
#include "common.cuh"

namespace bdsp {

enum { EW_SCALE = 0, EW_OFFSET = 1, EW_CONJ = 2, EW_ADD = 3, EW_SUB = 4, EW_MUL = 5, EW_DIV = 6 };
enum { C2R_MAG_HYPOT = 0, C2R_MAG_SQRT = 1, C2R_MAG_SQ = 2, C2R_PHASE = 3, C2R_REAL = 4, C2R_IMAG = 5 };

// a OP b for OP in EW_ADD .. EW_DIV, as the reference's CPU path computes it: on real values, and on complex values
// (float2 / double2) with the num-complex formulas
template <int OP, typename T> __device__ __forceinline__ T ew_real_op(T a, T b) {
    if (OP == EW_ADD) return add_rn(a, b);
    if (OP == EW_SUB) return sub_rn(a, b);
    if (OP == EW_MUL) return mul_rn(a, b);
    return div_rn(a, b);
}
template <int OP, typename C> __device__ __forceinline__ C ew_complex_op(C a, C b) {
    if (OP == EW_MUL) return cmul_nofma(a, b);
    if (OP == EW_DIV) return cdiv_nofma(a, b);
    a.x = ew_real_op<OP>(a.x, b.x);
    a.y = ew_real_op<OP>(a.y, b.y);
    return a;
}

template <typename T> int ew_scalar(int op, const void* in, void* out, size_t n_scalars, double c, cudaStream_t st);
template <typename T> int ew_complex_const(int op, const void* in, void* out, size_t points, double re, double im, cudaStream_t st);
template <typename T> int ew_binary(int op, const void* a, const void* b, void* out, size_t n_scalars, int is_complex, cudaStream_t st);
template <typename T> int ew_complex_to_real(int op, const void* in, void* out, size_t points, cudaStream_t st);
template <typename T> int ew_mag_phase(const void* in, void* mag, void* phase, size_t points, cudaStream_t st);
template <typename T>
int ew_scale_mul_mag_phase(void* v, const void* w, void* mag, void* phase, size_t points, double cre, double cim,
                           int complex_scale, int write_v, cudaStream_t st);
template <typename T> int ew_rotate(const void* in, void* out, size_t n_elems, size_t rot, int esz, cudaStream_t st);
template <typename T> int ew_zero_interleave(const void* in, void* out, size_t n_elems, int factor, int esz, cudaStream_t st);
template <typename T> int ew_fill(void* out, size_t n, double v, cudaStream_t st);
template <typename T> int ew_reverse(const void* in, void* out, size_t n_elems, int esz, cudaStream_t st);
template <typename T> int ew_decimate(const void* in, void* out, size_t out_elems, size_t factor, size_t delay, int esz, cudaStream_t st);
template <typename T> int ew_mul_freq_resp(void* data, size_t points, int is_complex, int kind, double rolloff, double ratio, cudaStream_t st);
// table == nullptr and resp_kind >= 0: built-in frequency response (0 sinc, 1 raised cosine) evaluated on the device
template <typename T> int ew_resample_spectrum(const void* in, void* out, size_t n, size_t dest, const void* table, double scale, int use_scale,
                                               double phase_inc, int use_phase, int resp_kind, double resp_rolloff, double resp_ratio, cudaStream_t st);
template <typename T> int ew_mul_shifted_resp(void* data, size_t points, int kind, double rolloff, double ratio, cudaStream_t st);
template <typename T> int ew_mirror(const void* in, void* out, size_t points, cudaStream_t st);
template <typename T> int ew_mul_cexp(void* data, size_t points, double a, double b, cudaStream_t st);
template <typename T> int ew_window(void* data, size_t points, int is_complex, int kind, int unapply, cudaStream_t st);
template <typename T> int ew_mul_table(void* data, const void* table, size_t points, int is_complex, int table_complex, cudaStream_t st);
// x[r * n + i] *= h[i] * scale for `rows` rows of n complex points: the spectrum product of a fast convolution
template <typename T> int ew_spectrum_mul_rows(void* x, const void* h, size_t n, size_t rows, double scale, cudaStream_t st);

}  // namespace bdsp
