/*
 * basic_dsp_b200 - C ABI of the B200-native (sm_100a) implementation of basic_dsp's FFT-centred
 * vector hot path.  The library is a drop-in for the hot-path subset of the reference's `interop`
 * crate: every function in section 1 has the name, argument order, return struct and error codes of
 * the `#[no_mangle] extern "C"` function it replaces (cited as file:line in the reference tree,
 * liebharc/basic_dsp v0.10.0).  `...64` variants are identical with f32 -> f64
 * (interop/src/facade64.rs is generated from facade32.rs by facade64_create.pl).
 *
 * Differences a caller must know about (all documented in INTEGRATION.md):
 *   - A vector handle owns DEVICE memory (HBM).  `data32`/`complex_data32` return a pointer to a
 *     host mirror that is refreshed by that call (device -> host copy + sync); writing through it
 *     does not change the vector.  Use bdsp_upload32/bdsp_download32 for bulk transfers.
 *   - plain_ifft32/ifft32 return a vector in the TIME domain (the reference leaves the domain tag of
 *     a GenDspVec at Frequency, SURVEY.md Q2).
 *   - Custom impulse-response callbacks are evaluated on the host to build tap tables; they are not
 *     supported by interpolatef_custom32 for non-integer factors (returns error 7).
 *   - There is no CPU fallback: every compute entry point fails with a negative code when no CUDA
 *     device is usable.
 *
 * Result codes (interop/src/lib.rs:107-151): 0 ok; -1 vector is in the error state (wrong
 * real/complex or time/freq for the operation); 1 same size; 2 meta data; 3 must be complex; 4 must
 * be real; 5 must be time domain; 6 must be frequency domain; 7 invalid argument length; 8 conj
 * symmetric; 9 odd length; 10 symmetric function; 11 combined-op arguments; 12 not empty; 13 even
 * length; 14 cannot resize.  Codes <= -1000 are CUDA errors (-(1000 + cudaError_t)); see
 * bdsp_last_error().
 */
#ifndef BASIC_DSP_B200_H
#define BASIC_DSP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

/* Opaque handles: InteropVec<f32> / InteropVec<f64> (interop/src/lib.rs:16-22). */
typedef struct BdspVec32 BdspVec32;
typedef struct BdspVec64 BdspVec64;

/* VectorInteropResult (interop/src/lib.rs:203-212): the vector handle is taken by value and handed
 * back; callers continue with the returned pointer. */
typedef struct { int32_t result_code; BdspVec32* vector; } BdspVecResult32;
typedef struct { int32_t result_code; BdspVec64* vector; } BdspVecResult64;

typedef struct { float re, im; } BdspComplex32;
typedef struct { double re, im; } BdspComplex64;

/* Callback types of the *_real / *_complex / *_custom entry points (interop/src/lib.rs:279-377). */
/* Statistics<T> (vector/src/vector_types/general/statistics.rs:11-31, #[repr(C)]) and the scalar results of
 * interop/src/lib.rs:229-242 */
typedef struct { float sum; size_t count; float average; float rms; float min; size_t min_index; float max; size_t max_index; } BdspStatistics32;
typedef struct { double sum; size_t count; double average; double rms; double min; size_t min_index; double max; size_t max_index; } BdspStatistics64;
typedef struct { BdspComplex32 sum; size_t count; BdspComplex32 average; BdspComplex32 rms; BdspComplex32 min; size_t min_index; BdspComplex32 max; size_t max_index; } BdspComplexStatistics32;
typedef struct { BdspComplex64 sum; size_t count; BdspComplex64 average; BdspComplex64 rms; BdspComplex64 min; size_t min_index; BdspComplex64 max; size_t max_index; } BdspComplexStatistics64;
typedef struct { int32_t result_code; const void* result; } BdspPointerResult;
typedef struct { int32_t result_code; float result; } BdspScalarResult32;
typedef struct { int32_t result_code; double result; } BdspScalarResult64;
typedef struct { int32_t result_code; BdspComplex32 result; } BdspComplexScalarResult32;
typedef struct { int32_t result_code; BdspComplex64 result; } BdspComplexScalarResult64;

/* expf32 / powf32 / expf64 / powf64 are also names of glibc's _Float32 / _Float64 functions (<math.h> with
 * _GNU_SOURCE).  The library exports the reference's symbol names; C and C++ callers use the bdsp_-prefixed
 * declarations below, which bind to those symbols. */
#if defined(__GNUC__)
#define BDSP_SYMBOL(name) __asm__(name)
#else
#define BDSP_SYMBOL(name)
#endif

typedef float (*BdspRealFn32)(const void* data, float x);
typedef double (*BdspRealFn64)(const void* data, double x);
typedef BdspComplex32 (*BdspComplexFn32)(const void* data, float x);
/* ForeignWindowFunction (interop/src/lib.rs): window(data, index, points) */
typedef float (*BdspWindowFn32)(const void* data, size_t i, size_t points);
typedef double (*BdspWindowFn64)(const void* data, size_t i, size_t points);
typedef BdspComplex64 (*BdspComplexFn64)(const void* data, double x);

/* ===================================================================================================
 * 1. Reference C ABI, hot-path subset (interop/src/facade32.rs; f64 twins in facade64.rs)
 * =================================================================================================== */

/* Threading (the reference: re-entrant per handle, interop/src/lib.rs): different threads may work on different
 * vectors at the same time, with or without bdsp_set_stream - scratch workspaces are per host thread.  A vector that is
 * only BORROWED by a call (`const BdspVec32*`, e.g. the impulse response of convolve_signal32) may be shared by several
 * threads; its cached spectrum is built under a lock and reference counted.
 * Errors: no entry point terminates the process.  Constructors return NULL when the device allocation fails
 * (bdsp_last_error() says why); other calls report CUDA failures as result codes <= -1000. */

/* ---- life cycle and meta data -------------------------------------------------------------------- */
BdspVec32* new32(int32_t is_complex, int32_t domain, float init_value, size_t length, float delta);     /* facade32.rs:22 */
BdspVec32* new_with_performance_options32(int32_t is_complex, int32_t domain, float init_value, size_t length,
                                          float delta, size_t core_limit);                                 /* :44, core_limit ignored */
BdspVec32* new_with_detailed_performance_options32(int32_t is_complex, int32_t domain, float init_value, size_t length,
                                                   float delta, size_t core_limit, size_t med_dual_core_threshold,
                                                   size_t med_multi_core_threshold, size_t large_dual_core_threshold,
                                                   size_t large_multi_core_threshold);                     /* :70 */
void delete_vector32(BdspVec32* vector);                                                                   /* :17 */
BdspVec32* clone32(BdspVec32* vector);                                                                     /* :687 (argument is NOT consumed here, unlike the reference which moves it) */
float get_value32(const BdspVec32* vector, size_t index);                                                  /* :105 */
void set_value32(BdspVec32* vector, size_t index, float value);                                            /* :110 */
int32_t is_complex32(const BdspVec32* vector);                                                             /* :115 */
int32_t get_domain32(const BdspVec32* vector);                                                             /* :130, 0 time / 1 frequency */
size_t get_len32(const BdspVec32* vector);                                                                 /* :138 */
void set_len32(BdspVec32* vector, size_t len);                                                             /* :143 */
size_t get_points32(const BdspVec32* vector);                                                              /* :148 */
float get_delta32(const BdspVec32* vector);                                                                /* :153 */
const float* data32(const BdspVec32* vector);                                                              /* :158, host mirror */
const BdspComplex32* complex_data32(const BdspVec32* vector);                                              /* :163, host mirror */
size_t get_allocated_len32(const BdspVec32* vector);                                                       /* :168 */
BdspVecResult32 overwrite_data32(BdspVec32* vector, const float* data, size_t len);                        /* :827, requires len < get_len32 (Q9) */

/* ---- elementwise ------------------------------------------------------------------------------------ */
BdspVecResult32 add32(BdspVec32* vector, const BdspVec32* operand);                                        /* :173 */
BdspVecResult32 sub32(BdspVec32* vector, const BdspVec32* operand);                                        /* :178 */
BdspVecResult32 div32(BdspVec32* vector, const BdspVec32* operand);                                        /* :183 */
BdspVecResult32 mul32(BdspVec32* vector, const BdspVec32* operand);                                        /* :188 */
BdspVecResult32 add_vector32(BdspVec32* vector, const BdspVec32* operand);                                 /* :704 */
BdspVecResult32 sub_vector32(BdspVec32* vector, const BdspVec32* operand);                                 /* :712 */
BdspVecResult32 div_vector32(BdspVec32* vector, const BdspVec32* operand);                                 /* :720 */
BdspVecResult32 mul_vector32(BdspVec32* vector, const BdspVec32* operand);                                 /* :728 */
BdspVecResult32 real_offset32(BdspVec32* vector, float value);                                             /* :363 */
BdspVecResult32 real_scale32(BdspVec32* vector, float value);                                              /* :368 */
BdspVecResult32 complex_offset32(BdspVec32* vector, float real, float imag);                               /* :532 */
BdspVecResult32 complex_scale32(BdspVec32* vector, float real, float imag);                                /* :541 */
BdspVecResult32 complex_divide32(BdspVec32* vector, float real, float imag);                               /* :550 */
BdspVecResult32 conj32(BdspVec32* vector);                                                                 /* :579 */
BdspVecResult32 to_complex32(BdspVec32* vector);                                                           /* :418 */

/* ---- complex -> real ---------------------------------------------------------------------------------- */
BdspVecResult32 magnitude32(BdspVec32* vector);                                                            /* :559 */
BdspVecResult32 magnitude_squared32(BdspVec32* vector);                                                    /* :574 */
BdspVecResult32 phase32(BdspVec32* vector);                                                                /* :662 */
BdspVecResult32 to_real32(BdspVec32* vector);                                                              /* :584 */
BdspVecResult32 to_imag32(BdspVec32* vector);                                                              /* :589 */
/* The getters return 9 on success (convert_void, interop/src/lib.rs:100-105, Q8).  The reference
 * takes `vector` by value and drops it; here the source vector stays valid and owned by the caller. */
int32_t get_magnitude32(BdspVec32* vector, BdspVec32* destination);                                        /* :564 */
int32_t get_magnitude_squared32(BdspVec32* vector, BdspVec32* destination);                                /* :569 */
int32_t get_phase32(BdspVec32* vector, BdspVec32* destination);                                            /* :667 */
int32_t get_real32(BdspVec32* vector, BdspVec32* destination);                                             /* :652 */
int32_t get_imag32(BdspVec32* vector, BdspVec32* destination);                                             /* :657 */
int32_t get_mag_phase32(BdspVec32* vector, BdspVec32* mag, BdspVec32* phase);                              /* :777 */

/* ---- transforms -------------------------------------------------------------------------------------------- */
BdspVecResult32 plain_fft32(BdspVec32* vector);                                                            /* :672 */
BdspVecResult32 plain_ifft32(BdspVec32* vector);                                                           /* :682 */
BdspVecResult32 fft32(BdspVec32* vector);                                                                  /* :934 */
BdspVecResult32 ifft32(BdspVec32* vector);                                                                 /* :944 */
BdspVecResult32 swap_halves32(BdspVec32* vector);                                                          /* :527 */
BdspVecResult32 fft_shift32(BdspVec32* vector);                                                            /* :963 (not exported by the reference: missing #[no_mangle], Q10) */
BdspVecResult32 ifft_shift32(BdspVec32* vector);                                                           /* :967 */
BdspVecResult32 zero_pad32(BdspVec32* vector, size_t points, int32_t padding_option);                      /* :330, 0 End / 1 Surround / 2 Center */
BdspVecResult32 zero_interleave32(BdspVec32* vector, int32_t factor);                                      /* :340 */

/* ---- convolution ---------------------------------------------------------------------------------------------- */
BdspVecResult32 convolve_signal32(BdspVec32* vector, const BdspVec32* impulse_response);                   /* :1171 */
BdspVecResult32 convolve32(BdspVec32* vector, int32_t impulse_response, float rolloff, float ratio, size_t len); /* :1231, 0 Sinc / else RaisedCosine */
BdspVecResult32 convolve_real32(BdspVec32* vector, BdspRealFn32 impulse_response, const void* impulse_response_data,
                                uint8_t is_symmetric, float ratio, size_t len);                            /* :1183 */
BdspVecResult32 convolve_complex32(BdspVec32* vector, BdspComplexFn32 impulse_response, const void* impulse_response_data,
                                   uint8_t is_symmetric, float ratio, size_t len);                         /* :1206 */
BdspVecResult32 multiply_frequency_response32(BdspVec32* vector, int32_t frequency_response, float rolloff, float ratio); /* :1293 */
BdspVecResult32 multiply_frequency_response_real32(BdspVec32* vector, BdspRealFn32 frequency_response,
                                                   const void* frequency_response_data, uint8_t is_symmetric, float ratio); /* :1247 */
BdspVecResult32 multiply_frequency_response_complex32(BdspVec32* vector, BdspComplexFn32 frequency_response,
                                                      const void* frequency_response_data, uint8_t is_symmetric, float ratio); /* :1269 */

/* ---- interpolation --------------------------------------------------------------------------------------------- */
BdspVecResult32 interpolatef32(BdspVec32* vector, int32_t impulse_response, float rolloff, float interpolation_factor,
                               float delay, size_t len);                                                   /* :1334 */
BdspVecResult32 interpolatef_custom32(BdspVec32* vector, BdspRealFn32 impulse_response, const void* impulse_response_data,
                                      uint8_t is_symmetric, float interpolation_factor, float delay, size_t len); /* :1308 */
BdspVecResult32 interpolate_lin32(BdspVec32* vector, float interpolation_factor, float delay);             /* :1437 */

/* ---- next rows of the scope table (SURVEY.md 8f): windows, correlation ("preparation" API), reverse, decimatei --- */
BdspVecResult32 apply_window32(BdspVec32* vector, int32_t window);       /* :980, 0 Triangular / 1 Hamming / 2 BlackmanHarris / else Rectangular */
BdspVecResult32 unapply_window32(BdspVec32* vector, int32_t window);     /* :987 */
BdspVecResult32 windowed_fft32(BdspVec32* vector, int32_t window);       /* :997 */
BdspVecResult32 windowed_ifft32(BdspVec32* vector, int32_t window);      /* :1011 */
BdspVecResult32 prepare_argument32(BdspVec32* vector);                   /* :1156 */
BdspVecResult32 prepare_argument_padded32(BdspVec32* vector);            /* :1161 */
BdspVecResult32 correlate32(BdspVec32* vector, const BdspVec32* other);  /* :1166 */
BdspVecResult32 reverse32(BdspVec32* vector);                            /* :1142 */
BdspVecResult32 decimatei32(BdspVec32* vector, uint32_t decimation_factor, uint32_t delay); /* :1147 */
BdspVecResult32 interpolatei32(BdspVec32* vector, int32_t frequency_response, float rolloff, int32_t interpolation_factor); /* :1426 */
BdspVecResult32 interpolatei_custom32(BdspVec32* vector, BdspRealFn32 frequency_response, const void* frequency_response_data,
                                      uint8_t is_symmetric, int32_t interpolation_factor);     /* :1402 */

/* FFT-based resampling, symmetric (real <-> half spectrum) transforms, complex exponential */
BdspVecResult32 interpolate32(BdspVec32* vector, int32_t frequency_response, float rolloff, size_t dest_points, float delay); /* :1379 */
BdspVecResult32 interpolate_custom32(BdspVec32* vector, BdspRealFn32 frequency_response, const void* frequency_response_data,
                                     uint8_t is_symmetric, size_t dest_points, float delay);   /* :1353 */
BdspVecResult32 interpft32(BdspVec32* vector, size_t dest_points);       /* :1390 */
BdspVecResult32 multiply_complex_exponential32(BdspVec32* vector, float a, float b); /* :695 */
BdspVecResult32 mirror32(BdspVec32* vector);                             /* :959 */
BdspVecResult32 plain_sfft32(BdspVec32* vector);                         /* :677; odd real length n -> (n + 1) / 2 bins */
BdspVecResult32 sfft32(BdspVec32* vector);                               /* :939 */
BdspVecResult32 windowed_sfft32(BdspVec32* vector, int32_t window);      /* :1004 */
BdspVecResult32 plain_sifft32(BdspVec32* vector);                        /* :949; result code 8 unless Im X[0] == 0 */
BdspVecResult32 sifft32(BdspVec32* vector);                              /* :954 */
BdspVecResult32 windowed_sifft32(BdspVec32* vector, int32_t window);     /* :1018 */

/* ---- rest of the C facade (SURVEY.md 8f row 4): elementwise math, reorganisation, reductions ----
 * (interop/src/facade32.rs:193-321 reductions, :348-524 math, :736-824 reorganisation, :848-931 split statistics,
 * :1030-1139 custom windows, :1446 hermite).  map_inplace_* / map_aggregate_* (:594-647) call a host function per element:
 * the vector is staged through host memory for them. */
BdspVecResult32 sin32(BdspVec32* vector);
BdspVecResult32 cos32(BdspVec32* vector);
BdspVecResult32 tan32(BdspVec32* vector);
BdspVecResult32 asin32(BdspVec32* vector);
BdspVecResult32 acos32(BdspVec32* vector);
BdspVecResult32 atan32(BdspVec32* vector);
BdspVecResult32 sinh32(BdspVec32* vector);
BdspVecResult32 cosh32(BdspVec32* vector);
BdspVecResult32 tanh32(BdspVec32* vector);
BdspVecResult32 asinh32(BdspVec32* vector);
BdspVecResult32 acosh32(BdspVec32* vector);
BdspVecResult32 atanh32(BdspVec32* vector);
BdspVecResult32 sqrt32(BdspVec32* vector);
BdspVecResult32 square32(BdspVec32* vector);
BdspVecResult32 ln32(BdspVec32* vector);
BdspVecResult32 exp32(BdspVec32* vector);
BdspVecResult32 abs32(BdspVec32* vector);
BdspVecResult32 ln_approx32(BdspVec32* vector);
BdspVecResult32 exp_approx32(BdspVec32* vector);
BdspVecResult32 sin_approx32(BdspVec32* vector);
BdspVecResult32 cos_approx32(BdspVec32* vector);
BdspVecResult32 diff32(BdspVec32* vector);
BdspVecResult32 diff_with_start32(BdspVec32* vector);
BdspVecResult32 cum_sum32(BdspVec32* vector);
BdspVecResult32 root32(BdspVec32* vector, float degree);
BdspVecResult32 log32(BdspVec32* vector, float base);
BdspVecResult32 wrap32(BdspVec32* vector, float divisor);
BdspVecResult32 unwrap32(BdspVec32* vector, float divisor);
BdspVecResult32 log_approx32(BdspVec32* vector, float base);
BdspVecResult32 expf_approx32(BdspVec32* vector, float base);
BdspVecResult32 powf_approx32(BdspVec32* vector, float exponent);
BdspVecResult32 bdsp_powf32(BdspVec32* vector, float exponent) BDSP_SYMBOL("powf32");
BdspVecResult32 bdsp_expf32(BdspVec32* vector, float base) BDSP_SYMBOL("expf32");
BdspVecResult32 add_smaller_vector32(BdspVec32* vector, const BdspVec32* operand);
BdspVecResult32 sub_smaller_vector32(BdspVec32* vector, const BdspVec32* operand);
BdspVecResult32 mul_smaller_vector32(BdspVec32* vector, const BdspVec32* operand);
BdspVecResult32 div_smaller_vector32(BdspVec32* vector, const BdspVec32* operand);
int32_t get_real_imag32(BdspVec32* vector, BdspVec32* real, BdspVec32* imag);
BdspVecResult32 set_real_imag32(BdspVec32* vector, const BdspVec32* real, const BdspVec32* imag);
BdspVecResult32 set_mag_phase32(BdspVec32* vector, const BdspVec32* mag, const BdspVec32* phase);
int32_t split_into32(const BdspVec32* vector, BdspVec32** targets, size_t len);
BdspVecResult32 merge32(BdspVec32* vector, BdspVec32* const* sources, size_t len);
BdspVecResult32 interpolate_hermite32(BdspVec32* vector, float interpolation_factor, float delay);
BdspVecResult32 map_inplace_real32(BdspVec32* vector, float (*map)(float value, size_t index));
BdspVecResult32 map_inplace_complex32(BdspVec32* vector, BdspComplex32 (*map)(BdspComplex32 value, size_t index));
BdspPointerResult map_aggregate_real32(const BdspVec32* vector, const void* (*map)(float value, size_t index),
                                       const void* (*aggregate)(const void* a, const void* b));
BdspPointerResult map_aggregate_complex32(const BdspVec32* vector, const void* (*map)(BdspComplex32 value, size_t index),
                                          const void* (*aggregate)(const void* a, const void* b));
BdspVecResult32 apply_custom_window32(BdspVec32* vector, BdspWindowFn32 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult32 unapply_custom_window32(BdspVec32* vector, BdspWindowFn32 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult32 windowed_custom_fft32(BdspVec32* vector, BdspWindowFn32 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult32 windowed_custom_ifft32(BdspVec32* vector, BdspWindowFn32 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult32 windowed_custom_sfft32(BdspVec32* vector, BdspWindowFn32 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult32 windowed_custom_sifft32(BdspVec32* vector, BdspWindowFn32 window, const void* window_data, uint8_t is_symmetric);
BdspScalarResult32 real_dot_product32(const BdspVec32* vector, const BdspVec32* operand);
BdspScalarResult32 real_dot_product_prec32(const BdspVec32* vector, const BdspVec32* operand);
BdspComplexScalarResult32 complex_dot_product32(const BdspVec32* vector, const BdspVec32* operand);
BdspComplexScalarResult32 complex_dot_product_prec32(const BdspVec32* vector, const BdspVec32* operand);
float real_sum32(const BdspVec32* vector);
float real_sum_sq32(const BdspVec32* vector);
BdspComplex32 complex_sum32(const BdspVec32* vector);
BdspComplex32 complex_sum_sq32(const BdspVec32* vector);
double real_sum_prec32(const BdspVec32* vector);
double real_sum_sq_prec32(const BdspVec32* vector);
BdspComplex64 complex_sum_prec32(const BdspVec32* vector);
BdspComplex64 complex_sum_sq_prec32(const BdspVec32* vector);
BdspStatistics32 real_statistics32(const BdspVec32* vector);
BdspComplexStatistics32 complex_statistics32(const BdspVec32* vector);
BdspStatistics64 real_statistics_prec32(const BdspVec32* vector);
BdspComplexStatistics64 complex_statistics_prec32(const BdspVec32* vector);
int32_t real_statistics_split32(const BdspVec32* vector, BdspStatistics32* data, size_t len);
int32_t complex_statistics_split32(const BdspVec32* vector, BdspComplexStatistics32* data, size_t len);
int32_t real_statistics_split_prec32(const BdspVec32* vector, BdspStatistics64* data, size_t len);
int32_t complex_statistics_split_prec32(const BdspVec32* vector, BdspComplexStatistics64* data, size_t len);

/* ---- f64 twins (interop/src/facade64.rs, same line numbers + 1) ------------------------------------------------ */
BdspVecResult64 apply_window64(BdspVec64* vector, int32_t window);
BdspVecResult64 unapply_window64(BdspVec64* vector, int32_t window);
BdspVecResult64 windowed_fft64(BdspVec64* vector, int32_t window);
BdspVecResult64 windowed_ifft64(BdspVec64* vector, int32_t window);
BdspVecResult64 prepare_argument64(BdspVec64* vector);
BdspVecResult64 prepare_argument_padded64(BdspVec64* vector);
BdspVecResult64 correlate64(BdspVec64* vector, const BdspVec64* other);
BdspVecResult64 reverse64(BdspVec64* vector);
BdspVecResult64 decimatei64(BdspVec64* vector, uint32_t decimation_factor, uint32_t delay);
BdspVecResult64 interpolatei64(BdspVec64* vector, int32_t frequency_response, double rolloff, int32_t interpolation_factor);
BdspVecResult64 interpolatei_custom64(BdspVec64* vector, BdspRealFn64 frequency_response, const void* frequency_response_data,
                                      uint8_t is_symmetric, int32_t interpolation_factor);

BdspVecResult64 interpolate64(BdspVec64* vector, int32_t frequency_response, double rolloff, size_t dest_points, double delay);
BdspVecResult64 interpolate_custom64(BdspVec64* vector, BdspRealFn64 frequency_response, const void* frequency_response_data,
                                     uint8_t is_symmetric, size_t dest_points, double delay);
BdspVecResult64 interpft64(BdspVec64* vector, size_t dest_points);
BdspVecResult64 multiply_complex_exponential64(BdspVec64* vector, double a, double b);
BdspVecResult64 mirror64(BdspVec64* vector);
BdspVecResult64 plain_sfft64(BdspVec64* vector);
BdspVecResult64 sfft64(BdspVec64* vector);
BdspVecResult64 windowed_sfft64(BdspVec64* vector, int32_t window);
BdspVecResult64 plain_sifft64(BdspVec64* vector);
BdspVecResult64 sifft64(BdspVec64* vector);
BdspVecResult64 windowed_sifft64(BdspVec64* vector, int32_t window);
BdspVecResult64 sin64(BdspVec64* vector);
BdspVecResult64 cos64(BdspVec64* vector);
BdspVecResult64 tan64(BdspVec64* vector);
BdspVecResult64 asin64(BdspVec64* vector);
BdspVecResult64 acos64(BdspVec64* vector);
BdspVecResult64 atan64(BdspVec64* vector);
BdspVecResult64 sinh64(BdspVec64* vector);
BdspVecResult64 cosh64(BdspVec64* vector);
BdspVecResult64 tanh64(BdspVec64* vector);
BdspVecResult64 asinh64(BdspVec64* vector);
BdspVecResult64 acosh64(BdspVec64* vector);
BdspVecResult64 atanh64(BdspVec64* vector);
BdspVecResult64 sqrt64(BdspVec64* vector);
BdspVecResult64 square64(BdspVec64* vector);
BdspVecResult64 ln64(BdspVec64* vector);
BdspVecResult64 exp64(BdspVec64* vector);
BdspVecResult64 abs64(BdspVec64* vector);
BdspVecResult64 ln_approx64(BdspVec64* vector);
BdspVecResult64 exp_approx64(BdspVec64* vector);
BdspVecResult64 sin_approx64(BdspVec64* vector);
BdspVecResult64 cos_approx64(BdspVec64* vector);
BdspVecResult64 diff64(BdspVec64* vector);
BdspVecResult64 diff_with_start64(BdspVec64* vector);
BdspVecResult64 cum_sum64(BdspVec64* vector);
BdspVecResult64 root64(BdspVec64* vector, double degree);
BdspVecResult64 log64(BdspVec64* vector, double base);
BdspVecResult64 wrap64(BdspVec64* vector, double divisor);
BdspVecResult64 unwrap64(BdspVec64* vector, double divisor);
BdspVecResult64 log_approx64(BdspVec64* vector, double base);
BdspVecResult64 expf_approx64(BdspVec64* vector, double base);
BdspVecResult64 powf_approx64(BdspVec64* vector, double exponent);
BdspVecResult64 bdsp_powf64(BdspVec64* vector, double exponent) BDSP_SYMBOL("powf64");
BdspVecResult64 bdsp_expf64(BdspVec64* vector, double base) BDSP_SYMBOL("expf64");
BdspVecResult64 add_smaller_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 sub_smaller_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 mul_smaller_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 div_smaller_vector64(BdspVec64* vector, const BdspVec64* operand);
int32_t get_real_imag64(BdspVec64* vector, BdspVec64* real, BdspVec64* imag);
BdspVecResult64 set_real_imag64(BdspVec64* vector, const BdspVec64* real, const BdspVec64* imag);
BdspVecResult64 set_mag_phase64(BdspVec64* vector, const BdspVec64* mag, const BdspVec64* phase);
int32_t split_into64(const BdspVec64* vector, BdspVec64** targets, size_t len);
BdspVecResult64 merge64(BdspVec64* vector, BdspVec64* const* sources, size_t len);
BdspVecResult64 interpolate_hermite64(BdspVec64* vector, double interpolation_factor, double delay);
BdspVecResult64 map_inplace_real64(BdspVec64* vector, double (*map)(double value, size_t index));
BdspVecResult64 map_inplace_complex64(BdspVec64* vector, BdspComplex64 (*map)(BdspComplex64 value, size_t index));
BdspPointerResult map_aggregate_real64(const BdspVec64* vector, const void* (*map)(double value, size_t index),
                                       const void* (*aggregate)(const void* a, const void* b));
BdspPointerResult map_aggregate_complex64(const BdspVec64* vector, const void* (*map)(BdspComplex64 value, size_t index),
                                          const void* (*aggregate)(const void* a, const void* b));
BdspVecResult64 apply_custom_window64(BdspVec64* vector, BdspWindowFn64 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult64 unapply_custom_window64(BdspVec64* vector, BdspWindowFn64 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult64 windowed_custom_fft64(BdspVec64* vector, BdspWindowFn64 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult64 windowed_custom_ifft64(BdspVec64* vector, BdspWindowFn64 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult64 windowed_custom_sfft64(BdspVec64* vector, BdspWindowFn64 window, const void* window_data, uint8_t is_symmetric);
BdspVecResult64 windowed_custom_sifft64(BdspVec64* vector, BdspWindowFn64 window, const void* window_data, uint8_t is_symmetric);
BdspScalarResult64 real_dot_product64(const BdspVec64* vector, const BdspVec64* operand);
BdspScalarResult64 real_dot_product_prec64(const BdspVec64* vector, const BdspVec64* operand);
BdspComplexScalarResult64 complex_dot_product64(const BdspVec64* vector, const BdspVec64* operand);
BdspComplexScalarResult64 complex_dot_product_prec64(const BdspVec64* vector, const BdspVec64* operand);
double real_sum64(const BdspVec64* vector);
double real_sum_sq64(const BdspVec64* vector);
BdspComplex64 complex_sum64(const BdspVec64* vector);
BdspComplex64 complex_sum_sq64(const BdspVec64* vector);
double real_sum_prec64(const BdspVec64* vector);
double real_sum_sq_prec64(const BdspVec64* vector);
BdspComplex64 complex_sum_prec64(const BdspVec64* vector);
BdspComplex64 complex_sum_sq_prec64(const BdspVec64* vector);
BdspStatistics64 real_statistics64(const BdspVec64* vector);
BdspComplexStatistics64 complex_statistics64(const BdspVec64* vector);
BdspStatistics64 real_statistics_prec64(const BdspVec64* vector);
BdspComplexStatistics64 complex_statistics_prec64(const BdspVec64* vector);
int32_t real_statistics_split64(const BdspVec64* vector, BdspStatistics64* data, size_t len);
int32_t complex_statistics_split64(const BdspVec64* vector, BdspComplexStatistics64* data, size_t len);
int32_t real_statistics_split_prec64(const BdspVec64* vector, BdspStatistics64* data, size_t len);
int32_t complex_statistics_split_prec64(const BdspVec64* vector, BdspComplexStatistics64* data, size_t len);
BdspVec64* new64(int32_t is_complex, int32_t domain, double init_value, size_t length, double delta);
BdspVec64* new_with_performance_options64(int32_t is_complex, int32_t domain, double init_value, size_t length, double delta, size_t core_limit);
BdspVec64* new_with_detailed_performance_options64(int32_t is_complex, int32_t domain, double init_value, size_t length,
                                                   double delta, size_t core_limit, size_t med_dual_core_threshold,
                                                   size_t med_multi_core_threshold, size_t large_dual_core_threshold,
                                                   size_t large_multi_core_threshold);
void delete_vector64(BdspVec64* vector);
BdspVec64* clone64(BdspVec64* vector);
double get_value64(const BdspVec64* vector, size_t index);
void set_value64(BdspVec64* vector, size_t index, double value);
int32_t is_complex64(const BdspVec64* vector);
int32_t get_domain64(const BdspVec64* vector);
size_t get_len64(const BdspVec64* vector);
void set_len64(BdspVec64* vector, size_t len);
size_t get_points64(const BdspVec64* vector);
double get_delta64(const BdspVec64* vector);
const double* data64(const BdspVec64* vector);
const BdspComplex64* complex_data64(const BdspVec64* vector);
size_t get_allocated_len64(const BdspVec64* vector);
BdspVecResult64 overwrite_data64(BdspVec64* vector, const double* data, size_t len);
BdspVecResult64 add64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 sub64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 div64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 mul64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 add_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 sub_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 div_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 mul_vector64(BdspVec64* vector, const BdspVec64* operand);
BdspVecResult64 real_offset64(BdspVec64* vector, double value);
BdspVecResult64 real_scale64(BdspVec64* vector, double value);
BdspVecResult64 complex_offset64(BdspVec64* vector, double real, double imag);
BdspVecResult64 complex_scale64(BdspVec64* vector, double real, double imag);
BdspVecResult64 complex_divide64(BdspVec64* vector, double real, double imag);
BdspVecResult64 conj64(BdspVec64* vector);
BdspVecResult64 to_complex64(BdspVec64* vector);
BdspVecResult64 magnitude64(BdspVec64* vector);
BdspVecResult64 magnitude_squared64(BdspVec64* vector);
BdspVecResult64 phase64(BdspVec64* vector);
BdspVecResult64 to_real64(BdspVec64* vector);
BdspVecResult64 to_imag64(BdspVec64* vector);
int32_t get_magnitude64(BdspVec64* vector, BdspVec64* destination);
int32_t get_magnitude_squared64(BdspVec64* vector, BdspVec64* destination);
int32_t get_phase64(BdspVec64* vector, BdspVec64* destination);
int32_t get_real64(BdspVec64* vector, BdspVec64* destination);
int32_t get_imag64(BdspVec64* vector, BdspVec64* destination);
int32_t get_mag_phase64(BdspVec64* vector, BdspVec64* mag, BdspVec64* phase);
BdspVecResult64 plain_fft64(BdspVec64* vector);
BdspVecResult64 plain_ifft64(BdspVec64* vector);
BdspVecResult64 fft64(BdspVec64* vector);
BdspVecResult64 ifft64(BdspVec64* vector);
BdspVecResult64 swap_halves64(BdspVec64* vector);
BdspVecResult64 fft_shift64(BdspVec64* vector);
BdspVecResult64 ifft_shift64(BdspVec64* vector);
BdspVecResult64 zero_pad64(BdspVec64* vector, size_t points, int32_t padding_option);
BdspVecResult64 zero_interleave64(BdspVec64* vector, int32_t factor);
BdspVecResult64 convolve_signal64(BdspVec64* vector, const BdspVec64* impulse_response);
BdspVecResult64 convolve64(BdspVec64* vector, int32_t impulse_response, double rolloff, double ratio, size_t len);
BdspVecResult64 convolve_real64(BdspVec64* vector, BdspRealFn64 impulse_response, const void* impulse_response_data,
                                uint8_t is_symmetric, double ratio, size_t len);
BdspVecResult64 convolve_complex64(BdspVec64* vector, BdspComplexFn64 impulse_response, const void* impulse_response_data,
                                   uint8_t is_symmetric, double ratio, size_t len);
BdspVecResult64 multiply_frequency_response64(BdspVec64* vector, int32_t frequency_response, double rolloff, double ratio);
BdspVecResult64 multiply_frequency_response_real64(BdspVec64* vector, BdspRealFn64 frequency_response,
                                                   const void* frequency_response_data, uint8_t is_symmetric, double ratio);
BdspVecResult64 multiply_frequency_response_complex64(BdspVec64* vector, BdspComplexFn64 frequency_response,
                                                      const void* frequency_response_data, uint8_t is_symmetric, double ratio);
BdspVecResult64 interpolatef64(BdspVec64* vector, int32_t impulse_response, double rolloff, double interpolation_factor,
                               double delay, size_t len);
BdspVecResult64 interpolatef_custom64(BdspVec64* vector, BdspRealFn64 impulse_response, const void* impulse_response_data,
                                      uint8_t is_symmetric, double interpolation_factor, double delay, size_t len);
BdspVecResult64 interpolate_lin64(BdspVec64* vector, double interpolation_factor, double delay);

/* ===================================================================================================
 * 2. Device-residency extensions (no counterpart in the reference: its vectors live in host memory)
 * =================================================================================================== */
const char* bdsp_version(void);
const char* bdsp_last_error(void);
int32_t bdsp_device_count(void);
int32_t bdsp_set_device(int32_t device);              /* device used by subsequent calls of this host thread */
int32_t bdsp_sync(void);                              /* wait for all work queued by this thread's stream */
void bdsp_set_stream(void* cuda_stream);              /* cudaStream_t for subsequent calls of this thread (default: stream 0) */
void* bdsp_stream_create(void);                       /* a new non-blocking cudaStream_t (for pipelining transfers against kernels) */
void bdsp_stream_destroy(void* cuda_stream);
int32_t bdsp_stream_sync(void* cuda_stream);
/* bulk transfers: `len` T scalars; upload resizes the vector (like set_len32) when len != get_len32 */
int32_t bdsp_upload32(BdspVec32* vector, const float* host, size_t len);
int32_t bdsp_download32(const BdspVec32* vector, float* host, size_t len);
/* like bdsp_download32 but does not wait: the copy is queued on the thread's stream (host must be pinned
 * for it to overlap); call bdsp_sync() before reading `host` */
int32_t bdsp_download_async32(const BdspVec32* vector, float* host, size_t len);
int32_t bdsp_download_async64(const BdspVec64* vector, double* host, size_t len);
int32_t bdsp_upload64(BdspVec64* vector, const double* host, size_t len);
int32_t bdsp_download64(const BdspVec64* vector, double* host, size_t len);
/* Device pointer of the vector's storage (interleaved).  Valid until the next call that mutates the vector: most
 * operations produce their result in the handle's scratch buffer and swap the two pointers, and growing a vector
 * reallocates.  The pointer gives mutable access, so the call also drops every cache derived from the vector's contents
 * (the impulse-response spectrum convolve_signal32 keeps inside its `impulse_response` argument): write through the
 * pointer first, then call convolve_signal32. */
void* bdsp_device_ptr32(BdspVec32* vector);
void* bdsp_device_ptr64(BdspVec64* vector);
/* fused chain of the sequential trait calls scale(c) -> mul(&w) -> get_mag_phase(&mut mag, &mut phase)
 * in ONE pass over memory; `vector` keeps scale(c)*w when write_back != 0 */
int32_t bdsp_scale_mul_mag_phase32(BdspVec32* vector, float scale_re, float scale_im, const BdspVec32* w,
                                   BdspVec32* mag, BdspVec32* phase, int32_t write_back);
int32_t bdsp_scale_mul_mag_phase64(BdspVec64* vector, double scale_re, double scale_im, const BdspVec64* w,
                                   BdspVec64* mag, BdspVec64* phase, int32_t write_back);
/* fft followed by magnitude in one kernel (fft(&mut buffer).magnitude(), the C3 chain) */
BdspVecResult32 bdsp_fft_magnitude32(BdspVec32* vector);
BdspVecResult64 bdsp_fft_magnitude64(BdspVec64* vector);

/* ===================================================================================================
 * 3. Batched kernels on raw device pointers (rows of the reference's MatrixMxN, matrix/src/time_freq.rs:
 *    52-74, processed in one launch).  Pointers are device pointers; `rows` independent vectors of
 *    `points` complex points each, row r at element offset r*points.  flags: see BDSP_F_*.
 * =================================================================================================== */
#define BDSP_F_INVERSE 1      /* inverse direction (unnormalised) */
#define BDSP_F_SHIFT 2        /* forward: fft_shift the result; inverse: scale(1/points) + ifft_shift the input (fft()/ifft() semantics) */
#define BDSP_F_MAGNITUDE 4    /* store |X| (points real scalars per row) */
#define BDSP_F_REAL_INPUT 8   /* rows hold `points` real scalars */
#define BDSP_F_WINDOW(kind) ((((kind) & 7) + 1) << 8) /* forward only: multiply every row by the built-in window `kind` (0 triangular,
                                                     * 1 Hamming, 2 Blackman-Harris, 3 rectangular; translate_to_window_function,
                                                     * interop/src/lib.rs:153-164) while loading it = windowed_fft per row
                                                     * (matrix/src/time_freq.rs:69-74, time_to_freq.rs:167-175) */
int32_t bdsp_fft_rows_c32(const void* in, void* out, size_t points, size_t rows, int32_t flags);
int32_t bdsp_fft_rows_c64(const void* in, void* out, size_t points, size_t rows, int32_t flags);
/* Windowed transforms of overlapping (or spaced) frames of one signal: a short-time Fourier transform / spectrogram.
 * Frame f is the `points` points (complex, or real scalars with BDSP_F_REAL_INPUT) that start at point f*hop of `in`,
 * which must hold (frames-1)*hop + points points: frames = 1 + (len - points) / hop, no padding, no centring; hop > points
 * skips the samples between frames.  Row f of `out` is byte for byte what bdsp_fft_rows_* writes for the same points,
 * frames and flags when the frames lie back to back; BDSP_F_WINDOW(kind) | BDSP_F_MAGNITUDE gives a spectrogram.
 * flags: BDSP_F_SHIFT, BDSP_F_MAGNITUDE, BDSP_F_REAL_INPUT, BDSP_F_WINDOW(kind).  Returns 0; -2 for BDSP_F_INVERSE, hop == 0
 * or sizes that overflow size_t; -3 when the input range and the output overlap (bdsp_last_error says which).
 * points == 0 or frames == 0 returns 0 without a launch. */
int32_t bdsp_fft_frames_c32(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags);
int32_t bdsp_fft_frames_c64(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags);
#define BDSP_F_REAL_OUTPUT 16 /* bdsp_ifft_frames_*: out holds real scalars, the real part of the synthesis */
/* The inverse of bdsp_fft_frames_*: a signal from the spectra of its overlapping frames (inverse short-time Fourier
 * transform).  `in` holds `frames` rows of `points` complex spectra back to back (what bdsp_fft_frames_* writes without
 * BDSP_F_MAGNITUDE); `out` receives len = (frames-1)*hop + points points, complex or, with BDSP_F_REAL_OUTPUT, the real
 * parts as scalars (the imaginary parts are dropped, Hermitian symmetry is not checked).  Weighted overlap-add with
 * least-squares normalisation, as torch.istft(center=False) and scipy.signal.istft:
 *   y_f = ifft(X_f) / points (BDSP_F_SHIFT: X_f ifft-shifted first, the inverse of the forward call's BDSP_F_SHIFT),
 *   out[t] = sum_f w[t-f*hop] y_f[t-f*hop] / sum_f w[t-f*hop]^2 over the frames that cover t,
 * w = the built-in window BDSP_F_WINDOW(kind), or 1 without it (out[t] = the mean of the frames that cover t).  So
 * bdsp_ifft_frames(bdsp_fft_frames(x, W), W) returns x within rounding for every hop <= points.
 * flags: BDSP_F_SHIFT, BDSP_F_REAL_OUTPUT, BDSP_F_WINDOW(kind).  Returns 0; -2 for any other flag (bdsp_last_error names
 * it), hop == 0, hop > points (samples that no frame covers) or sizes that overflow size_t; -3 when the output range and
 * the input range overlap.  points == 0 or frames == 0 returns 0 without a launch. */
int32_t bdsp_ifft_frames_c32(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags);
int32_t bdsp_ifft_frames_c64(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags);
#define BDSP_F_ONESIDED 32        /* bdsp_welch_*, bdsp_csd_*, bdsp_coherence_*: real input only, points/2 + 1 bins, interior
                                     bins doubled (coherence: not doubled, the doubling cancels) */
#define BDSP_F_POWER_SPECTRUM 64  /* bdsp_welch_*, bdsp_csd_*: scaling 1/(sum w)^2 (power per bin) instead of the density
                                     1/(fs sum w^2) */
/* Welch's averaged periodogram of a device signal (scipy.signal.welch with detrend=False, MATLAB pwelch): the power
 * spectrum estimate from the frames of bdsp_fft_frames_* (frame f = the `points` points, or real scalars with
 * BDSP_F_REAL_INPUT, that start at point f*hop; no padding, no centring, hop > points allowed):
 *   out[k] = scale / frames * sum_f |X_f[k]|^2,  X_f = DFT(w * frame f),
 * w = the built-in window BDSP_F_WINDOW(kind), or 1 without it; scale = 1/(fs sum w^2) (density, the default) or, with
 * BDSP_F_POWER_SPECTRUM, 1/(sum w)^2 (fs is then ignored).  `out` receives `points` real values (float for c32, double
 * for c64) in np.fft.fftfreq order, fftshift order with BDSP_F_SHIFT; with BDSP_F_ONESIDED (real input only) points/2 + 1
 * values, bins 0 .. points/2, each doubled but bin 0 and the Nyquist bin of an even `points`.  The sums run in a fixed
 * order without atomics: repeated calls, on any device, give the same bytes.  The frames' spectra are never stored
 * whole: the workspace stays bounded whatever `frames` is.
 * flags: BDSP_F_REAL_INPUT, BDSP_F_SHIFT, BDSP_F_WINDOW(kind), BDSP_F_ONESIDED, BDSP_F_POWER_SPECTRUM.  Returns 0; -2 for
 * any other flag (bdsp_last_error names it), BDSP_F_ONESIDED without BDSP_F_REAL_INPUT or with BDSP_F_SHIFT, hop == 0,
 * fs not finite or not > 0 (unless BDSP_F_POWER_SPECTRUM), sizes that overflow size_t; -3 when the output overlaps the
 * input range.  points == 0 or frames == 0 returns 0 without a launch and leaves `out` untouched. */
int32_t bdsp_welch_c32(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags, float fs);
int32_t bdsp_welch_c64(const void* in, void* out, size_t points, size_t hop, size_t frames, int32_t flags, double fs);
/* Cross-spectral density of two device signals (scipy.signal.csd with detrend=False): the frames of x and of y are taken
 * as bdsp_welch_* takes its input's (frame f = the `points` points, or real scalars with BDSP_F_REAL_INPUT, that start at
 * point f*hop of each signal), and
 *   out[k] = scale / frames * sum_f conj(X_f[k]) * Y_f[k],  X_f = DFT(w * frame f of x),  Y_f = DFT(w * frame f of y),
 * with bdsp_welch_*'s window w, scale, order and one-sided fold.  `out` receives complex values (interleaved float2 for
 * c32, double2 for c64): `points` of them, or points/2 + 1 with BDSP_F_ONESIDED.  The sums run in a fixed order without
 * atomics: repeated calls, on any device, give the same bytes; the workspace stays bounded whatever `frames` is.
 * x and y are only read and may be the same buffer.
 * flags: BDSP_F_REAL_INPUT, BDSP_F_SHIFT, BDSP_F_WINDOW(kind), BDSP_F_ONESIDED, BDSP_F_POWER_SPECTRUM.  Returns 0; -2 for
 * any other flag (bdsp_last_error names it), BDSP_F_ONESIDED without BDSP_F_REAL_INPUT or with BDSP_F_SHIFT, hop == 0,
 * fs not finite or not > 0 (unless BDSP_F_POWER_SPECTRUM), sizes that overflow size_t; -3 when the output overlaps the
 * range of x or of y.  points == 0 or frames == 0 returns 0 without a launch and leaves `out` untouched. */
int32_t bdsp_csd_c32(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags, float fs);
int32_t bdsp_csd_c64(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags, double fs);
/* Magnitude-squared coherence of two device signals (scipy.signal.coherence with detrend=False), over the frames of
 * bdsp_csd_*:
 *   out[k] = |sum_f conj(X_f[k]) Y_f[k]|^2 / (sum_f |X_f[k]|^2 * sum_f |Y_f[k]|^2),
 * in [0, 1]; NaN in a bin where x or y has no power.  The scale and the one-sided doubling cancel, so there is no fs.
 * `out` receives `points` real values (float for c32, double for c64), or points/2 + 1 with BDSP_F_ONESIDED, in the order
 * of bdsp_csd_*.  Same guarantees as bdsp_csd_*.
 * flags: BDSP_F_REAL_INPUT, BDSP_F_SHIFT, BDSP_F_WINDOW(kind), BDSP_F_ONESIDED.  Returns 0; -2 for any other flag
 * (BDSP_F_POWER_SPECTRUM included), BDSP_F_ONESIDED without BDSP_F_REAL_INPUT or with BDSP_F_SHIFT, hop == 0, sizes that
 * overflow size_t; -3 when the output overlaps the range of x or of y.  points == 0 or frames == 0 returns 0 without a
 * launch and leaves `out` untouched. */
int32_t bdsp_coherence_c32(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags);
int32_t bdsp_coherence_c64(const void* x, const void* y, void* out, size_t points, size_t hop, size_t frames, int32_t flags);
/* convolve_signal for every row with one impulse response of h_points complex taps (device pointer);
 * `plan` caches the impulse-response spectrum between calls (create once, reuse, destroy) */
typedef struct BdspConvPlan BdspConvPlan;
BdspConvPlan* bdsp_conv_plan_create_c32(const void* h_device, size_t h_points);
BdspConvPlan* bdsp_conv_plan_create_c64(const void* h_device, size_t h_points);
void bdsp_conv_plan_destroy(BdspConvPlan* plan);
int32_t bdsp_convolve_signal_rows_c32(const void* in, void* out, size_t points, size_t rows, const BdspConvPlan* plan);
int32_t bdsp_convolve_signal_rows_c64(const void* in, void* out, size_t points, size_t rows, const BdspConvPlan* plan);

/* More batched (matrix-row) forms: the reference's MatrixMxN applies the vector operation to every row in turn
 * (matrix/src/time_freq.rs:52-74 interpolatef ..., matrix/src/complex.rs:18-26 magnitude / phase ...).  Rows sit back to
 * back in device memory; `in` / `out` are raw device pointers (bdsp_malloc or bdsp_device_ptr32), in != out.
 * magnitude = hypot(re, im) as ComplexToRealTransformsOps::magnitude (complex_to_real.rs:374-379), phase = atan2(im, re).
 * out: rows * points real scalars. */
int32_t bdsp_magnitude_rows_c32(const void* in, void* out, size_t points, size_t rows);
int32_t bdsp_magnitude_rows_c64(const void* in, void* out, size_t points, size_t rows);
int32_t bdsp_magnitude_squared_rows_c32(const void* in, void* out, size_t points, size_t rows);
int32_t bdsp_magnitude_squared_rows_c64(const void* in, void* out, size_t points, size_t rows);
int32_t bdsp_phase_rows_c32(const void* in, void* out, size_t points, size_t rows);
int32_t bdsp_phase_rows_c64(const void* in, void* out, size_t points, size_t rows);
/* rows of the fused chain of bdsp_scale_mul_mag_phase32: v <- v * scale * w (written back iff write_back), magnitude and
 * phase of the product; v, w: rows * points complex points, magnitude, phase: rows * points real scalars */
int32_t bdsp_scale_mul_mag_phase_rows_c32(void* v, const void* w, void* magnitude, void* phase, size_t points, size_t rows,
                                          float scale_re, float scale_im, int32_t write_back);
int32_t bdsp_scale_mul_mag_phase_rows_c64(void* v, const void* w, void* magnitude, void* phase, size_t points, size_t rows,
                                          double scale_re, double scale_im, int32_t write_back);
/* interpolatef32 (facade32.rs:1334) on every one of `rows` rows of `points` points (is_complex: interleaved complex
 * points, else real scalars) with a built-in impulse response (0 Sinc, else RaisedCosine(rolloff)); delay is in samples
 * (delta = 1).  out must hold rows * new_points points, new_points = round(len * factor) rounded up to even in scalars
 * (interpolation.rs:406-410), also returned through *new_points (may be NULL).  The tap tables are built once. */
int32_t bdsp_interpolatef_rows32(const void* in, void* out, size_t points, size_t rows, int32_t is_complex, int32_t impulse_response,
                                 float rolloff, float interpolation_factor, float delay, size_t len, size_t* new_points);
int32_t bdsp_interpolatef_rows64(const void* in, void* out, size_t points, size_t rows, int32_t is_complex, int32_t impulse_response,
                                 double rolloff, double interpolation_factor, double delay, size_t len, size_t* new_points);
/* raw memory helpers so that non-CUDA hosts (ctypes, cgo, JNI) can drive section 3 */
void* bdsp_malloc(size_t bytes);
void bdsp_free(void* device_ptr);
size_t bdsp_mem_free(void);                           /* free device memory in bytes (cudaMemGetInfo), 0 on error */
void* bdsp_malloc_host(size_t bytes);                 /* pinned host memory */
void bdsp_free_host(void* host_ptr);
int32_t bdsp_memcpy_h2d(void* device_dst, const void* host_src, size_t bytes);   /* async on the thread's stream */
int32_t bdsp_memcpy_d2h(void* host_dst, const void* device_src, size_t bytes);   /* async on the thread's stream */
int32_t bdsp_memset(void* device_dst, int32_t value, size_t bytes);
/* CUDA-event timing on the thread's stream (the stream the kernels above are launched on) */
void* bdsp_event_create(void);
void bdsp_event_destroy(void* event);
int32_t bdsp_event_record(void* event);
float bdsp_event_elapsed_ms(void* start, void* stop);  /* synchronises on `stop` */
/* number of kernels launched by this library since process start (all threads) */
uint64_t bdsp_kernel_launch_count(void);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* BASIC_DSP_B200_H */
