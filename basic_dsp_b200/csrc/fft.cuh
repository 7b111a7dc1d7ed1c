// Host-side FFT entry point shared by the C ABI and the convolution code.
#pragma once
#include "common.cuh"

namespace bdsp {

struct FftOpts {
    int inverse = 0;        // 0: exp(-i...), 1: exp(+i...); never normalised (rustfft semantics)
    int real_input = 0;     // input holds n real scalars per sequence (imag = 0), output complex
    size_t in_rot = 0;      // read sequence element (i + in_rot) mod n   (ifft_shift fused on load)
    size_t out_rot = 0;     // write result k to (k + out_rot) mod n      (fft_shift fused on store)
    double scale = 1.0;     // multiply input by scale while loading (ifft's 1/points)
    int magnitude = 0;      // epilogue: store hypot(re, im) as n real scalars per sequence
    InMul in_mul;           // multiply input element g of every sequence by a table entry / window value while loading
                            // (windowed_fft: time_to_freq.rs:167-175; spectrum multiply of the frequency-domain
                            // convolution: convolution.rs:427-429,444-446) - no separate pass over memory
    size_t in_stride = 0;   // points between the starts of consecutive input sequences; 0 means n
};

// Transforms `batch` sequences of n complex points (sequence b at element offset b*n; real input:
// b*n scalars).  With opts.in_stride = s (not 0 or n), sequence b is the n points (scalars) that start at
// point b*s instead: overlapping or spaced frames of one signal, the last one ending at (batch-1)*s + n; such a
// call must not write into its input.  `work` must hold n*batch complex values when the transform needs a scratch pass
// (n > block limit or non power of two); pass nullptr to use the library's grow-only workspace.
// in == out is allowed.  Returns 0 or a negative error code (see set_last_error()).
template <typename T>
int fft_exec(const void* in, void* out, size_t n, size_t batch, const FftOpts& opts, void* work,
             size_t work_bytes, cudaStream_t stream);

// Inverse short-time transform: the inverse transforms of `frames` spectra of n points (back to back in `in`) under `opts`
// (inverse, scale, in_rot), then their least-squares overlap-add at `hop` points apart into (frames-1)*hop + n points of
// `out`: out[t] = sum_f w[t-f*hop] y_f[t-f*hop] / sum_f w[t-f*hop]^2.  opts.in_mul (kind 3, a built-in window, or none) is the
// synthesis window w, applied in the overlap-add rather than on the transform's load.  real_out: `out` holds the real parts
// as scalars.  Needs hop <= n, so that a frame covers every point, and `out` apart from `in`.  Returns 0 or a negative error.
template <typename T>
int ifft_frames_exec(const void* in, void* out, size_t n, size_t hop, size_t frames, const FftOpts& opts, bool real_out,
                     cudaStream_t stream);

// Welch's averaged periodogram (bdsp_welch_*): out[k] = scale / frames * sum_f |DFT(w x_f)[k]|^2 over the `frames` frames x_f
// of n points (real scalars with opts.real_input) that start f*hop points apart; w = the built-in window of opts.in_mul
// (kind 3) or 1, scale = 1 / (fs sum w^2), or 1 / (sum w)^2 with power_spectrum.  out holds n values in fftfreq order
// (opts.out_rot != 0: fftshift order), or with onesided bins 0 .. n/2, all but bin 0 and the Nyquist bin of an even n
// doubled.  Bit-reproducible: no atomics, every sum in an order fixed by n, hop, frames and the options.  Returns 0 or a
// negative error.
template <typename T>
int welch_exec(const void* in, T* out, size_t n, size_t hop, size_t frames, const FftOpts& opts, bool onesided, bool power_spectrum,
               double fs, cudaStream_t stream);

// largest n the single-CTA shared-memory kernel handles for this precision
template <typename T> size_t fft_block_max_n();

// device pointer to the master twiddle table W_{2^14}^i for the current device
template <typename T> const typename CpxOf<T>::type* twiddle_table();

// grow-only per-device workspace (device memory); not thread safe across host threads sharing a device
void* workspace(size_t bytes, int slot);
void workspace_bind_stream(cudaStream_t st);
void workspace_release_stream(cudaStream_t st);

}  // namespace bdsp
