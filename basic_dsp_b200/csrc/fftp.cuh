// Shared pieces of the packed-FP32x2 FFT kernels (fftp.cu, fftp16k.cu): shared-memory layout and twiddle table offsets.
#pragma once
#include <type_traits>

#include "fft.cuh"
#include "fft_route.h"
#include "ols4096.cuh"

namespace bdsp {

// floats per sub-block plane: 16 rows of 272 plus a pad that spreads the sub-blocks over the 16-byte
// bank windows, so that the 8 lanes of every quarter-warp of the 128-bit loads in F3 (lanes walk
// sub-block, then row) hit 8 different windows: NSB = 2 -> +8 floats, NSB = 4 -> +4 floats
#define FP_B_OF(NSB_) (4352 + ((NSB_) == 2 ? 8 : (NSB_) == 4 ? 4 : 0))

// layout inside a sub-block: p = 256*row + 16*g + j  ->  272*row + 16*g + ((j + 4*(rot(g) + (row>>1))) & 15)
__device__ __forceinline__ int fp_rot(int row, int g) { return (((g >> 1) + (row >> 1)) & 3); }

// twiddle table (floats): [0,256) Re W4096^c, [256,512) Im W4096^c, [512,1024) stride-16 table (see ols4096.cu),
// [1024 + 8192*i + c] Re W_{8192<<i}^c, [1024 + 8192*i + 4096 + c] Im, c in [0,4096), i in {0,1}
// [1024 + 16384 + 4*(16*ka + b)] splat table {c, c, s, s} of W256^{ka*b} (first pass of the 2^20 transform)
#define FP_TW_SPLAT (1024 + 2 * 8192)
// [FP_TW_1K + c] Re W1024^c, [FP_TW_1K + 256 + c] Im, c in [0,256)
#define FP_TW_1K (FP_TW_SPLAT + 1024)
// same for W512^c and W2048^c
#define FP_TW_512 (FP_TW_1K + 512)
#define FP_TW_2K (FP_TW_512 + 512)
// second-stage tables of the short-row mode: float4 index (8*kg + j/2) = {Re(j), Re(j+1), Im(j), Im(j+1)} of W_{16P}^{kg*j}
#define FP_TW_S4 (FP_TW_2K + 512)
#define FP_TW_S8 (FP_TW_S4 + 128)
#define FP_TW_FLOATS (FP_TW_S8 + 256)

// per-device table (nullptr and last error set on failure)
const float* fftp_twiddles();

// Calls launch(INV, SHIFT_IN, SHIFT_OUT, MAG) with std::bool_constant arguments for the variant a packed kernel has.  Every
// packed kernel has the four forward variants (fft_shift and magnitude on the store, nothing on the load); HAS_INV adds the
// plain inverse one, HAS_INV_SI the inverse one with ifft_shift on the load.  A combination without a kernel is an error.
template <bool HAS_INV, bool HAS_INV_SI, typename L>
int fftp_with_flags(bool inv, bool si, bool so, bool mag, const L& launch) {
    const std::true_type y;
    const std::false_type n;
    if (!inv && !si) {
        if (mag) return so ? launch(n, n, y, y) : launch(n, n, n, y);
        return so ? launch(n, n, y, n) : launch(n, n, n, n);
    }
    if constexpr (HAS_INV) {
        if (inv && !so && !mag) {
            if constexpr (HAS_INV_SI) { if (si) return launch(y, y, n, n); }
            if (!si) return launch(y, n, n, n);
        }
    }
    set_last_error("fftp: no kernel for inverse %d, ifft_shift %d, fft_shift %d, magnitude %d", (int)inv, (int)si, (int)so, (int)mag);
    return -2;
}

}  // namespace bdsp
