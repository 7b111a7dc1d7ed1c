// Which kernels run one level of an FFT (fft.cu fft_any): the one place that picks the path.  Plain C++ (no CUDA), so that
// the routing table can be checked without a GPU (tests/cpp/fft_route_driver.cpp, tests/cpp/fft_frames_route_driver.cpp,
// tests/cpp/welch_route_driver.cpp for welch_route below).
// A strided input (FftRouteIn::in_stride other than 0 or n) takes one of the two frame routes; every other input the
// rules apply to in the order of FftRoute, and the first one that matches wins.
#pragma once
#include <cstddef>
#include <cstdint>

namespace bdsp {

enum class FftRoute {
    MulPass,         // in_mul_rows_kernel applies the multiplier, the product is routed again
    RealRows,        // packed single pass over rows of real scalars (fftp_kernel<RIN>)
    Complexify,      // real -> complex pass, the complex rows are routed again
    Packed,          // packed single pass (fftp_kernel: SQ for 64 / 128, NATQ for 256 .. 2048, R0 = 1 / 2 / 4 for 4096 .. 16384)
    Packed16k,       // persistent 16384-point kernel (fftp16k_kernel)
    Cluster,         // 2^16 points on a 16-CTA cluster (fftc65536_kernel)
    TwoPass,         // packed column pass + packed row pass, 2^15 .. 2^20
    ThreePass,       // packed column passes A and B + packed row pass, 2^21 .. 2^24
    C64Rows,         // f64_row_kernel, 1024 .. 4096 c64 points
    Block,           // fft_block_kernel, n <= fft_block_max_n
    Hybrid,          // generic column pass + packed 1024-point row pass (c32, 2^15 .. 2^20)
    Tiles,           // two or three passes of generic tiles
    QThreePass,      // f64 q * 2^k: three tile passes, radix-q step inside the first one
    QRowsInterleave, // radix-q pass, rows of P points routed again into a second buffer, interleave pass
    QRows,           // radix-q pass, generic rows that store interleaved
    Bluestein,       // chirp-z
    PackedFrames,    // strided frames: packed single pass with the frame addressing and the multiplier on its first load
                     // (fftp_kernel<FRAMES>)
    FramePass,       // strided frames: gather_frames_kernel copies them back to back, the copy is routed again
};

struct FftRouteIn {
    bool f64 = false;
    size_t n = 0, batch = 0;
    bool inverse = false, real_input = false, magnitude = false;
    int in_mul = 0;                // multiplier kind after the window table is materialised: 0 none, 1 real, 2 complex table
    size_t in_rot = 0, out_rot = 0;   // reduced mod n
    uintptr_t in = 0, out = 0;
    uintptr_t work = 0;            // scratch of the multi-pass routes (n = 2^k > fft_block_max_n), 0 when none is needed
    bool cluster_ok = false;       // the 16-CTA cluster kernel can be placed on this device
    bool generic_only = false;     // the generic kernels only: rows with a strided output map, the Bluestein sub-transforms
    size_t in_stride = 0;          // points between the starts of consecutive input sequences; 0 means n
};

struct FftPlan {
    FftRoute route;
    size_t groups = 0;             // CTAs of the packed single pass, row groups of the packed last pass
    int n1 = 0;                    // first-pass column length: n1 (two-pass), nA (three-pass), n / 1024 (hybrid), q * 2^a (q three-pass)
    int log2n2 = 0, log2n3 = 0;    // log2 of the later passes' lengths (two-pass: rows; three-pass: rows in log2n3; q three-pass: both)
    size_t q = 1, P = 0;           // q * 2^k routes: n = q * P
};

constexpr size_t FFT_BLOCK_MAX_C32 = 16384, FFT_BLOCK_MAX_C64 = 8192;
constexpr size_t FFT_GRID_MAX = 0x7fffffff;

inline int route_log2(size_t v) { int l = 0; while ((size_t(2) << l) <= v) l++; return l; }

inline FftPlan fft_route(const FftRouteIn& a) {
    const size_t n = a.n, rows = a.batch;
    const bool c32 = !a.f64;
    const size_t block_max = a.f64 ? FFT_BLOCK_MAX_C64 : FFT_BLOCK_MAX_C32;
    auto aligned = [](uintptr_t p, uintptr_t bytes) { return (p & (bytes - 1)) == 0; };
    // The packed kernels shift by half a sequence only (ifft_shift on load, fft_shift on store), their inverse variants
    // have no fft_shift or magnitude epilogue, and their forward single-pass variants no ifft_shift.
    const bool half_rot = (a.in_rot == 0 || a.in_rot == n / 2) && (a.out_rot == 0 || a.out_rot == n / 2);
    const bool inv_store = !(a.inverse && (a.magnitude || a.out_rot != 0));
    const bool pow2 = n && !(n & (n - 1));
    if (a.in_stride != 0 && a.in_stride != n) {
        // Frames that overlap or leave gaps: fused where fft_route would take Packed or RealRows (after MulPass) for the
        // same frames laid back to back, and where every frame start keeps the alignment of the paired loads (even stride:
        // 16 B for complex points, 8 B for real scalars).  Everything else is gathered first and then routed as rows.
        const size_t per = n >= 64 && n < 4096 ? 4096 / n : 1;
        const bool grid_ok = a.real_input ? rows / per * 2 <= FFT_GRID_MAX : (n < 4096 ? rows / per : rows * 2) <= FFT_GRID_MAX;
        if (c32 && !a.inverse && pow2 && n >= 64 && n <= 8192 && a.in_rot == 0 && half_rot && (a.in_mul == 0 || a.in_mul == 1) &&
            n * rows >= (1u << 16) && rows % per == 0 && grid_ok && aligned(a.in, a.real_input ? 8 : 16) && aligned(a.out, 8) &&
            a.in_stride % 2 == 0 && a.in != a.out)
            return {FftRoute::PackedFrames, rows / per};
        return {FftRoute::FramePass};
    }
    if (pow2 && !a.generic_only) {
        // the packed single-pass kernels take no first-load multiplier: in their throughput regime one elementwise pass +
        // the packed kernel beats the generic kernel with the multiplier fused
        if (c32 && a.in_mul && n >= 64 && n <= 16384 && n * rows >= (1u << 16)) return {FftRoute::MulPass};
        if (c32 && !a.in_mul && a.real_input && !a.inverse && a.in_rot == 0 && n >= 64 && n <= 16384 && n * rows >= (1u << 16)) {
            // rows of real scalars, single pass: 4 B read + 8 B written per point; whole groups of 4096 points
            const size_t per = n < 4096 ? 4096 / n : 1;
            if (half_rot && aligned(a.in, 8) && aligned(a.out, 8) && a.in != a.out && rows % per == 0 && rows / per * 2 <= FFT_GRID_MAX)
                return {FftRoute::RealRows, rows / per};
        }
        if (c32 && a.real_input && (a.inverse || a.in_rot != 0) && n >= 512 && n <= (1u << 24) && (n >= (1u << 15) || n * rows >= (1u << 18)) &&
            (n >= 4096 || rows % (4096 / n) == 0))
            // real f32 input in the throughput regime: one complexifying pass (4 B read + 8 B written per point) and the
            // packed complex passes beat the generic kernels that fuse the conversion into their first load
            return {FftRoute::Complexify};
        if (c32 && !a.in_mul && !a.real_input && n >= 64 && n <= 16384 && half_rot && inv_store && (a.inverse || a.in_rot == 0) &&
            aligned(a.in, 16) && aligned(a.out, 8) && a.in != a.out) {
            // out of place only: a CTA's stores may land on rows other CTAs still read.  Below 4096 points a CTA takes
            // 4096 / n rows, so only whole groups of 4096 points.
            const size_t per = n < 4096 ? 4096 / n : 1;
            if (rows % per == 0 && (n < 4096 ? rows / per : rows * 2) <= FFT_GRID_MAX)
                return {n == 16384 && rows >= 2 ? FftRoute::Packed16k : FftRoute::Packed, rows / per};
        }
        // few 2^16-point vectors: one launch on a 16-CTA cluster, transposition through distributed shared memory
        if (c32 && n == 65536 && !a.real_input && !a.in_mul && !a.magnitude && rows <= 8 && a.in != a.out && half_rot &&
            aligned(a.in, 8) && aligned(a.out, 8) && a.cluster_ok)
            return {FftRoute::Cluster};
        // Packed multi-pass transforms (16 B/point of traffic per pass).  Real input reaches them forward and unrotated
        // only (the complexifying pass takes the rest); the column passes take a table multiplier.
        const bool multi_ok = half_rot && inv_store && aligned(a.in, a.real_input ? 8 : 16) && aligned(a.out, 8) && aligned(a.work, 16) &&
                              a.work != a.in && a.work != a.out;
        if (c32 && n >= (1u << 15) && n <= (1u << 20) && multi_ok) {
            // n = n1 * N2:  2^15 = 32 x 1024, 2^16 = 256 x 256, 2^17 = 256 x 512, 2^18 = 256 x 1024, 2^19 = 512 x 1024,
            // 2^20 = 256 x 4096.  (Two adjacent 2048-point rows give only 16-byte store runs: 16 x 2048 took 0.46 ms and
            // 256 x 2048 0.48 ms per 2^26 points.)  Last pass: 16/Q adjacent rows of N2 = 256*Q points per 128-thread CTA
            // (Q = N2/256 <= 8), or four 4096-point rows per 512-thread CTA.
            static const int n1s[6] = {32, 256, 256, 256, 512, 256}, log2n2s[6] = {10, 8, 9, 10, 10, 12};
            const int i = route_log2(n) - 15, rows_per_cta = log2n2s[i] < 12 ? 16 >> (log2n2s[i] - 8) : 4;
            const size_t groups = rows * (size_t)(n1s[i] / rows_per_cta);
            if (groups <= FFT_GRID_MAX && rows * 4096 <= FFT_GRID_MAX) return {FftRoute::TwoPass, groups, n1s[i], log2n2s[i]};
        }
        if (c32 && n >= (1u << 21) && n <= (1u << 24) && multi_ok && rows * (n >> 4) <= FFT_GRID_MAX) {
            // n = nA * 256 * N3 with nA in {16, 32, 256}, N3 = 256 * Q; the last pass takes 16/Q rows per CTA
            static const int nAs[4] = {16, 16, 32, 256}, log2n3s[4] = {9, 10, 10, 8};
            const int i = route_log2(n) - 21;
            return {FftRoute::ThreePass, rows * (size_t)(nAs[i] / (16 >> (log2n3s[i] - 8))) * 256, nAs[i], 0, log2n3s[i]};
        }
    }
    if (pow2) {
        if (n <= block_max) {
            // c64 rows of 1024 / 2048 / 4096 points: in place only with the plain row layout (a row's loads all precede
            // its stores, rows do not overlap)
            if (a.f64 && n >= 1024 && n <= 4096 && rows <= FFT_GRID_MAX && (a.in != a.out || (!a.real_input && !a.magnitude)))
                return {FftRoute::C64Rows};
            return {FftRoute::Block};
        }
        // c32, n = n1 * 1024 with n1 <= 2^10: generic column pass (any input form: real, rotated, scaled) followed by the
        // packed four-rows-per-CTA 1024-point pass
        if (c32 && n <= (1u << 20) && (a.out_rot == 0 || a.out_rot == n / 2) && inv_store && a.work != a.in && a.work != a.out &&
            aligned(a.work, 16) && aligned(a.out, 8) && rows * (n / 4096) <= FFT_GRID_MAX)
            return {FftRoute::Hybrid, rows * (n / 4096), (int)(n / 1024)};
        return {FftRoute::Tiles};
    }
    FftPlan p;
    p.P = 1;
    while (n % (2 * p.P) == 0) p.P *= 2;
    p.q = n / p.P;
    if (p.q > 31 || p.P < 2) { p.route = FftRoute::Bluestein; return p; }
    if (a.f64 && p.P > block_max && !a.magnitude) {
        // n = N1 * N2 * N3 with N1 = q * 2^a <= ~1024 points per column; the first pass takes 4 lanes of 64-byte rows
        int la = 8 - (p.q > 3 ? route_log2(p.q) - 1 : 0);
        if (la < 4) la = 4;
        const int rest = route_log2(p.P) - la, mx = 9;
        if (rest >= 1 && rest <= 2 * mx && n / (p.q << la) % 4 == 0) {
            p.route = FftRoute::QThreePass;
            p.n1 = (int)(p.q << la);
            p.log2n2 = rest <= mx ? 0 : (rest + 1) / 2;   // 0: no middle pass
            p.log2n3 = rest - p.log2n2;
            return p;
        }
    }
    // c32 rows with a packed single-pass kernel (whole groups of 4096 points) in the throughput regime: packed rows +
    // interleave pass beat the generic kernel with the interleave fused into its stores (3072-point rows: 0.69 ms vs the
    // three-kernel path per 2^26 points)
    const bool packed_rows = c32 && p.P >= 256 && p.P <= block_max && n * rows >= (1u << 18) && (p.P >= 4096 || rows * p.q % (4096 / p.P) == 0);
    p.route = p.P > block_max || packed_rows ? FftRoute::QRowsInterleave : FftRoute::QRows;
    return p;
}

// Welch power sums (fft.cu welch_exec, bdsp_welch_*): fused into the packed frames kernel (fftp_kernel<FRAMES, PSUM>) for c32
// frames of a power-of-two n in [64, 8192], an even hop and the paired loads' alignment (16 B complex, 8 B real), within
// the grid limit.  Unlike PackedFrames there is no whole-group condition (the missing frames of the last group load zeros)
// and no out != in (the kernel writes a workspace).  `ctas` CTAs loop over the `groups` groups of N / n frames (N = 4096,
// or 8192), each summing into its own partial row of N floats: a function of n and the frame count only, so that the
// order of every sum, and with it the result, does not depend on the device.  WELCH_CTAS is the B200's residency, 148
// SMs x 4 CTAs of 128 threads (2 of 256 threads for 8192 points): one wave, 9.7 MB of partial rows in the 126 MB L2.
struct WelchPlan {
    bool fused = false;
    size_t groups = 0, ctas = 0;
};
constexpr size_t WELCH_CTAS = 592, WELCH_CTAS_8192 = 296;

inline WelchPlan welch_route(bool f64, size_t n, size_t hop, size_t frames, bool real_input, uintptr_t in) {
    const size_t per = n >= 64 && n < 4096 ? 4096 / n : 1;
    const size_t groups = frames / per + (frames % per != 0);
    const bool pow2 = n && !(n & (n - 1));
    if (f64 || !pow2 || n < 64 || n > 8192 || hop % 2 != 0 || (in & (real_input ? 7 : 15)) != 0 || groups > FFT_GRID_MAX) return {};
    const size_t cap = n == 8192 ? WELCH_CTAS_8192 : WELCH_CTAS;
    return {true, groups, groups < cap ? groups : cap};
}

}  // namespace bdsp
