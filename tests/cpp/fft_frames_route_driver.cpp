// Prints the FFT route (basic_dsp_b200/csrc/fft_route.h) for each input line, strided input included:
//   f64 n batch inverse real_input magnitude in_mul in_rot out_rot in out work cluster_ok generic_only in_stride
// (integers; pointers in hex) -> "route groups n1 log2n2 log2n3 q P".
#include <cstdio>

#include "fft_route.h"

static const char* const NAMES[] = {"mul-pass", "real-rows", "complexify", "packed", "packed-16k", "cluster", "two-pass", "three-pass",
                                    "c64-rows", "block", "hybrid", "tiles", "q-three-pass", "q-rows-interleave", "q-rows", "bluestein",
                                    "packed-frames", "frame-pass"};

int main() {
    unsigned long long n, batch, in_rot, out_rot, in, out, work, in_stride;
    int f64, inverse, real_input, magnitude, in_mul, cluster_ok, generic_only;
    while (std::scanf("%d %llu %llu %d %d %d %d %llu %llu %llx %llx %llx %d %d %llu", &f64, &n, &batch, &inverse, &real_input, &magnitude,
                      &in_mul, &in_rot, &out_rot, &in, &out, &work, &cluster_ok, &generic_only, &in_stride) == 15) {
        bdsp::FftRouteIn r;
        r.f64 = f64; r.n = n; r.batch = batch;
        r.inverse = inverse; r.real_input = real_input; r.magnitude = magnitude; r.in_mul = in_mul;
        r.in_rot = in_rot; r.out_rot = out_rot;
        r.in = in; r.out = out; r.work = work;
        r.cluster_ok = cluster_ok; r.generic_only = generic_only;
        r.in_stride = in_stride;
        const bdsp::FftPlan p = bdsp::fft_route(r);
        std::printf("%s %zu %d %d %d %zu %zu\n", NAMES[(int)p.route], p.groups, p.n1, p.log2n2, p.log2n3, p.q, p.P);
        std::fflush(stdout);   // one answer per line to a caller that waits for it
    }
    return 0;
}
