// Prints the chunk plan of bdsp_csd_* / bdsp_coherence_* (basic_dsp_b200/csrc/fft_route.h csd_plan) and the route fft_route
// gives each chunk's frame transforms of x and of y, as csd_exec calls them (frame stride = hop, no shift, the window table
// as a real multiplier, x's spectra at `spec` and y's right after them).  First line: CSD_CHUNK_POINTS.  Then for each
// input line
//   f64 n hop frames real_input window x y spec   (integers; the three pointers in hex)
// -> "chunk slabs count cf_0 route_x_0 route_y_0 ... cf_count-1 route_x route_y" (routes as FftRoute values).
#include <cstdio>

#include "fft_route.h"

int main() {
    std::printf("%zu\n", bdsp::CSD_CHUNK_POINTS);
    std::fflush(stdout);
    unsigned long long n, hop, frames, x, y, spec;
    int f64, real_input, window;
    while (std::scanf("%d %llu %llu %llu %d %d %llx %llx %llx", &f64, &n, &hop, &frames, &real_input, &window, &x, &y, &spec) == 9) {
        const bdsp::CsdPlan p = bdsp::csd_plan(f64, n, frames);
        const size_t esz = (f64 ? 8 : 4) * (real_input ? 1 : 2), csz = f64 ? 16 : 8;
        std::printf("%zu %zu %llu", p.chunk, p.slabs, p.chunk ? (frames + p.chunk - 1) / p.chunk : 0);
        for (size_t f0 = 0; p.chunk && f0 < frames; f0 += p.chunk) {
            const size_t cf = frames - f0 < p.chunk ? frames - f0 : p.chunk;
            bdsp::FftRouteIn a;
            a.f64 = f64;
            a.n = n;
            a.batch = cf;
            a.real_input = real_input;
            a.in_mul = window ? 1 : 0;
            a.in_stride = hop;
            a.in = x + f0 * hop * esz;
            a.out = spec;
            const int rx = (int)bdsp::fft_route(a).route;
            a.in = y + f0 * hop * esz;
            a.out = spec + p.chunk * n * csz;
            const int ry = (int)bdsp::fft_route(a).route;
            std::printf(" %zu %d %d", cf, rx, ry);
        }
        std::printf("\n");
        std::fflush(stdout);   // one answer per line to a caller that waits for it
    }
    return 0;
}
