// Prints the Welch power-sum route (basic_dsp_b200/csrc/fft_route.h welch_route) for each input line:
//   f64 n hop frames real_input in   (integers; the input pointer in hex) -> "fused groups ctas".
#include <cstdio>

#include "fft_route.h"

int main() {
    unsigned long long n, hop, frames, in;
    int f64, real_input;
    while (std::scanf("%d %llu %llu %llu %d %llx", &f64, &n, &hop, &frames, &real_input, &in) == 6) {
        const bdsp::WelchPlan p = bdsp::welch_route(f64, n, hop, frames, real_input, in);
        std::printf("%d %zu %zu\n", (int)p.fused, p.groups, p.ctas);
        std::fflush(stdout);   // one answer per line to a caller that waits for it
    }
    return 0;
}
