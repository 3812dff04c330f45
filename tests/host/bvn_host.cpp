// Host build of csrc/bvn.cuh (__host__ __device__): lets the CPU test-suite check the bivariate normal CDF of the
// closed-form pair probabilities against scipy without a GPU.
//   no arguments: stdin = n, then n records  h k rho  (text);  stdout = Phi2(h, k; rho) per record, %.17g
//   "--tables":   stdout = the Gauss-Legendre half tables, one line per rule: H x_1 .. x_H w_1 .. w_H
#define __host__
#define __device__
#define __forceinline__ inline
#include <cstdio>
#include <cstring>

#include "../../mpvae-1_b200/csrc/bvn.cuh"

template <int H>
static void print_rule() {
    double x[H], w[H];
    mpv::gauss_legendre_half<H>(x, w);
    std::printf("%d", H);
    for (int i = 0; i < H; ++i) std::printf(" %.17g", x[i]);
    for (int i = 0; i < H; ++i) std::printf(" %.17g", w[i]);
    std::printf("\n");
}

int main(int argc, char** argv) {
    if (argc > 1 && std::strcmp(argv[1], "--tables") == 0) {
        print_rule<3>();
        print_rule<6>();
        print_rule<10>();
        return 0;
    }
    int n = 0;
    if (std::scanf("%d", &n) != 1) return 1;
    for (int i = 0; i < n; ++i) {
        double h, k, r;
        if (std::scanf("%lf %lf %lf", &h, &k, &r) != 3) return 2;
        std::printf("%.17g\n", mpv::bvn_cdf(h, k, r));
    }
    return 0;
}
