// Host build of the operand-scale helpers of the tcgen05 contraction (mpvae-1_b200/csrc/common.cuh is
// __host__ __device__ there): lets the CPU test-suite sweep every fp32 exponent through them without a GPU.
//   stdin : n, then n records  a_bits b_bits acc_bits   (decimal uint32: two operand maxima and one accumulated value)
//   stdout: per record  ka kb sa_bits sb_bits main_bits extra_bits out_bits
// where ka, kb are log2 of the two scales, sa, sb the scales, main / extra the descale factors and out the descaled
// value as the GEMM epilogue forms it: (acc * extra) * main in fp32.
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../mpvae-1_b200/csrc/common.cuh"

static uint32_t bits_of(float f) {
    uint32_t b;
    std::memcpy(&b, &f, 4);
    return b;
}

static float float_of(uint32_t b) {
    float f;
    std::memcpy(&f, &b, 4);
    return f;
}

int main() {
    int n = 0;
    if (std::scanf("%d", &n) != 1) return 1;
    for (int i = 0; i < n; ++i) {
        unsigned a, b, c;
        if (std::scanf("%u %u %u", &a, &b, &c) != 3) return 2;
        const mpv::Descale d = mpv::descale_from_absmax_bits(a, b);
        volatile float scaled = float_of(c) * d.extra;   // two roundings, as on the device
        const float out = scaled * d.main;
        std::printf("%d %d %u %u %u %u %u\n", mpv::scale_exp_from_absmax_bits(a), mpv::scale_exp_from_absmax_bits(b),
                    bits_of(mpv::scale_from_absmax_bits(a)), bits_of(mpv::scale_from_absmax_bits(b)), bits_of(d.main),
                    bits_of(d.extra), bits_of(out));
    }
    return 0;
}
