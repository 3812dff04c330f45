// Shared host/device helpers for the mpvae_b200 CUDA library (error slot, launch counter, warp reductions).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>

namespace mpv {

// ---- host: thread-local error string + launch counter (defined in capi.cu) ----
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
// returns 0 when the last launch was accepted by the driver
int check_launch(const char* what);

constexpr int kNumSMs = 148;   // B200

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Per-tensor power-of-two scale of the fp16 operand split (contract_tc.cu): s = 2^(14 - e) with e the exponent of
// `bits` (max |x|, or an upper bound of it, as raw fp32 bits), so that max|x| * s lies in [2^14, 2^15): one binade
// under the fp16 maximum, which keeps the hi piece normal for elements down to 2^-28 of the maximum and the lo piece
// normal down to 2^-17 of it.  0, Inf or NaN (e.g. the NaN gradients of degenerate rows) -> s = 1, values pass through.
#ifdef __CUDACC__
__host__ __device__
#endif
static inline float scale_from_absmax_bits(uint32_t bits) {
    bits &= 0x7FFFFFFFu;
    if (bits == 0u || bits >= 0x7F800000u) return 1.0f;
    int e = (int)(bits >> 23) - 127;
    if (e < -100) e = -100;
    if (e > 100) e = 100;
    const uint32_t sb = (uint32_t)(127 + 14 - e) << 23;
    float f;
    memcpy(&f, &sb, 4);
    return f;
}

#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Log-mean-exp over the S per-sample log-likelihoods of one row (mpvae.py:188-190), by one whole warp in a fixed order:
//   m = max_s fp32(lp_s);  se = sum_s (double) exp(fp32(lp_s) - m)  (lane-strided, then the butterfly);  fse = fp32(se)
//   nll = -log(fse / S) - m    (the row's negative log-likelihood; -nll is the log of the Monte Carlo mean of exp(lp))
// lp(s) returns fp32(lp_s).  The per-row tail of the loss and the conditional prediction both call this, so the two
// share every bit of it.
struct LogMeanExp { float m; double se; float fse, nll; };
template <typename LP>
__device__ __forceinline__ LogMeanExp warp_log_mean_exp(int S, int lane, LP lp) {
    LogMeanExp r;
    float m = -INFINITY;
    for (int s = lane; s < S; s += 32) m = fmaxf(m, lp(s));
    r.m = warp_max(m);
    double se = 0.0;
    for (int s = lane; s < S; s += 32) se += (double)expf(lp(s) - r.m);
    r.se = warp_sum(se);
    r.fse = (float)r.se;
    r.nll = -logf(r.fse / (float)S) - r.m;
    return r;
}
#endif

}  // namespace mpv
