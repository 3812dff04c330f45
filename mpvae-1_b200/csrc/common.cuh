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
// normal down to 2^-17 of it.  e is clamped to [-112, 127], where s and 1 / s are both fp32 normals: every finite
// maximum from 2^-112 up is scaled into [2^14, 2^15); a smaller one only scales to less.  0, Inf or NaN (e.g. the NaN
// gradients of degenerate rows) -> s = 1, values pass through.  The function returns log2(s).
#ifdef __CUDACC__
__host__ __device__
#endif
static inline int scale_exp_from_absmax_bits(uint32_t bits) {
    bits &= 0x7FFFFFFFu;
    if (bits == 0u || bits >= 0x7F800000u) return 0;
    int e = (int)(bits >> 23) - 127;
    if (e < -112) e = -112;
    return 14 - e;
}

// 2^k as fp32 for k in [-126, 127]
#ifdef __CUDACC__
__host__ __device__
#endif
static inline float pow2f(int k) {
    const uint32_t b = (uint32_t)(127 + k) << 23;
    float f;
    memcpy(&f, &b, 4);
    return f;
}

#ifdef __CUDACC__
__host__ __device__
#endif
static inline float scale_from_absmax_bits(uint32_t bits) { return pow2f(scale_exp_from_absmax_bits(bits)); }

// Undoing both operands' scales: a product accumulated from scaled pieces is multiplied by 2^-(ka + kb), which lies in
// [2^-252, 2^226] and so is not always one fp32 number.  It is applied as two powers of two: `extra` first, then `main`
// = 2^clamp(-(ka + kb), -126, 127).  Either order of the two products is exact whenever the descaled value is an fp32
// normal (the intermediate then lies between the scaled and the descaled value); when the whole factor fits one fp32
// number, extra = 1 and the result is the single product acc * main.
struct Descale { float main, extra; };
#ifdef __CUDACC__
__host__ __device__
#endif
static inline Descale descale_from_absmax_bits(uint32_t a_bits, uint32_t b_bits) {
    const int k = -(scale_exp_from_absmax_bits(a_bits) + scale_exp_from_absmax_bits(b_bits));
    const int km = k < -126 ? -126 : (k > 127 ? 127 : k);
    return {pow2f(km), pow2f(k - km)};
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
// warp_sum of N values at once (N a power of two, <= 32) with fewer shuffles: at each of the first log2(N) xor levels a
// lane keeps half of its values (the upper half where the level's bit of the lane is set) and trades the other half
// with its partner; the remaining levels reduce the one value left as warp_sum does.  Every partial is added to the
// same partner's partial at the same level as in warp_sum, with the lower lane's partial as the first operand: the
// order lane 0 of warp_sum adds in at every level.  So each total has the bits of warp_sum's result in lane 0, NaN
// payloads included (an fp64 add keeps its first NaN operand's payload; fp32 adds return the canonical NaN).  On return
// v[0] holds the total of value lane >> (5 - log2 N); the other entries of v are clobbered.
template <int N, typename T>
__device__ __forceinline__ void warp_sum_transposed(T (&v)[N], int lane) {
    static_assert(N >= 1 && N <= 32 && (N & (N - 1)) == 0, "N must be a power of two <= 32");
    int o = 16;
#pragma unroll
    for (int n = N; n > 1; n >>= 1, o >>= 1) {
        const bool upper = (lane & o) != 0;
#pragma unroll
        for (int k = 0; k < n / 2; ++k) {
            const T recv = __shfl_xor_sync(0xffffffffu, upper ? v[k] : v[k + n / 2], o);
            v[k] = (upper ? recv : v[k]) + (upper ? v[k + n / 2] : recv);
        }
    }
#pragma unroll
    for (; o > 0; o >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
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
