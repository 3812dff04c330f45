// Closed-form predictive distribution of the probit layer: the S -> infinity limit of what predict.cu estimates with S
// samples.  The probit noise enters linearly, n_l = R_l . eps with eps ~ N(0, I_Z), so for a = fx_out
//   E_n[Phi(a_l + n_l)]          = Phi(h_l),                 h_l = a_l * scale_l,  scale_l = 1 / sqrt(1 + |R_l|^2)
//   E_n[Phi(a_i + n_i) Phi(a_j + n_j)] = Phi2(h_i, h_j; rho_ij),  rho_ij = R_i . R_j * scale_i * scale_j
// and the clamp E = c + k Phi (probit_math.cuh) is affine, so it passes through both expectations:
//   P(y_l = 1)          = c + k Phi(h_l)                          (predict_exact_kernel)
//   P(y_i = 1, y_j = 1) = c^2 + c k (Phi(h_i) + Phi(h_j)) + k^2 Phi2(h_i, h_j; rho_ij)   (predict_pairs_kernel)
// fx_out itself stays random through the encoder's reparameterisation; only the probit noise is integrated out.
//
// Every reduction is a fixed sequence (lane partials over z in order, then the xor shuffle tree), so results do not
// change from run to run, nor with the batch the rows come in.
#include "bvn.cuh"
#include "common.cuh"
#include "probit_math.cuh"
#include "rows.h"

namespace mpv {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr double kC = (double)kHalfEps;              // eps1 / 2, eps1 = fp32(1e-6)
constexpr double kK = 1.0 - (double)kEps1;           // 1 - eps1

// the fp32 probability of the marginal: E(x') with x' = fp32(fx_out * scale) rounded once, through the same probit_E /
// probit_E_stable as every other path
template <bool STABLE>
__device__ __forceinline__ float exact_E(float fx, double scale) {
    const float x = __double2float_rn((double)fx * scale);
    if (STABLE) {
        float E, om;
        probit_E_stable(x, E, om);
        return E;
    }
    return probit_E(x);
}

// one warp per label row: s_l = sum_z R[l, z]^2 in fp64, lane partials over z = lane, lane + 32, ... then the tree
__global__ void __launch_bounds__(kThreads)
predictive_scale_kernel(const float* __restrict__ r, int L, int Z, double* __restrict__ scale) {
    const int lane = threadIdx.x & 31;
    const int l = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (l >= L) return;
    const float* row = r + (size_t)l * Z;
    double s = 0.0;
    for (int z = lane; z < Z; z += 32) {
        const double v = row[z];
        s = fma(v, v, s);
    }
    s = warp_sum(s);
    if (lane == 0) scale[l] = 1.0 / sqrt(1.0 + s);
}

// one warp per pair; the pair is taken as (min, max) so that (i, j) and (j, i) give the same bits
__global__ void __launch_bounds__(kThreads)
predictive_rho_kernel(const float* __restrict__ r, int L, int Z, const double* __restrict__ scale,
                      const int2* __restrict__ pairs, int P, double* __restrict__ rho) {
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (p >= P) return;
    const int2 ij = pairs[p];
    if (ij.x < 0 || ij.x >= L || ij.y < 0 || ij.y >= L) {
        if (lane == 0) rho[p] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    const int i = min(ij.x, ij.y), j = max(ij.x, ij.y);
    const float* ri = r + (size_t)i * Z;
    const float* rj = r + (size_t)j * Z;
    double s = 0.0;
    for (int z = lane; z < Z; z += 32) s = fma((double)ri[z], (double)rj[z], s);
    s = warp_sum(s);
    if (lane == 0) rho[p] = s * scale[i] * scale[j];
}

// elementwise over (B, L); `vec`: rows of a multiple of 4 floats and 16-byte aligned pointers -> one float4 per thread
template <bool STABLE, bool VEC>
__global__ void __launch_bounds__(kThreads)
predict_exact_kernel(const float* __restrict__ fx, int L, size_t n, const double* __restrict__ scale,
                     float* __restrict__ out) {
    const size_t stride = (size_t)gridDim.x * kThreads;
    if (VEC) {
        for (size_t q = (size_t)blockIdx.x * kThreads + threadIdx.x; q < n / 4; q += stride) {
            const float4 v = __ldcs(reinterpret_cast<const float4*>(fx) + q);
            const int l = (int)((q * 4) % (size_t)L);
            float4 e;
            e.x = exact_E<STABLE>(v.x, scale[l]);
            e.y = exact_E<STABLE>(v.y, scale[l + 1]);
            e.z = exact_E<STABLE>(v.z, scale[l + 2]);
            e.w = exact_E<STABLE>(v.w, scale[l + 3]);
            __stcs(reinterpret_cast<float4*>(out) + q, e);
        }
    } else {
        for (size_t q = (size_t)blockIdx.x * kThreads + threadIdx.x; q < n; q += stride)
            out[q] = exact_E<STABLE>(fx[q], scale[q % (size_t)L]);
    }
}

// one thread per (row, pair) cell, pair index fastest; h, Phi and Phi2 in fp64, one rounding to fp32 at the end
template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
predict_pairs_kernel(const float* __restrict__ fx, int L, const double* __restrict__ scale, const int2* __restrict__ pairs,
                     const double* __restrict__ rho, int P, size_t n, float* __restrict__ out) {
    const size_t stride = (size_t)gridDim.x * kThreads;
    for (size_t q = (size_t)blockIdx.x * kThreads + threadIdx.x; q < n; q += stride) {
        const size_t b = q / (size_t)P;
        const int p = (int)(q - b * (size_t)P);
        const int2 ij = pairs[p];
        const double r = rho[p];
        if (ij.x < 0 || ij.x >= L || ij.y < 0 || ij.y >= L || r != r) {
            out[q] = __int_as_float(0x7fc00000);
            continue;
        }
        const int i = min(ij.x, ij.y), j = max(ij.x, ij.y);
        const float* row = fx + b * (size_t)L;
        if (i == j) {   // P(y_i = 1, y_i = 1) = P(y_i = 1): the marginal's bits
            out[q] = exact_E<STABLE>(row[i], scale[i]);
            continue;
        }
        const double hi = (double)row[i] * scale[i], hj = (double)row[j] * scale[j];
        const double pi = phi_cdf(hi), pj = phi_cdf(hj);
        const double b2 = bvn_cdf(hi, hj, r);
        out[q] = __double2float_rn(kC * kC + kC * kK * (pi + pj) + kK * kK * b2);
    }
}

int grid_for(size_t work, int per_sm) {
    const size_t g = (work + kThreads - 1) / kThreads;
    const size_t cap = (size_t)kNumSMs * per_sm;
    return (int)(g < cap ? g : cap);
}

}  // namespace

int launch_predictive_scale(const float* r, int L, int Z, double* scale, cudaStream_t stream) {
    predictive_scale_kernel<<<ceil_div(L, kWarps), kThreads, 0, stream>>>(r, L, Z, scale);
    return check_launch("predictive_scale_kernel");
}

int launch_predictive_rho(const float* r, int L, int Z, const double* scale, const int* pairs, int P, double* rho,
                          cudaStream_t stream) {
    if (P == 0) return 0;
    predictive_rho_kernel<<<ceil_div(P, kWarps), kThreads, 0, stream>>>(r, L, Z, scale,
                                                                       reinterpret_cast<const int2*>(pairs), P, rho);
    return check_launch("predictive_rho_kernel");
}

int launch_predict_exact(const float* fx_out, int B, int L, const double* scale, bool stable, float* out,
                         cudaStream_t stream) {
    if (B == 0) return 0;
    const size_t n = (size_t)B * L;
    const bool vec = L % 4 == 0 && ((reinterpret_cast<uintptr_t>(fx_out) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
    const int grid = grid_for(vec ? n / 4 : n, 16);
    if (vec) {
        if (stable) predict_exact_kernel<true, true><<<grid, kThreads, 0, stream>>>(fx_out, L, n, scale, out);
        else predict_exact_kernel<false, true><<<grid, kThreads, 0, stream>>>(fx_out, L, n, scale, out);
    } else {
        if (stable) predict_exact_kernel<true, false><<<grid, kThreads, 0, stream>>>(fx_out, L, n, scale, out);
        else predict_exact_kernel<false, false><<<grid, kThreads, 0, stream>>>(fx_out, L, n, scale, out);
    }
    return check_launch("predict_exact_kernel");
}

int launch_predict_pairs(const float* fx_out, int B, int L, const double* scale, const int* pairs, const double* rho, int P,
                         bool stable, float* out, cudaStream_t stream) {
    if (B == 0 || P == 0) return 0;
    const size_t n = (size_t)B * P;
    const int grid = grid_for(n, 32);
    const int2* pr = reinterpret_cast<const int2*>(pairs);
    if (stable) predict_pairs_kernel<true><<<grid, kThreads, 0, stream>>>(fx_out, L, scale, pr, rho, P, n, out);
    else predict_pairs_kernel<false><<<grid, kThreads, 0, stream>>>(fx_out, L, scale, pr, rho, P, n, out);
    return check_launch("predict_pairs_kernel");
}

}  // namespace mpv
