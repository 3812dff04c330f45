// Conditional prediction with many observed labels: a GHK sampler for the probit posterior.
//
// The clamped probit model in latent form: u = fx + R eps + w (eps ~ N(0, I_Z), w ~ N(0, I_L)) and
// P(y_l = 1 | u_l) = c + k 1[u_l > 0] (c = eps1 / 2, k = 1 - eps1), which is E = c + k Phi(fx + R eps) with w integrated
// out.  Per row b, with O the observed labels in ascending order and G = R R^T (fp32, read from its lower triangle):
//   factor   Sigma_O = I + G[O, O] = C C^T                                  (fp64, one CTA per row)
//   chain    per sample s, for k = 1..|O|:  m_k = fx_{o_k} + sum_{j<k} C_kj eta_j,  a = -m_k / C_kk
//              lw_s += log(c + k Phi(+-m_k / C_kk))                         (the cell probability of the observed y)
//              eta_k = the inverse CDF of the density proportional to (c + k 1[eta on y's side of a]) phi(eta) at U
//              w_k   = (n_{s,o_k} + zeta_k - sum_{j<k} C_kj w_j) / C_kk      (forward solve w = C^-1 (n_O + zeta))
//            then v_s = C^-T (eta - w)                                      (backward solve)
//   update   x_s = n_s + G[:, O] v_s, in place on nr: R eps_s for an exact draw of eps given u_O = fx_O + C eta_s
//            (Matheron's rule: prior sample n_s = R xi_s of predict, fresh zeta_s for w_O)
//   rows     predict.cu's conditional weights and predict kernels with lw_s in the lp slot: the loss's log-mean-exp,
//            then the weighted mean of E(fx + x_s) over the samples
// With O empty: lw = 0 and no update, so prob is predict's bits.  zeta and U are either the caller's (S, B, L) tensors
// (read at observed cells only) or a Philox stream with its own key, counter = (s, global row, label), so predict's
// noise xi is untouched.
//
// Launches after predict's nt product: [G product] gather, factor, chain, update, weights, predict.
#include "../../include/mpvae_b200.h"
#include "common.cuh"
#include "philox.cuh"
#include "probit_math.cuh"
#include "rows.h"
#include "small_rows.cuh"   // row_of

namespace mpv {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr double kC = 0.5 * (double)kEps1;   // the clamp E = c + k Phi, in fp64
constexpr double kK = 1.0 - (double)kEps1;
constexpr size_t kChainSmem = 48 * 1024;     // row block of C staged per chain step (no opt-in needed)
constexpr uint32_t kGhkKey = 0x47484B21u;    // xor-ed into the Philox key: a stream disjoint from predict's noise

// Draw eta from the density proportional to (c + k 1[eta > a]) phi(eta) by inverting its CDF at U (V = 1 - U, exact):
//   Z = c + k Q(a);  lower part (eta <= a) has mass c Phi(a), upper part (c + k) Q(a)   (Q = 1 - Phi)
//   lower:  Phi(eta) = U Z / c,              complement  Q(eta) = V - U k Q(a) / c
//   upper:  Q(eta)   = V Z / (c + k),        complement  Phi(eta) = (U c + k (1 - V Q(a))) / (c + k)
// Each branch inverts whichever of Phi / Q is below 1/2, so the far tails keep their precision, and the result is
// clamped to its side of a.  Returns eta and Z (the cell probability).
__device__ __forceinline__ double ghk_draw_upper(double a, double U, double V, double& Z) {
    const double Qa = 0.5 * erfc(a * 0.7071067811865476);
    Z = kC + kK * Qa;
    double t;
    if (V * Z >= (kC + kK) * Qa) {   // lower part
        const double p = U * Z / kC;
        t = p <= 0.5 ? normcdfinv(p) : -normcdfinv(V - U * kK * Qa / kC);
        t = fmin(t, a);
    } else {
        const double q = V * Z / (kC + kK);
        t = q <= 0.5 ? -normcdfinv(q) : normcdfinv((U * kC + kK * (1.0 - V * Qa)) / (kC + kK));
        t = fmax(t, a);
    }
    return t;
}

// y = 1: eta > a is y's side; y = 0: eta < a, drawn as the reflection so that F_0(eta) = U as well
__device__ __forceinline__ double ghk_draw(double a, int y, double U, double& Z) {
    const double V = 1.0 - U;
    return y ? ghk_draw_upper(a, U, V, Z) : -ghk_draw_upper(-a, V, U, Z);
}

// Gather: row b's observed labels in ascending order into idx[b][0..n), n into nobs[b]; a row with more than mo observed
// labels gets nobs = -1 (its outputs become NaN).  One warp per row.
__global__ void __launch_bounds__(32)
ghk_gather_kernel(const int8_t* __restrict__ observed, int L, int mo, int* __restrict__ nobs, int* __restrict__ idx) {
    const int b = blockIdx.x, lane = threadIdx.x;
    const int8_t* __restrict__ row = observed + (size_t)b * L;
    int n = 0;
    for (int l0 = 0; l0 < L; l0 += 32) {
        const int l = l0 + lane;
        const int v = l < L ? (int)row[l] : -1;
        const bool o = v == 0 || v == 1;
        const unsigned bal = __ballot_sync(0xffffffffu, o);
        const int pos = n + __popc(bal & ((1u << lane) - 1u));
        if (o && pos < mo) idx[(size_t)b * mo + pos] = l;
        n += __popc(bal);
    }
    if (lane == 0) nobs[b] = n > mo ? -1 : n;
}

// Factor: F = I + G[O, O] (lower triangle of G: o_i > o_j for i > j), then its Cholesky factor C in place, column by
// column (Crout): C_jj = sqrt(F_jj - sum_{k<j} C_jk^2), C_ij = (F_ij - sum_{k<j} C_ik C_jk) / C_jj.  F is n x n with
// row pitch n; C sits in the lower triangle and is mirrored into the upper one (F[j][i] = C_ij), so that both the
// chain (row k of C) and the backward solve (column k of C) read contiguous memory.
__global__ void __launch_bounds__(kThreads)
ghk_factor_kernel(const float* __restrict__ G, int L, int mo, const int* __restrict__ nobs, const int* __restrict__ idx,
                  double* __restrict__ fac) {
    const int b = blockIdx.x;
    const int n = nobs[b];
    if (n <= 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int* __restrict__ o = idx + (size_t)b * mo;
    double* __restrict__ F = fac + (size_t)b * mo * mo;
    for (int e = threadIdx.x; e < n * n; e += kThreads) {
        const int i = e / n, j = e % n;
        if (j <= i) F[(size_t)i * n + j] = (double)G[(size_t)o[i] * L + o[j]] + (i == j ? 1.0 : 0.0);
    }
    __syncthreads();
    for (int j = 0; j < n; ++j) {
        const double* __restrict__ Fj = F + (size_t)j * n;
        if (warp == 0) {
            double s = 0.0;
            for (int k = lane; k < j; k += 32) s += Fj[k] * Fj[k];
            s = warp_sum(s);
            if (lane == 0) F[(size_t)j * n + j] = sqrt(Fj[j] - s);
        }
        __syncthreads();
        const double cjj = Fj[j];
        for (int i = j + 1 + warp; i < n; i += kWarps) {
            double* __restrict__ Fi = F + (size_t)i * n;
            double s = 0.0;
            for (int k = lane; k < j; k += 32) s += Fi[k] * Fj[k];
            s = warp_sum(s);
            if (lane == 0) {
                const double cij = (Fi[j] - s) / cjj;
                Fi[j] = cij;
                F[(size_t)j * n + i] = cij;
            }
        }
        __syncthreads();
    }
}

struct ChainArgs {
    int S, B, L, mo, kb;            // kb: rows of C per shared-memory block
    const int *nobs, *idx;
    const double* fac;
    double *eta, *wv;               // (B, S, mo) each: eta, then w -> eta - w -> v in place
    const int8_t* observed;
    const float *zeta, *uniform;    // (S, B, L) or nullptr
    int Bg, row0;
    uint2 key, off;
    const unsigned long long* off_dev;
};

// the GHK draws of cell (s, b, o): zeta ~ N(0, 1) and U in (0, 1)
__device__ __forceinline__ void ghk_noise(const ChainArgs& g, int s, int b, int o, double& zeta, double& U) {
    if (g.zeta && g.uniform) {
        const size_t e = ((size_t)s * g.B + b) * g.L + o;
        zeta = (double)g.zeta[e];
        U = (double)g.uniform[e];
        return;
    }
    const unsigned long long c = ((unsigned long long)s * g.Bg + (unsigned long long)(g.row0 + b)) * g.L + o;
    const uint2 off = philox_offset(g.off, g.off_dev);
    const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), off.x, off.y), g.key);
    float n0, n1;
    box_muller(r.x, r.y, n0, n1);
    const double Ur = ((double)(r.z >> 9) + 0.5) * (1.0 / 8388608.0);   // (0, 1): 1 - U exact
    zeta = g.zeta ? (double)g.zeta[((size_t)s * g.B + b) * g.L + o] : (double)n0;
    U = g.uniform ? (double)g.uniform[((size_t)s * g.B + b) * g.L + o] : Ur;
}

// Chain: one CTA per row, a warp per sample (samples warp, warp + 8, ...), C streamed through shared memory in blocks
// of kb rows that all the row's samples use.  Leaves lw_s in a.lp[b * S + s] and v_s in wv.  Dot products: lane-strided
// fp64 sums, then the butterfly (a fixed order).
__global__ void __launch_bounds__(kThreads)
ghk_chain_kernel(const RowArgs a, const ChainArgs g) {
    extern __shared__ double sm[];
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int S = g.S, mo = g.mo;
    const int n = g.nobs[b];
    double* __restrict__ lp = a.lp + (size_t)b * S;
    if (n <= 0) {
        for (int s = threadIdx.x; s < S; s += kThreads) lp[s] = n == 0 ? 0.0 : (double)NAN;
        return;
    }
    const int* __restrict__ o = g.idx + (size_t)b * mo;
    const double* __restrict__ F = g.fac + (size_t)b * mo * mo;
    const int8_t* __restrict__ yrow = g.observed + (size_t)b * g.L;
    const float* __restrict__ fx = a.fx_out + (size_t)b * g.L;
    for (int s = threadIdx.x; s < S; s += kThreads) lp[s] = 0.0;
    // forward: the draws and w = C^-1 (n_O + zeta)
    for (int k0 = 0; k0 < n; k0 += g.kb) {
        const int k1 = min(n, k0 + g.kb);
        __syncthreads();
        for (int r = k0; r < k1; ++r)
            for (int j = threadIdx.x; j <= r; j += kThreads) sm[(size_t)(r - k0) * n + j] = F[(size_t)r * n + j];
        __syncthreads();
        for (int s = warp; s < S; s += kWarps) {
            double* __restrict__ eta = g.eta + ((size_t)b * S + s) * mo;
            double* __restrict__ w = g.wv + ((size_t)b * S + s) * mo;
            const float* __restrict__ nrow = a.nr + (size_t)row_of(a, s, b) * a.ldn;
            double lw = 0.0;
            for (int k = k0; k < k1; ++k) {
                const double* __restrict__ ck = sm + (size_t)(k - k0) * n;
                double d1 = 0.0, d2 = 0.0;
                for (int j = lane; j < k; j += 32) {
                    d1 += ck[j] * eta[j];
                    d2 += ck[j] * w[j];
                }
                d1 = warp_sum(d1);
                d2 = warp_sum(d2);
                if (lane == 0) {
                    const int ok = o[k];
                    const double ckk = ck[k];
                    const double m = (double)fx[ok] + d1;
                    double zeta, U, Z;
                    ghk_noise(g, s, b, ok, zeta, U);
                    eta[k] = ghk_draw(-m / ckk, yrow[ok] == 1, U, Z);
                    w[k] = ((double)nrow[ok] + zeta - d2) / ckk;
                    lw += log(Z);
                }
                __syncwarp();
            }
            if (lane == 0) lp[s] += lw;
        }
    }
    __syncthreads();
    // eta - w, in w's place
    for (int s = warp; s < S; s += kWarps) {
        const double* __restrict__ eta = g.eta + ((size_t)b * S + s) * mo;
        double* __restrict__ w = g.wv + ((size_t)b * S + s) * mo;
        for (int j = lane; j < n; j += 32) w[j] = eta[j] - w[j];
    }
    // backward: v = C^-T (eta - w), v_k = (d_k - sum_{j>k} C_jk v_j) / C_kk with C_jk = F[k][j] (the mirror)
    for (int k1 = n; k1 > 0; k1 -= g.kb) {
        const int k0 = max(0, k1 - g.kb);
        __syncthreads();
        for (int r = k0; r < k1; ++r)
            for (int j = r + threadIdx.x; j < n; j += kThreads) sm[(size_t)(r - k0) * n + j] = F[(size_t)r * n + j];
        __syncthreads();
        for (int s = warp; s < S; s += kWarps) {
            double* __restrict__ v = g.wv + ((size_t)b * S + s) * mo;
            for (int k = k1 - 1; k >= k0; --k) {
                const double* __restrict__ ck = sm + (size_t)(k - k0) * n;
                double d = 0.0;
                for (int j = k + 1 + lane; j < n; j += 32) d += ck[j] * v[j];
                d = warp_sum(d);
                if (lane == 0) v[k] = (v[k] - d) / ck[k];
                __syncwarp();
            }
        }
    }
}

// Update: x_s = n_s + G[:, O] v_s in place on nr, per row a (S x n) . (n x L) product with G's rows read by index
// (G[o, l] = G[l, o] up to the product's rounding).  gemm_fma_kernel's tiling: 64 x 64 tiles, 4 x 4 per thread, k in a
// fixed order, fp32 accumulation; the sum is added to nr with one rounding.  Rows with nothing observed are skipped.
constexpr int kUB = 64, kUK = 16;
__global__ void __launch_bounds__(256)
ghk_update_kernel(const RowArgs a, const float* __restrict__ G, int mo, const int* __restrict__ nobs,
                  const int* __restrict__ idx, const double* __restrict__ wv) {
    const int b = blockIdx.z;
    const int n = nobs[b];
    if (n <= 0) return;
    __shared__ __align__(16) float As[kUK][kUB + 4];
    __shared__ __align__(16) float Bs[kUK][kUB + 4];
    const int S = a.S, L = a.L;
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const int s0 = blockIdx.y * kUB, l0 = blockIdx.x * kUB;
    const int* __restrict__ o = idx + (size_t)b * mo;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < n; k0 += kUK) {
        for (int e = tid; e < kUB * kUK; e += 256) {
            const int r = e / kUK, c = e % kUK;          // A: (sample, k), k fastest
            const int s = s0 + r, k = k0 + c;
            As[c][r] = (s < S && k < n) ? (float)wv[((size_t)b * S + s) * mo + k] : 0.f;
            const int kk = k0 + e / kUB, l = l0 + e % kUB;   // B: (k, label), label fastest
            Bs[e / kUB][e % kUB] = (kk < n && l < L) ? G[(size_t)o[kk] * L + l] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kUK; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* __restrict__ nr = const_cast<float*>(a.nr);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int s = s0 + ty * 4 + i;
        if (s >= S) continue;
        float* __restrict__ xr = nr + (size_t)row_of(a, s, b) * a.ldn;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int l = l0 + tx * 4 + j;
            if (l < L) xr[l] = __fadd_rn(xr[l], acc[i][j]);
        }
    }
}

}  // namespace

GhkLayout ghk_layout(int S, int B, int L, int mo, size_t gram_scratch) {
    GhkLayout w{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    w.gram = take((size_t)L * L * sizeof(float));
    w.gram_scratch = take(gram_scratch);
    w.nobs = take((size_t)B * sizeof(int));
    w.idx = take((size_t)B * mo * sizeof(int));
    w.fac = take((size_t)B * mo * mo * sizeof(double));
    w.eta = take((size_t)B * S * mo * sizeof(double));
    w.wv = take((size_t)B * S * mo * sizeof(double));
    w.total = off;
    return w;
}

int launch_ghk_rows(RowArgs a, const GhkInputs& in, cudaStream_t stream) {
    const int B = a.B, S = a.S, L = a.L, mo = in.max_observed;
    char* base = static_cast<char*>(in.ws);
    const GhkLayout& w = in.layout;
    int* nobs = reinterpret_cast<int*>(base + w.nobs);
    int* idx = reinterpret_cast<int*>(base + w.idx);
    double* fac = reinterpret_cast<double*>(base + w.fac);
    ghk_gather_kernel<<<B, 32, 0, stream>>>(in.observed, L, mo, nobs, idx);
    if (int rc = check_launch("ghk_gather_kernel")) return rc;
    if (mo > 0) {
        ghk_factor_kernel<<<B, kThreads, 0, stream>>>(in.gram, L, mo, nobs, idx, fac);
        if (int rc = check_launch("ghk_factor_kernel")) return rc;
    }
    ChainArgs g{};
    g.S = S; g.B = B; g.L = L; g.mo = mo;
    g.kb = mo > 0 ? (int)(kChainSmem / ((size_t)mo * sizeof(double))) : 1;
    if (g.kb > 32) g.kb = 32;
    if (g.kb < 1) g.kb = 1;
    g.nobs = nobs; g.idx = idx; g.fac = fac;
    g.eta = reinterpret_cast<double*>(base + w.eta);
    g.wv = reinterpret_cast<double*>(base + w.wv);
    g.observed = in.observed;
    g.zeta = in.zeta; g.uniform = in.uniform;
    g.Bg = in.rows.b_global; g.row0 = in.rows.row0;
    g.key = make_uint2((uint32_t)in.rows.seed ^ kGhkKey, (uint32_t)(in.rows.seed >> 32));
    g.off = make_uint2((uint32_t)in.rows.offset, (uint32_t)(in.rows.offset >> 32));
    g.off_dev = reinterpret_cast<const unsigned long long*>(in.rows.offset_dev);
    const size_t smem = (size_t)g.kb * (mo > 0 ? mo : 1) * sizeof(double);
    if (smem > kChainSmem) {
        const cudaError_t e = cudaFuncSetAttribute(ghk_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("ghk_chain_kernel: %zu bytes of shared memory: %s", smem, cudaGetErrorString(e)); return 2; }
    }
    ghk_chain_kernel<<<B, kThreads, smem, stream>>>(a, g);
    if (int rc = check_launch("ghk_chain_kernel")) return rc;
    if (mo > 0) {
        const dim3 grid(ceil_div(L, kUB), ceil_div(S, kUB), B);
        ghk_update_kernel<<<grid, 256, 0, stream>>>(a, in.gram, mo, nobs, idx, g.wv);
        if (int rc = check_launch("ghk_update_kernel")) return rc;
    }
    // the rows pass of the importance estimator, on lw and the conditioned x
    return launch_conditional_tail(a, in.observed, nullptr, 0, in.log_evidence, in.ess, stream);
}

}  // namespace mpv
