// Sampled prediction: the row passes that follow the nt product (nr in the workspace, either row layout) and the
// small regime's one-launch kernel.
//
// predict: indiv_prob[b, l] = mean_s E(nr[s, b, l] + fx_out[b, l]) (mpvae.py:170,180,203), the feature branch alone.
// Scoring new rows needs no labels, so none of the loss forward's other work happens here: no label branch, no
// log-likelihoods, no ranking factors, no per-(row, sample) statistics, no per-row tail.
//
// The predictions are bit-equal to the indiv_prob of the loss forward by construction: E comes from the same
// probit_math.cuh functions (probit_E, or probit_E_stable under MPVAE_FLAG_STABLE_CDF), and the mean over samples is
// taken in the forward kernels' order -- pair sums E_s + E_{s+1}, pairs added in sample order, then / S.
//
// Conditional prediction: P(y_l = 1 | the row's observed labels, x) by importance-weighting the S probit samples that
// predict draws.  Sample s of row b has the likelihood of the observed labels O_b,
//     lp_s = sum_{o in O_b} ll(x_{s,o}, y_o)       (cell_forward's ll, fp64 sums in the tiled forward's order)
// and the unobserved cells take the self-normalised weighted mean of E over the samples:
//     m = max_s fp32(lp_s),  u_s = exp(fp32(lp_s) - m),  se = sum_s (double) u_s,  fse = fp32(se)
//     prob[b, l] = (sum_s u_s E_{s,l}) / fse       (l not in O_b; pairs (u0 E0 + u1 E1) added in sample order)
//     prob[b, l] = observed[b, l]                  (l in O_b: exactly 0 or 1)
//     log_evidence[b] = log(fse / S) + m,   ess[b] = se^2 / sum_s (double) u_s^2
// The log-mean-exp is the loss's own (common.cuh: warp_log_mean_exp), so with every label observed -log_evidence is
// the row's nll_loss_x, and with none observed (u = 1, fse = S) prob is predict's indiv_prob, bit for bit.
//
// Three launches after the unchanged nt product:
//   pass A    probit_cond_loglik_kernel   per (sample-row, 128-label chunk) fp64 partial of lp -> fuse_part records
//   rows      probit_cond_weights_kernel  chunk partials added in the finalize kernel's order; m, u_s, fse, outputs
//   pass B    probit_cond_predict_kernel  probit_predict_rows_kernel with the weights u_s
// observed[b, l]: 0 or 1 = observed with that value, any other byte = unobserved.
#include "common.cuh"
#include "probit_math.cuh"
#include "rows.h"
#include "sample_rows.cuh"   // kThreads, kChunk, kLL, for_sample_pairs, rows_grid
#include "small_rows.cuh"

namespace mpv {

namespace {

// A warp owns 128 neighbouring labels of one batch row and walks the S samples with the four running sums in registers.
template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
probit_predict_rows_kernel(const RowArgs a, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S;
    const size_t yoff = (size_t)b * L;
    const float fS = (float)S;
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        if (l0 >= L) continue;
        float fx[kLL], acc[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) {
            fx[j] = l0 + j < L ? a.fx_out[yoff + l0 + j] : 0.f;
            acc[j] = 0.f;
        }
        for_sample_pairs(a, S, b, l0, true, [&](int s0, const float (&v)[2][kLL]) {
            const bool two = s0 + 1 < S;
#pragma unroll
            for (int j = 0; j < kLL; ++j) {
                float pl = predict_E<STABLE>(v[0][j] + fx[j]);   // mpvae.py:170,180
                if (two) pl += predict_E<STABLE>(v[1][j] + fx[j]);
                acc[j] += pl;
            }
        });
#pragma unroll
        for (int j = 0; j < kLL; ++j)
            if (l0 + j < L) a.indiv_prob[yoff + l0 + j] = acc[j] / fS;   // mpvae.py:203
    }
}

// Small regime, one launch, one CTA per batch row: R staged by the TMA bulk copy, the noise of a sample pair per warp
// (Philox in registers or the caller's tensor), the warp-level FMA chain, E of the feature branch; pair sums in shared
// memory, added in pair order at the end.
template <bool STABLE>
__global__ void __launch_bounds__(kSmallThreads)
probit_small_predict_kernel(const SmallArgs p) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ __align__(8) unsigned long long s_bar;
    const RowArgs& a = p.a;
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.L, S = a.S, Z = p.Z;
    const int npairs = (S + 1) >> 1;
    float* Rs = reinterpret_cast<float*>(s_raw);                           // [L][Z]
    float* nz = Rs + (((size_t)L * Z + 3) & ~(size_t)3);                   // [kSmallWarps][2][Z]
    float* ps = nz + (size_t)kSmallWarps * 2 * Z;                          // [npairs][L] pair sums of E
    const bool bulk = small_r_stage<kSmallThreads>(Rs, p.r, L, Z, &s_bar);
    const int nch = (L + 31) >> 5;
    float fxv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int l = (c << 5) + lane;
        fxv[c] = (c < nch && l < L) ? a.fx_out[(size_t)b * L + l] : 0.f;
    }
    small_r_wait(bulk, &s_bar);
    __syncthreads();
    const uint2 off = philox_offset(p.off, p.off_dev);
    float* nzw = nz + (size_t)warp * 2 * Z;
    for (int pair = warp; pair < npairs; pair += kSmallWarps) {
        const int s0 = pair << 1;
        small_noise_pair(nzw, p, s0, b, off, lane);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int l = (c << 5) + lane;
            if (c >= nch || l >= L) continue;
            float acc0, acc1;
            small_nr_pair(Rs + (size_t)l * Z, nzw, Z, acc0, acc1);
            float pl = predict_E<STABLE>(acc0 + fxv[c]);
            if (s0 + 1 < S) pl += predict_E<STABLE>(acc1 + fxv[c]);
            ps[(size_t)pair * L + l] = pl;
        }
        __syncwarp();   // nzw is rewritten by the next pair
    }
    __syncthreads();
    const float fS = (float)S;
    for (int l = tid; l < L; l += kSmallThreads) {
        float sx = 0.f;
        for (int q = 0; q < npairs; ++q) sx += ps[(size_t)q * L + l];
        a.indiv_prob[(size_t)b * L + l] = sx / fS;
    }
}

// a lane's four observed states: y[j] in {0, 1} where obs[j]
struct LaneObs { float y[kLL]; bool obs[kLL]; bool any_obs, any_free; };

__device__ __forceinline__ LaneObs lane_obs(const int8_t* __restrict__ row, int l0, int L) {
    LaneObs o;
    o.any_obs = o.any_free = false;
#pragma unroll
    for (int j = 0; j < kLL; ++j) {
        const int v = l0 + j < L ? (int)row[l0 + j] : -1;   // rows start at b * L bytes: no vector load
        o.obs[j] = (v == 0 || v == 1) && l0 + j < L;
        o.y[j] = v == 1 ? 1.0f : 0.0f;
        o.any_obs |= o.obs[j];
        o.any_free |= (!o.obs[j] && l0 + j < L);
    }
    return o;
}

// Pass A: the warp and grid layout of probit_predict_rows_kernel.  Per (sample, chunk) the lane's observed cells are
// added in label order, the warp's lanes by the butterfly -- the order of probit_row_fwd_tiled_kernel -- and lane 0
// leaves the sum as the chunk's FusePart::lp_x.  A chunk with no observed label writes zeros and loads nothing; a lane
// with none loads no nr.
template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
probit_cond_loglik_kernel(const RowArgs a, const int8_t* __restrict__ observed, FusePart* __restrict__ part, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S;
    const size_t yoff = (size_t)b * L;
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        const LaneObs o = lane_obs(observed + yoff, l0, L);
        FusePart* __restrict__ pc = part + (size_t)b * S * nchunks + c;
        if (!__any_sync(0xffffffffu, o.any_obs)) {
            for (int s = lane; s < S; s += 32) pc[(size_t)s * nchunks].lp_x = 0.0;
            continue;
        }
        float fx[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) fx[j] = o.obs[j] ? a.fx_out[yoff + l0 + j] : 0.f;
        for_sample_pairs(a, S, b, l0, o.any_obs, [&](int s0, const float (&v)[2][kLL]) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (s0 + i >= S) continue;
                double lp = 0.0;
#pragma unroll
                for (int j = 0; j < kLL; ++j)
                    if (o.obs[j]) lp += (double)cell_forward<STABLE>(v[i][j] + fx[j], o.y[j]).ll;   // mpvae.py:170,180
                lp = warp_sum(lp);
                if (lane == 0) pc[(size_t)(s0 + i) * nchunks].lp_x = lp;
            }
        });
    }
}

// Row reduction, one CTA per row: lp_s = the chunk partials added as probit_row_finalize_kernel adds them (a lane per
// chunk, stride 32, then the butterfly), then warp 0 runs the loss's log-mean-exp and leaves u_s in a.wts (B, S) and fse
// in a.rowaux[2b].  part == nullptr: lp_s is already in a.lp (the GHK sampler's log-weights).
__global__ void __launch_bounds__(kThreads)
probit_cond_weights_kernel(const RowArgs a, const FusePart* __restrict__ part, int nchunks, float* __restrict__ log_evidence,
                           float* __restrict__ ess) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int S = a.S;
    if (part) {
        for (int s = warp; s < S; s += kWarps) {
            const FusePart* __restrict__ pp = part + ((size_t)b * S + s) * nchunks;
            double l = 0.0;
            for (int t = lane; t < nchunks; t += 32) l += pp[t].lp_x;
            l = warp_sum(l);
            if (lane == 0) a.lp[(size_t)b * S + s] = l;
        }
        __syncthreads();
    }
    if (warp != 0) return;
    const double* __restrict__ lp = a.lp + (size_t)b * S;
    const LogMeanExp lme = warp_log_mean_exp(S, lane, [&](int s) { return (float)lp[s]; });
    double s2 = 0.0;
    for (int s = lane; s < S; s += 32) {
        const float u = expf((float)lp[s] - lme.m);
        a.wts[(size_t)b * S + s] = u;
        s2 += (double)u * (double)u;
    }
    s2 = warp_sum(s2);
    if (lane == 0) {
        a.rowaux[(size_t)b * 2] = lme.fse;
        log_evidence[b] = -lme.nll;              // log(fse / S) + m
        ess[b] = (float)(lme.se * lme.se / s2);
    }
}

// Pass B: probit_predict_rows_kernel with the weights: per pair MPV_ADD(u0 E0, u1 E1), pairs added in sample order,
// then / fse.  With u = 1 and fse = S these are predict's operations.  A lane whose labels are all observed loads no nr.
template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
probit_cond_predict_kernel(const RowArgs a, const int8_t* __restrict__ observed, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S;
    const size_t yoff = (size_t)b * L;
    const float* __restrict__ u = a.wts + (size_t)b * S;
    const float fse = a.rowaux[(size_t)b * 2];
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        if (l0 >= L) continue;
        const LaneObs o = lane_obs(observed + yoff, l0, L);
        float fx[kLL], acc[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) {
            fx[j] = l0 + j < L ? a.fx_out[yoff + l0 + j] : 0.f;
            acc[j] = 0.f;
        }
        if (o.any_free) {
            for_sample_pairs(a, S, b, l0, true, [&](int s0, const float (&v)[2][kLL]) {
                const bool two = s0 + 1 < S;
                const float u0 = u[s0], u1 = two ? u[s0 + 1] : 0.f;
#pragma unroll
                for (int j = 0; j < kLL; ++j) {
                    float pl = MPV_MUL(u0, predict_E<STABLE>(v[0][j] + fx[j]));   // mpvae.py:170,180
                    if (two) pl = MPV_ADD(pl, MPV_MUL(u1, predict_E<STABLE>(v[1][j] + fx[j])));
                    acc[j] = MPV_ADD(acc[j], pl);
                }
            });
        }
#pragma unroll
        for (int j = 0; j < kLL; ++j)
            if (l0 + j < L) a.indiv_prob[yoff + l0 + j] = o.obs[j] ? o.y[j] : acc[j] / fse;
    }
}

}  // namespace

int launch_predict_rows(RowArgs a, cudaStream_t stream) {
    const int nchunks = (a.L + kChunk - 1) / kChunk;
    const dim3 grid = rows_grid(a, nchunks);
    if (a.stable) probit_predict_rows_kernel<true><<<grid, kThreads, 0, stream>>>(a, nchunks);
    else probit_predict_rows_kernel<false><<<grid, kThreads, 0, stream>>>(a, nchunks);
    return check_launch("probit_predict_rows_kernel");
}

int launch_small_predict(RowArgs a, const SmallNoise& n, cudaStream_t stream) {
    // no more than the loss forward's shared memory (which small_regime_fits bounds): R, the noise pairs, one branch
    const size_t smem = ((((size_t)a.L * n.Z + 3) & ~(size_t)3) + (size_t)kSmallWarps * 2 * n.Z +
                         (size_t)((a.S + 1) / 2) * a.L) * sizeof(float);
    static bool configured[kMaxDevices] = {};
    const int dev = device_slot();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(probit_small_predict_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(probit_small_predict_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(small predict): %s", cudaGetErrorString(e)); return 4; }
        configured[dev] = true;
    }
    const SmallArgs p = small_args(a, n);
    if (a.stable) probit_small_predict_kernel<true><<<a.B, kSmallThreads, smem, stream>>>(p);
    else probit_small_predict_kernel<false><<<a.B, kSmallThreads, smem, stream>>>(p);
    return check_launch("probit_small_predict_kernel");
}

int launch_conditional_rows(RowArgs a, const int8_t* observed, FusePart* part, float* log_evidence, float* ess,
                            cudaStream_t stream) {
    const int nchunks = (a.L + kChunk - 1) / kChunk;
    const dim3 grid = rows_grid(a, nchunks);
    if (a.stable) probit_cond_loglik_kernel<true><<<grid, kThreads, 0, stream>>>(a, observed, part, nchunks);
    else probit_cond_loglik_kernel<false><<<grid, kThreads, 0, stream>>>(a, observed, part, nchunks);
    if (int rc = check_launch("probit_cond_loglik_kernel")) return rc;
    return launch_conditional_tail(a, observed, part, nchunks, log_evidence, ess, stream);
}

int launch_conditional_tail(RowArgs a, const int8_t* observed, const FusePart* part, int part_chunks, float* log_evidence,
                            float* ess, cudaStream_t stream) {
    probit_cond_weights_kernel<<<a.B, kThreads, 0, stream>>>(a, part, part_chunks, log_evidence, ess);
    if (int rc = check_launch("probit_cond_weights_kernel")) return rc;
    const int nchunks = (a.L + kChunk - 1) / kChunk;
    const dim3 grid = rows_grid(a, nchunks);
    if (a.stable) probit_cond_predict_kernel<true><<<grid, kThreads, 0, stream>>>(a, observed, nchunks);
    else probit_cond_predict_kernel<false><<<grid, kThreads, 0, stream>>>(a, observed, nchunks);
    return check_launch("probit_cond_predict_kernel");
}

}  // namespace mpv
