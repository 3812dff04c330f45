// Row kernels of the probit ELBO: everything in compute_loss (mpvae.py:145-210) after the contraction
// noise.R^T, and the closed-form backward (SURVEY.md 8a-12), one CTA per batch row.
//
//   forward  : nr (S,B,L) + y / fe_out / fx_out (B,L) + mu/logvar (B,D)
//              -> per-(s,b) log-likelihoods, ranking factors, KL row term, predictions (B,L) x2,
//                 six scalars (last CTA reduces the per-row partials in a fixed order)
//   backward : same inputs + saved per-(s,b) statistics + upstream cotangents
//              -> g_fe_out, g_fx_out (B,L), gxs = gx_l + gx_x (S,B,L) for g_R, mu/logvar grads
//
// Work decomposition inside a CTA (8 warps): lanes run along the label axis (coalesced 128 B reads of
// nr / y / logits); the 8 warps are split nws x nwl over samples x 32-label chunks so that short label
// rows (L = 14..81) still keep every warp busy.  Reductions over labels are warp shuffles (+ one smem
// hop when nwl > 1); log-likelihood sums are carried in fp64 so the result is independent of the
// summation order to ~1e-13 (the fp32 reference itself carries ~ulp(lp) of order noise, see DESIGN.md).
#include <stddef.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "philox.cuh"
#include "probit_math.cuh"
#include "rows.h"
#include "small_rows.cuh"

namespace mpv {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = 8;
constexpr int kST = 2;   // samples per inner tile (unrolled)

struct BlockCounts { int npos, nneg; };

// One lane's inputs for one 32-label chunk and kST samples.  obs: the label is observed (always, unmasked); an
// unobserved label's y reads as 0.  w0 / w1: the label's weights (LW only).
struct RowChunk { float y, fe, fx, nr[kST], w0, w1; bool obs; };

template <bool MASKED, bool LW>
__device__ __forceinline__ void load_chunk(RowChunk& in, const RowArgs& a, const float* __restrict__ yrow,
                                           const float* __restrict__ ferow, const float* __restrict__ fxrow, int c, int lane,
                                           int b, int s0) {
    const int l = (c << 5) + lane;
    if (l < a.L) {
        in.obs = !MASKED || a.mask[(size_t)b * a.L + l] != 0;
        in.y = in.obs ? yrow[l] : 0.0f; in.fe = ferow[l]; in.fx = fxrow[l];
        if (LW) { in.w0 = a.label_weight[l]; in.w1 = a.label_weight[a.L + l]; }
#pragma unroll
        for (int i = 0; i < kST; ++i)
            in.nr[i] = (s0 + i < a.S) ? a.nr[row_of(a, s0 + i, b) * a.ldn + l] : 0.0f;
    }
}

// n_pos / n_neg of a row; MASKED: over its observed labels only (mrow: the row's mask bytes)
template <int NT = kThreads, bool MASKED = false>
__device__ __forceinline__ BlockCounts count_labels(const float* __restrict__ yrow, const uint8_t* __restrict__ mrow, int L,
                                                    int* s_tmp) {
    constexpr int kWarps = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int cp = 0, cn = 0;
    for (int l = tid; l < L; l += NT) {
        if (MASKED && mrow[l] == 0) continue;
        const float v = yrow[l];
        cp += (v == 1.0f);   // torch.eq(labels, ones)   mpvae.py:107
        cn += (v == 0.0f);   // torch.eq(labels, zeros)  mpvae.py:108
    }
    cp = warp_sum(cp);
    cn = warp_sum(cn);
    if (lane == 0) { s_tmp[warp] = cp; s_tmp[kWarps + warp] = cn; }
    __syncthreads();
    BlockCounts c{0, 0};
#pragma unroll
    for (int w = 0; w < kWarps; ++w) { c.npos += s_tmp[w]; c.nneg += s_tmp[kWarps + w]; }
    return c;
}

// total_loss from the five terms (mpvae.py:207-208): the same operations for the batch means and for one row's terms
__device__ __forceinline__ float loss_total(const RowArgs& a, float nll, float nllx, float c, float cx, float kl) {
    return MPV_ADD(MPV_ADD(MPV_MUL(MPV_ADD(nll, nllx), a.nll_coeff), MPV_MUL(MPV_ADD(c, cx), a.c_coeff)), MPV_MUL(kl, 1.1f));
}

// The divisor of the batch means in the backward's coefficients: B, or 1 for per-row outputs
__device__ __forceinline__ float mean_div(const RowArgs& a) { return a.per_row ? 1.0f : (float)a.B; }

// The per-row tail of the forward, shared by every forward kernel: label counts, KL row term (mpvae.py:147-148), per-row
// log-mean-exp over samples, softmax weights, ranking sums (mpvae.py:188-190,115-122), and -- in the last CTA to
// arrive -- the batch means and the total (mpvae.py:190,122,147,207-208) in a fixed summation order.  Expects the
// row's a.lp / a.stat entries to have been written by threads of this CTA (any of them); blockDim.x == NT.  MASKED: the
// label counts run over the observed labels (a.mask); the rest is unchanged.  Per-row outputs (a.per_row): the row's
// own six values instead of the batch means -- w_b t_b formed in fp64 and rounded once (exactly 0 for a zero weight),
// then the total from them as for the means, so that B = 1 gives the bits of the means.
template <int NT = kThreads, bool MASKED = false>
__device__ __forceinline__ void row_tail(const RowArgs& a, int b) {
    constexpr int kWarps = NT / 32;
    __shared__ int s_cnt[2 * kWarps];
    __shared__ double s_kl[kWarps];
    __shared__ double s_fin[8];
    __shared__ int s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = a.S, B = a.B;
    const BlockCounts cnt = count_labels<NT, MASKED>(a.y + (size_t)b * a.L, MASKED ? a.mask + (size_t)b * a.L : nullptr,
                                                     a.L, s_cnt);   // contains a __syncthreads()
    {
        double kp = 0.0;
        const size_t o = (size_t)b * a.D;
        for (int d = tid; d < a.D; d += NT)
            kp += (double)kl_cell(a.fe_mu[o + d], a.fe_logvar[o + d], a.fx_mu[o + d], a.fx_logvar[o + d]).term;
        kp = warp_sum(kp);
        if (lane == 0) s_kl[warp] = kp;
    }
    __syncthreads();   // also orders the lp/stat global writes before warp 0 reads them back
    if (warp == 0) {
        const float norm5 = 5.0f * ((float)cnt.npos * (float)cnt.nneg);
        double outv[5];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const LogMeanExp lme =
                warp_log_mean_exp(S, lane, [&](int s) { return (float)a.lp[((size_t)b * S + s) * 2 + q]; });
            const float m = lme.m, fse = lme.fse;
            outv[q] = (double)lme.nll;
            double cs = 0.0;
            for (int s = lane; s < S; s += 32) {
                const size_t o = (size_t)b * S + s;
                a.wts[o * 2 + q] = expf((float)a.lp[o * 2 + q] - m) / fse;
                const float pos = a.stat[o * 4 + 2 * q], neg = a.stat[o * 4 + 2 * q + 1];
                float v = (pos * neg) / norm5;
                if (isnan(v) || isinf(v)) v = 0.0f;   // torch.where(isinf | isnan, 0, loss), mpvae.py:120
                cs += (double)v;
            }
            outv[2 + q] = warp_sum(cs);
        }
        double kl = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) kl += s_kl[w];
        outv[4] = 0.5 * kl;
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 5; ++q) a.rowout[(size_t)b * 8 + q] = outv[q];
            a.rowaux[(size_t)b * 2 + 0] = (float)cnt.npos;
            a.rowaux[(size_t)b * 2 + 1] = (float)cnt.nneg;
            if (a.per_row) {
                const double w = a.row_weight ? (double)a.row_weight[b] : 1.0, dS = (double)S;
                float t[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};   // a zero-weight row: 0 even where its terms are inf / NaN
                if (w != 0.0) {
                    t[0] = (float)(w * outv[0]); t[1] = (float)(w * outv[1]);
                    t[2] = (float)(w * outv[2] / dS); t[3] = (float)(w * outv[3] / dS);
                    t[4] = (float)(w * outv[4]);
                }
                a.scalars[0][b] = loss_total(a, t[0], t[1], t[2], t[3], t[4]);
#pragma unroll
                for (int q = 0; q < 5; ++q) a.scalars[q + 1][b] = t[q];
            }
        }
    }
    if (a.per_row) return;   // no batch means: the last-CTA counter is never touched and stays 0
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (warp < 5) {
        double acc = 0.0;
        if (a.row_weight == nullptr) {
            for (int r = lane; r < B; r += 32) acc += __ldcg(&a.rowout[(size_t)r * 8 + warp]);
        } else {
            // sum_r w_r t_r in the same order; a zero-weight row is skipped, so its inf / NaN terms stay out of the sum
            for (int r = lane; r < B; r += 32) {
                const float w = a.row_weight[r];
                if (w != 0.0f) acc += (double)w * __ldcg(&a.rowout[(size_t)r * 8 + warp]);
            }
        }
        acc = warp_sum(acc);
        if (lane == 0) s_fin[warp] = acc;
    }
    __syncthreads();
    if (tid == 0) {
        const double dB = (double)B, dSB = (double)S * (double)B;
        const float nll = (float)(s_fin[0] / dB), nllx = (float)(s_fin[1] / dB);
        const float c = (float)(s_fin[2] / dSB), cx = (float)(s_fin[3] / dSB);
        const float kl = (float)(s_fin[4] / dB);
        *a.scalars[0] = loss_total(a, nll, nllx, c, cx, kl); *a.scalars[1] = nll; *a.scalars[2] = nllx;
        *a.scalars[3] = c; *a.scalars[4] = cx; *a.scalars[5] = kl;
        *a.counter = 0u;   // ready for the next launch on this workspace
    }
}

// Second half of the tiled forward: adds the per-(sample-row, chunk) partials the cell kernel left, in a fixed order,
// and runs the per-row tail.  One CTA per batch row.
template <bool MASKED>
__global__ void __launch_bounds__(kThreads, 4)
probit_row_finalize_kernel(const RowArgs a) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // a warp per sample-row, a lane per chunk (stride 32), then a butterfly: a fixed order whatever the grid was
    for (int s = warp; s < a.S; s += kWarps) {
        const FusePart* __restrict__ pp = a.part + ((size_t)b * a.S + s) * a.part_tiles;
        double l0 = 0.0, l1 = 0.0;
        float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
        for (int t = lane; t < a.part_tiles; t += 32) {
            const FusePart p = pp[t];
            l0 += p.lp_l; l1 += p.lp_x;
            q0 += p.pos_l; q1 += p.neg_l; q2 += p.pos_x; q3 += p.neg_x;
        }
        l0 = warp_sum(l0); l1 = warp_sum(l1);
        q0 = warp_sum(q0); q1 = warp_sum(q1); q2 = warp_sum(q2); q3 = warp_sum(q3);
        if (lane == 0) {
            const size_t o = (size_t)b * a.S + s;
            a.lp[o * 2 + 0] = l0; a.lp[o * 2 + 1] = l1;
            reinterpret_cast<float4*>(a.stat)[o] = make_float4(q0, q1, q2, q3);
        }
    }
    row_tail<kThreads, MASKED>(a, b);
}

// Cell work of the forward, tiled (b, 128-label chunk): a warp owns 128 neighbouring labels of one batch row (a lane:
// four of them) and walks the S samples with y / logits / the prediction sums in registers -- no shared-memory
// accumulators, 16-byte loads of nr and 16-byte stores of the saved probabilities.  Per (sample, chunk) the warp reduces
// the six label sums and leaves them as a FusePart; probit_row_finalize_kernel adds the chunks in a fixed order and
// runs the per-row tail.  Grid (B, G): the chunks of a row are dealt out to G CTAs so that the grid fills the GPU
// whatever B is.
constexpr int kChunk = 128;   // labels per warp and iteration
constexpr int kLL = 4;        // labels per lane
static_assert(offsetof(FusePart, lp_x) == offsetof(FusePart, lp_l) + 8 && offsetof(FusePart, neg_x) == offsetof(FusePart, pos_l) + 12,
              "the tiled forward stores FusePart's two double and four float sums as arrays");

// MASKED: an unobserved cell (a.mask[b, l] == 0) reads y as 0 and adds nothing to the log-likelihood or the ranking sums;
// its E still enters the predictions and the saved E_l / E_x.  The mask bytes are byte loads (b * L need not be a
// multiple of 4).  LW: each lane loads its four labels' weights once per chunk, and cell_forward weighs the cell
// log-likelihoods before they enter the sums.
template <bool STABLE, int MINB, bool MASKED, bool LW>
__global__ void __launch_bounds__(kThreads, MINB)
probit_row_fwd_tiled_kernel(const RowArgs a, FusePart* __restrict__ part, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S;
    const size_t yoff = (size_t)b * L;
    const float fS = (float)S;
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        float y[kLL], fe[kLL], fx[kLL], accl[kLL], accx[kLL], w0[kLL], w1[kLL];
        bool obs[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) {
            y[j] = fe[j] = fx[j] = accl[j] = accx[j] = 0.f;
            if (l0 + j < L) { y[j] = a.y[yoff + l0 + j]; fe[j] = a.fe_out[yoff + l0 + j]; fx[j] = a.fx_out[yoff + l0 + j]; }
            if (LW) {
                w0[j] = w1[j] = 0.f;
                if (l0 + j < L) { w0[j] = a.label_weight[l0 + j]; w1[j] = a.label_weight[L + l0 + j]; }
            }
            if (MASKED) {
                obs[j] = l0 + j < L && a.mask[yoff + l0 + j] != 0;
                if (!obs[j]) y[j] = 0.f;
            }
        }
        // rows are 16-byte aligned (ldn % 4 == 0) and l0 is a multiple of 4: 16-byte accesses whenever the lane starts
        // inside the row; the pitch padding [L, ldn) is loaded but never used as a label
        const bool any = l0 < L;
        auto load = [&](int s) {
            float4 n = make_float4(0.f, 0.f, 0.f, 0.f);
            if (s < S && any) n = __ldcs(reinterpret_cast<const float4*>(a.nr + row_of(a, s, b) * a.ldn + l0));
            return n;
        };
        float4 n0 = load(0), n1 = load(1);
        for (int s0 = 0; s0 < S; s0 += kST) {
            const float4 m0 = load(s0 + 2), m1 = load(s0 + 3);        // next pair in flight
            float pl[kLL] = {0.f, 0.f, 0.f, 0.f}, px[kLL] = {0.f, 0.f, 0.f, 0.f};   // same pairwise order as before
            // the pair's six label sums, laid out for warp_sum_transposed: {lp_l, lp_x} and {pos_l, neg_l, pos_x, neg_x}
            // per sample; a sample >= S (odd S) keeps zeros, so the reductions below run on every lane unconditionally
            double lp[2 * kST];
            float pn[4 * kST];
#pragma unroll
            for (int k = 0; k < 2 * kST; ++k) lp[k] = 0.0;
#pragma unroll
            for (int k = 0; k < 4 * kST; ++k) pn[k] = 0.f;
#pragma unroll
            for (int i = 0; i < kST; ++i) {
                const int s = s0 + i;
                if (s >= S) continue;
                const float4 n4 = i == 0 ? n0 : n1;
                const float nv[kLL] = {n4.x, n4.y, n4.z, n4.w};
                float el[kLL], ex[kLL];
#pragma unroll
                for (int j = 0; j < kLL; ++j) {
                    el[j] = ex[j] = 0.f;
                    if (l0 + j < L) {
                        const CellFwd cl = cell_forward<STABLE, LW>(nv[j] + fe[j], y[j], LW ? w0[j] : 1.f, LW ? w1[j] : 1.f);   // mpvae.py:168,177
                        const CellFwd cx = cell_forward<STABLE, LW>(nv[j] + fx[j], y[j], LW ? w0[j] : 1.f, LW ? w1[j] : 1.f);   // mpvae.py:170,180
                        if (!MASKED || obs[j]) {
                            lp[2 * i] += (double)cl.ll; lp[2 * i + 1] += (double)cx.ll;
                            pn[4 * i] += cl.epos; pn[4 * i + 1] += cl.eneg; pn[4 * i + 2] += cx.epos; pn[4 * i + 3] += cx.eneg;
                        }
                        pl[j] += cl.E; px[j] += cx.E;
                        el[j] = cl.E; ex[j] = cx.E;
                    }
                }
                if (a.E_l && any) {   // kept for the backward (training)
                    const size_t o = row_of(a, s, b) * a.ldn + l0;
                    *reinterpret_cast<float4*>(a.E_l + o) = make_float4(el[0], el[1], el[2], el[3]);
                    *reinterpret_cast<float4*>(a.E_x + o) = make_float4(ex[0], ex[1], ex[2], ex[3]);
                }
            }
#pragma unroll
            for (int j = 0; j < kLL; ++j) { accl[j] += pl[j]; accx[j] += px[j]; }
            // warp_sum's bits for each of the six sums; lane 8k holds lp[k], lane 4k holds pn[k]
            warp_sum_transposed(lp, lane);
            warp_sum_transposed(pn, lane);
            FusePart* __restrict__ dst = part + ((size_t)b * S + s0) * nchunks + c;
            if (s0 + (lane >> 4) < S) {
                char* rec = reinterpret_cast<char*>(dst + (size_t)(lane >> 4) * nchunks);
                if ((lane & 7) == 0) reinterpret_cast<double*>(rec + offsetof(FusePart, lp_l))[(lane >> 3) & 1] = lp[0];
                if ((lane & 3) == 0) reinterpret_cast<float*>(rec + offsetof(FusePart, pos_l))[(lane >> 2) & 3] = pn[0];
            }
            n0 = m0; n1 = m1;
        }
        // predictions: mean over samples (mpvae.py:203-204)
#pragma unroll
        for (int j = 0; j < kLL; ++j)
            if (l0 + j < L) {
                a.indiv_prob_label[yoff + l0 + j] = accl[j] / fS;
                a.indiv_prob[yoff + l0 + j] = accx[j] / fS;
            }
    }
}

// Per-row coefficients of the backward (see cell_backward): effective weights of the loss terms = d objective / d term
// (mpvae.py:207-208 + upstream cotangents), the ranking normaliser k_b and the log-likelihood factor -(a_nll / B).
// Weighted rows: a_nll, a_c and a_kl are multiplied by w_b before the divisions (a weight of 1 keeps the unweighted
// bits); a zero-weight row gets all-zero coefficients, returned before the 0/0 of a degenerate row.
// Per-row outputs (a.per_row): row b's own cotangents and the divisor 1 (mean_div); a row whose six cotangents are all 0
// gets all-zero coefficients as a zero-weight row does, so a degenerate row left out of the objective gets no NaN.
struct RowCoeffs { float kb[2], cnb[2], a_kl; };

__device__ __forceinline__ RowCoeffs row_coeffs(const RowArgs& a, int b) {
    const int gi = a.per_row ? b : 0;
    const float gt = a.g_scalars[0] ? a.g_scalars[0][gi] : 0.0f, g1 = a.g_scalars[1] ? a.g_scalars[1][gi] : 0.0f,
                g2 = a.g_scalars[2] ? a.g_scalars[2][gi] : 0.0f, g3 = a.g_scalars[3] ? a.g_scalars[3][gi] : 0.0f,
                g4 = a.g_scalars[4] ? a.g_scalars[4][gi] : 0.0f, g5 = a.g_scalars[5] ? a.g_scalars[5][gi] : 0.0f;
    if (a.per_row && gt == 0.0f && g1 == 0.0f && g2 == 0.0f && g3 == 0.0f && g4 == 0.0f && g5 == 0.0f)
        return RowCoeffs{{0.0f, 0.0f}, {0.0f, 0.0f}, 0.0f};
    float a_nll[2] = {gt * a.nll_coeff + g1, gt * a.nll_coeff + g2};
    float a_c[2] = {gt * a.c_coeff + g3, gt * a.c_coeff + g4};
    RowCoeffs rc;
    rc.a_kl = gt * 1.1f + g5;
    if (a.row_weight != nullptr) {
        const float w = a.row_weight[b];
        if (w == 0.0f) return RowCoeffs{{0.0f, 0.0f}, {0.0f, 0.0f}, 0.0f};
        a_nll[0] = MPV_MUL(a_nll[0], w); a_nll[1] = MPV_MUL(a_nll[1], w);
        a_c[0] = MPV_MUL(a_c[0], w); a_c[1] = MPV_MUL(a_c[1], w);
        rc.a_kl = MPV_MUL(rc.a_kl, w);
    }
    const float npos = a.rowaux[(size_t)b * 2], nneg = a.rowaux[(size_t)b * 2 + 1];
    const float norm5 = 5.0f * (npos * nneg);
    const float fS = (float)a.S, fB = mean_div(a);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        if (norm5 == 0.0f) {
            // the reference back-propagates 0/0 through torch.div here (mpvae.py:118): NaN for the whole row
            rc.kb[q] = a.sanitize ? 0.0f : __fdiv_rn(0.0f, norm5);
        } else {
            rc.kb[q] = (a_c[q] / (fS * fB)) / norm5;
        }
        rc.cnb[q] = -(a_nll[q] / fB);
    }
    return rc;
}

// Upper bound of |gxs| for one (row, sample), from cell_backward:
//   |dL/dx| <= |cn| * max(phi/E, phi/(1-E)) + max(|cp| e^{-5E}, |cq| e^{5E}) * phi + |gp| * phi
// with phi/E <= 4.3 (the clamp E >= eps/2 caps the inverse Mills ratio near x = -4.2; same by symmetry for 1-E),
// e^{5E} phi <= 16.1 (x ~ 1) and phi <= 0.4.  Constants rounded up: 5, 17, 0.4.  The bound only has to be an upper
// bound within a few binades: it sets the power-of-two scale of the fp16 planes (common.cuh).
// MASKED: an unobserved cell's |dL/dx| is |gp| * phi, a term of the bound already.  One change: a row with no observed
// positive and no observed negative (e.g. nothing observed) puts no ranking term on any cell, so its ranking part of the
// bound is 0 -- not the 0/0 NaN of its normaliser, which would leave the whole batch's planes unscaled although the
// row's gradients are finite.
// LW: every cell's log-likelihood coefficient is cn * w0_l or cn * w1_l, so the log-likelihood part scales by
// W = max_l max(|w0_l|, |w1_l|), which the caller left as fp32 bits in *lw_absmax (tc_absmax over the 2L weights).
template <bool MASKED, bool LW>
__global__ void __launch_bounds__(256)
gxs_bound_kernel(const RowArgs a, const unsigned int* __restrict__ gp_absmax, unsigned int* __restrict__ out_bits,
                 const unsigned int* __restrict__ lw_absmax) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int bits = 0u;
    if (i < a.B * a.S) {
        const int b = i / a.S;
        const RowCoeffs rc = row_coeffs(a, b);
        const float4 st = reinterpret_cast<const float4*>(a.stat)[i];
        const float2 w = reinterpret_cast<const float2*>(a.wts)[i];
        const float gp = gp_absmax ? (__uint_as_float(gp_absmax[0]) + __uint_as_float(gp_absmax[1])) / (float)a.S : 0.0f;
        float kl = fabsf(rc.kb[0]), kx = fabsf(rc.kb[1]);
        if (MASKED && a.rowaux[(size_t)b * 2] == 0.0f && a.rowaux[(size_t)b * 2 + 1] == 0.0f) kl = kx = 0.0f;
        float nl = fabsf(rc.cnb[0] * w.x), nx = fabsf(rc.cnb[1] * w.y);
        if (LW) {
            const float W = __uint_as_float(*lw_absmax);
            nl *= W; nx *= W;
        }
        const float bl = 5.0f * nl + 17.0f * 5.0f * kl * fmaxf(st.x, st.y);
        const float bx = 5.0f * nx + 17.0f * 5.0f * kx * fmaxf(st.z, st.w);
        bits = __float_as_uint(bl + bx + 0.4f * gp) & 0x7FFFFFFFu;   // NaN (degenerate row) sorts highest
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned int t = __shfl_xor_sync(0xffffffffu, bits, o);
        bits = t > bits ? t : bits;
    }
    if ((threadIdx.x & 31) == 0 && bits != 0u) atomicMax(out_bits, bits);
}

// MASKED: an unobserved cell gets the cotangent of indiv_prob / indiv_prob_label alone (its y reads as 0 and its
// log-likelihood and ranking coefficients as 0).  LW: cell_backward weighs each observed cell's log-likelihood
// coefficient by its label's weight.
template <bool STABLE, bool MASKED, bool LW>
__global__ void __launch_bounds__(kThreads, 4)
probit_row_bwd_kernel(const RowArgs a) {
    extern __shared__ float s_gacc[];   // [nws][2][L] logit-gradient partial sums
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.L, S = a.S;
    const int nwl = a.nwl, nws = kWarps / nwl;
    const int wl = warp % nwl, ws = warp / nwl;
    const int nchunks = (L + 31) >> 5;
    const float* __restrict__ yrow = a.y + (size_t)b * L;
    const float* __restrict__ ferow = a.fe_out + (size_t)b * L;
    const float* __restrict__ fxrow = a.fx_out + (size_t)b * L;

    for (int i = tid; i < nws * 2 * L; i += kThreads) s_gacc[i] = 0.0f;

    const RowCoeffs rc = row_coeffs(a, b);
    const float fS = (float)S, fB = mean_div(a);
    const float a_kl = rc.a_kl;
    const float* kb = rc.kb;
    const float* cnb = rc.cnb;
    const bool has_gp = a.g_indiv_prob != nullptr, has_gpl = a.g_indiv_prob_label != nullptr;
    const float gscale = a.gxs_planes ? scale_from_absmax_bits(*a.gxs_scale) : 1.0f;
    __syncthreads();

    unsigned int gmax = 0u;
    const int steps = (S + kST * nws - 1) / (kST * nws);
    for (int step = 0; step < steps; ++step) {
        const int s0 = (step * nws + ws) * kST;
        if (s0 >= S) continue;
        float cn[kST][2], cp[kST][2], cq[kST][2];
#pragma unroll
        for (int i = 0; i < kST; ++i) {
            const int s = min(s0 + i, S - 1);
            const size_t o = (size_t)b * S + s;
            const float4 st = reinterpret_cast<const float4*>(a.stat)[o];
            const float2 w = reinterpret_cast<const float2*>(a.wts)[o];
            cn[i][0] = cnb[0] * w.x;           cn[i][1] = cnb[1] * w.y;
            cp[i][0] = -5.0f * kb[0] * st.y;   cp[i][1] = -5.0f * kb[1] * st.w;   // x neg sums
            cq[i][0] = 5.0f * kb[0] * st.x;    cq[i][1] = 5.0f * kb[1] * st.z;    // x pos sums
        }
        float* __restrict__ gacc = s_gacc + (size_t)ws * 2 * L;
        RowChunk cur, nxt;
        int c = wl;
        if (c < nchunks) load_chunk<MASKED, LW>(cur, a, yrow, ferow, fxrow, c, lane, b, s0);
        for (; c < nchunks; c += nwl) {
            if (c + nwl < nchunks) load_chunk<MASKED, LW>(nxt, a, yrow, ferow, fxrow, c + nwl, lane, b, s0);
            const int l = (c << 5) + lane;
            if (l < L) {
                const float gpl = has_gpl ? a.g_indiv_prob_label[(size_t)b * L + l] / fS : 0.0f;
                const float gpx = has_gp ? a.g_indiv_prob[(size_t)b * L + l] / fS : 0.0f;
                float gl = 0.0f, gx = 0.0f;
#pragma unroll
                for (int i = 0; i < kST; ++i) {
                    if (s0 + i < S) {
                        float dl, dx;
                        if (!MASKED || cur.obs) {
                            dl = cell_backward<STABLE, LW>(cur.nr[i] + cur.fe, cur.y, cn[i][0], cp[i][0], cq[i][0], gpl,
                                                           LW ? cur.w0 : 1.f, LW ? cur.w1 : 1.f);
                            dx = cell_backward<STABLE, LW>(cur.nr[i] + cur.fx, cur.y, cn[i][1], cp[i][1], cq[i][1], gpx,
                                                           LW ? cur.w0 : 1.f, LW ? cur.w1 : 1.f);
                        } else {
                            dl = cell_backward<STABLE>(cur.nr[i] + cur.fe, 0.0f, 0.0f, 0.0f, 0.0f, gpl);
                            dx = cell_backward<STABLE>(cur.nr[i] + cur.fx, 0.0f, 0.0f, 0.0f, 0.0f, gpx);
                        }
                        gl += dl; gx += dx;
                        if (a.gxs_planes) {
                            // operand planes of gxs^T . noise: hi = fp16(g s), lo = fp16(g s - hi)
                            const float g = (dl + dx) * gscale;
                            const __half hi = __float2half_rn(g);
                            __half* __restrict__ dst = a.gxs_planes + row_of(a, s0 + i, b) * a.gxs_pitch + l;
                            dst[0] = hi;
                            dst[a.gxs_plane_elems] = __float2half_rn(g - __half2float(hi));
                        } else if (a.gxs) {
                            const float g = dl + dx;
                            a.gxs[row_of(a, s0 + i, b) * a.ldn + l] = g;
                            const unsigned int gb = __float_as_uint(g) & 0x7FFFFFFFu;   // |g| as ordered bits, NaN highest
                            gmax = gb > gmax ? gb : gmax;
                        }
                    }
                }
                gacc[l] += gl;
                gacc[L + l] += gx;
            }
            cur = nxt;
        }
    }
    if (a.gxs_planes) {   // pad columns [L, pitch) of this row's S plane rows
        const int pad = a.gxs_pitch - L;
        for (int i = tid; i < S * pad; i += kThreads) {
            __half* __restrict__ dst = a.gxs_planes + row_of(a, i / pad, b) * a.gxs_pitch + L + (i % pad);
            dst[0] = __float2half_rn(0.0f);
            dst[a.gxs_plane_elems] = __float2half_rn(0.0f);
        }
    }
    if (a.gxs_absmax && !a.gxs_planes) {   // one atomic per warp: scale of the fp16 operand split of gxs (contract_tc.cu)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned int t = __shfl_xor_sync(0xffffffffu, gmax, o);
            gmax = t > gmax ? t : gmax;
        }
        if (lane == 0 && gmax != 0u) atomicMax(a.gxs_absmax, gmax);
    }
    __syncthreads();
    for (int l = tid; l < L; l += kThreads) {
        float sl = 0.0f, sx = 0.0f;
        for (int g = 0; g < nws; ++g) { sl += s_gacc[(size_t)g * 2 * L + l]; sx += s_gacc[(size_t)g * 2 * L + L + l]; }
        a.g_fe_out[(size_t)b * L + l] = sl;
        a.g_fx_out[(size_t)b * L + l] = sx;
    }
    // KL gradients (SURVEY 8a-12): c = a_kl * 0.5 / B (1 per row)
    const float kc = a_kl * 0.5f / fB;
    const size_t o = (size_t)b * a.D;
    for (int d = tid; d < a.D; d += kThreads) {
        const KlCell k = kl_cell(a.fe_mu[o + d], a.fe_logvar[o + d], a.fx_mu[o + d], a.fx_logvar[o + d]);
        a.g_fe_mu[o + d] = kc * k.d_fe_mu;
        a.g_fe_logvar[o + d] = kc * k.d_fe_lv;
        a.g_fx_mu[o + d] = kc * k.d_fx_mu;
        a.g_fx_logvar[o + d] = kc * k.d_fx_lv;
    }
}

// Backward from the SAVED probabilities (training path, faithful mode): no erf, the special functions on the SFU
// (cell_backward_saved), so the kernel is bound by its HBM streams (reads nr, E_l, E_x; writes the gxs planes) instead of
// by instruction issue.  A warp owns 64 neighbouring labels of one batch row (a lane: two of them) and walks the S
// samples with the logit-gradient sums in registers: no shared-memory accumulators, 8-byte loads, 4-byte plane stores.
// Grid (B, G): the 64-label chunks of a row are dealt out to G CTAs so that small batches still fill the GPU.
// MASKED: an unobserved cell gets the cotangent of indiv_prob / indiv_prob_label alone (y, cn, cp, cq read as 0).
// LW: a lane loads its two labels' weights once per chunk; cell_backward_saved weighs the log-likelihood coefficient.
template <bool MASKED, bool LW>
__global__ void __launch_bounds__(kThreads, 4)
probit_row_bwd_saved_kernel(const RowArgs a) {
    extern __shared__ float s_coef[];   // [S][6]: cn_l, cn_x, cp_l, cp_x, cq_l, cq_x
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.L, S = a.S;
    const RowCoeffs rc = row_coeffs(a, b);
    for (int s = tid; s < S; s += kThreads) {
        const size_t o = (size_t)b * S + s;
        const float4 st = reinterpret_cast<const float4*>(a.stat)[o];
        const float2 w = reinterpret_cast<const float2*>(a.wts)[o];
        float* c = s_coef + s * 6;
        c[0] = rc.cnb[0] * w.x;           c[1] = rc.cnb[1] * w.y;
        c[2] = -5.0f * rc.kb[0] * st.y;   c[3] = -5.0f * rc.kb[1] * st.w;   // x neg sums
        c[4] = 5.0f * rc.kb[0] * st.x;    c[5] = 5.0f * rc.kb[1] * st.z;    // x pos sums
    }
    __syncthreads();
    const float fS = (float)S, fB = mean_div(a);
    const bool has_gp = a.g_indiv_prob != nullptr, has_gpl = a.g_indiv_prob_label != nullptr;
    const float gscale = a.gxs_planes ? scale_from_absmax_bits(*a.gxs_scale) : 1.0f;
    // chunks of 64 labels; with operand planes the chunks run to the plane pitch (a multiple of 64): pad columns get zeros
    const int nchunks = a.gxs_planes ? a.gxs_pitch / 64 : (L + 63) / 64;
    const size_t yoff = (size_t)b * L;
    // FULL: all 64 labels of the chunk lie inside the row (every chunk but a row's last and the plane pitch's padding)
    auto chunk = [&](int c, auto full) {
        constexpr bool FULL = decltype(full)::value;
        const int l0 = c * 64 + 2 * lane;
        const bool in0 = FULL || l0 < L, in1 = FULL || l0 + 1 < L;
        float y0 = 0.f, y1 = 0.f, fe0 = 0.f, fe1 = 0.f, fx0 = 0.f, fx1 = 0.f, gpl0 = 0.f, gpl1 = 0.f, gpx0 = 0.f, gpx1 = 0.f;
        bool ob0 = true, ob1 = true;
        if (MASKED) { ob0 = in0 && a.mask[yoff + l0] != 0; ob1 = in1 && a.mask[yoff + l0 + 1] != 0; }
        if (in0) { if (ob0) y0 = a.y[yoff + l0]; fe0 = a.fe_out[yoff + l0]; fx0 = a.fx_out[yoff + l0]; }
        if (in1) { if (ob1) y1 = a.y[yoff + l0 + 1]; fe1 = a.fe_out[yoff + l0 + 1]; fx1 = a.fx_out[yoff + l0 + 1]; }
        if (has_gpl) { if (in0) gpl0 = a.g_indiv_prob_label[yoff + l0] / fS; if (in1) gpl1 = a.g_indiv_prob_label[yoff + l0 + 1] / fS; }
        if (has_gp) { if (in0) gpx0 = a.g_indiv_prob[yoff + l0] / fS; if (in1) gpx1 = a.g_indiv_prob[yoff + l0 + 1] / fS; }
        float w00 = 1.f, w01 = 1.f, w10 = 1.f, w11 = 1.f;   // w<y><label>
        if (LW) {
            if (in0) { w00 = a.label_weight[l0]; w10 = a.label_weight[L + l0]; }
            if (in1) { w01 = a.label_weight[l0 + 1]; w11 = a.label_weight[L + l0 + 1]; }
        }
        float gl0 = 0.f, gl1 = 0.f, gx0 = 0.f, gx1 = 0.f;
        // rows are 16-byte aligned (ldn % 4 == 0) and l0 is even: 8-byte loads; columns [L, ldn) of the cubes are pitch
        // padding that is never read as a label (in0 / in1)
        const bool pair = FULL || l0 + 1 < a.ldn;
        struct Cell3 { float2 n, l, x; };
        auto load = [&](int s) {
            Cell3 v;
            v.n = v.l = v.x = make_float2(0.f, 0.f);
            if (s < S && in0) {
                const size_t o = row_of(a, s, b) * a.ldn + l0;
                if (pair) {
                    v.n = __ldcs(reinterpret_cast<const float2*>(a.nr + o));
                    v.l = __ldcs(reinterpret_cast<const float2*>(a.E_l + o));
                    v.x = __ldcs(reinterpret_cast<const float2*>(a.E_x + o));
                } else {
                    v.n.x = a.nr[o]; v.l.x = a.E_l[o]; v.x.x = a.E_x[o];
                }
            }
            return v;
        };
        Cell3 cur[2] = {load(0), load(1)};
        for (int s0 = 0; s0 < S; s0 += 2) {
            const Cell3 nxt[2] = {load(s0 + 2), load(s0 + 3)};   // the next two samples' loads in flight meanwhile
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int s = s0 + i;
                if (s >= S) continue;
                const float* cf = s_coef + s * 6;
                const Cell3& v = cur[i];
                float d0 = 0.f, d1 = 0.f;
                if (in0) {
                    const float dl = cell_backward_saved<LW>(v.n.x + fe0, v.l.x, y0, ob0 ? cf[0] : 0.0f, ob0 ? cf[2] : 0.0f,
                                                             ob0 ? cf[4] : 0.0f, gpl0, w00, w10);
                    const float dx = cell_backward_saved<LW>(v.n.x + fx0, v.x.x, y0, ob0 ? cf[1] : 0.0f, ob0 ? cf[3] : 0.0f,
                                                             ob0 ? cf[5] : 0.0f, gpx0, w00, w10);
                    gl0 += dl; gx0 += dx; d0 = dl + dx;
                }
                if (in1) {
                    const float dl = cell_backward_saved<LW>(v.n.y + fe1, v.l.y, y1, ob1 ? cf[0] : 0.0f, ob1 ? cf[2] : 0.0f,
                                                             ob1 ? cf[4] : 0.0f, gpl1, w01, w11);
                    const float dx = cell_backward_saved<LW>(v.n.y + fx1, v.x.y, y1, ob1 ? cf[1] : 0.0f, ob1 ? cf[3] : 0.0f,
                                                             ob1 ? cf[5] : 0.0f, gpx1, w01, w11);
                    gl1 += dl; gx1 += dx; d1 = dl + dx;
                }
                if (a.gxs_planes) {
                    // operand planes of gxs^T . noise: hi = fp16(g s), lo = fp16(g s - hi); two labels per 4-byte store
                    const float g0 = d0 * gscale, g1 = d1 * gscale;
                    const __half2 hi = __floats2half2_rn(g0, g1);
                    const float2 hf = __half22float2(hi);
                    const __half2 lo = __floats2half2_rn(g0 - hf.x, g1 - hf.y);
                    __half* __restrict__ dst = a.gxs_planes + row_of(a, s, b) * a.gxs_pitch + l0;
                    *reinterpret_cast<__half2*>(dst) = hi;
                    *reinterpret_cast<__half2*>(dst + a.gxs_plane_elems) = lo;
                } else if (a.gxs) {
                    const size_t o = row_of(a, s, b) * a.ldn + l0;
                    if (in0) a.gxs[o] = d0;
                    if (in1) a.gxs[o + 1] = d1;
                }
            }
            cur[0] = nxt[0]; cur[1] = nxt[1];
        }
        if (in0) { a.g_fe_out[yoff + l0] = gl0; a.g_fx_out[yoff + l0] = gx0; }
        if (in1) { a.g_fe_out[yoff + l0 + 1] = gl1; a.g_fx_out[yoff + l0 + 1] = gx1; }
    };
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        if ((c + 1) * 64 <= L) chunk(c, std::true_type{});
        else chunk(c, std::false_type{});
    }
    if (blockIdx.y == 0) {   // KL gradients (SURVEY 8a-12): c = a_kl * 0.5 / B (1 per row)
        const float kc = rc.a_kl * 0.5f / fB;
        const size_t o = (size_t)b * a.D;
        for (int d = tid; d < a.D; d += kThreads) {
            const KlCell k = kl_cell(a.fe_mu[o + d], a.fe_logvar[o + d], a.fx_mu[o + d], a.fx_logvar[o + d]);
            a.g_fe_mu[o + d] = kc * k.d_fe_mu;
            a.g_fe_logvar[o + d] = kc * k.d_fe_lv;
            a.g_fx_mu[o + d] = kc * k.d_fx_mu;
            a.g_fx_logvar[o + d] = kc * k.d_fx_lv;
        }
    }
}

// ------------------------------------------------------------------------------------------------ small regime
// Label / rank sets that fit an SM (L, Z <= 128, L * Z <= 8192: the mirflickr, yeast and NUS-WIDE shapes of BASELINE.json)
// are not GEMM-shaped work: the whole forward of a batch row is ONE CTA of ONE launch.
//   R (L x Z fp32)  staged in shared memory by a TMA bulk copy (cp.async.bulk + mbarrier)
//   noise           Philox4x32-10 + Box-Muller in registers, two sample rows at a time per warp (or read from the
//                   caller's tensor), staged through 2 x Z floats of shared memory per warp; also written out as fp32
//                   for the backward's g_R product
//   contraction     nr[s, l] = sum_z noise[s, z] R[l, z]: a lane per label, warp-level FMA chain in k order -- the same
//                   chain as contract_fma.cu, so the two paths agree bit for bit
//   row math        cell_forward for both branches; label sums by warp shuffles; prediction sums in the sample order of
//                   the other forward kernels (pair sums, then pairs in order), so predictions are bit-equal too
//   tail            row_tail(): KL, log-mean-exp over samples, softmax weights, ranking sums, last-CTA batch means
// The backward is one CTA per row as well (cell_backward_saved from the kept E and nr, logit gradients, KL gradients)
// and leaves the row's contribution to g_R = gxs^T . noise in a scratch slab; a second, tiny kernel adds the slabs over
// the batch in row order (deterministic).  R staging, the noise draw and the contraction are small_rows.cuh's.
// MASKED, LW: unobserved cells and label weights as in probit_row_fwd_tiled_kernel.
template <bool STABLE, bool MASKED, bool LW>
__global__ void __launch_bounds__(kSmallThreads)
probit_small_fwd_kernel(const SmallArgs p) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ __align__(8) unsigned long long s_bar;
    const RowArgs& a = p.a;
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.L, S = a.S, Z = p.Z, B = a.B;
    const int npairs = (S + 1) >> 1;
    float* Rs = reinterpret_cast<float*>(s_raw);                           // [L][Z]
    float* nz = Rs + (((size_t)L * Z + 3) & ~(size_t)3);                   // [kSmallWarps][2][Z]
    float* ps = nz + (size_t)kSmallWarps * 2 * Z;                               // [npairs][2][L] pair sums of E
    const bool bulk = small_r_stage<kSmallThreads>(Rs, p.r, L, Z, &s_bar);
    // this lane's labels (L <= 128: at most four 32-label chunks)
    const int nch = (L + 31) >> 5;
    float yv[4], fev[4], fxv[4], w0v[4], w1v[4];
    bool ov[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int l = (c << 5) + lane;
        yv[c] = fev[c] = fxv[c] = 0.f;
        if (c < nch && l < L) { yv[c] = a.y[(size_t)b * L + l]; fev[c] = a.fe_out[(size_t)b * L + l]; fxv[c] = a.fx_out[(size_t)b * L + l]; }
        if (LW) {
            w0v[c] = w1v[c] = 0.f;
            if (c < nch && l < L) { w0v[c] = a.label_weight[l]; w1v[c] = a.label_weight[L + l]; }
        }
        if (MASKED) {
            ov[c] = c < nch && l < L && a.mask[(size_t)b * L + l] != 0;
            if (!ov[c]) yv[c] = 0.f;
        }
    }
    small_r_wait(bulk, &s_bar);
    __syncthreads();
    // ---- pairs of samples, a warp each ----
    const uint2 off = philox_offset(p.off, p.off_dev);
    float* nzw = nz + (size_t)warp * 2 * Z;
    for (int pair = warp; pair < npairs; pair += kSmallWarps) {
        const int s0 = pair << 1;
        const bool two = s0 + 1 < S;
        small_noise_pair(nzw, p, s0, b, off, lane);
        __syncwarp();
        if (p.noise_out) {
            for (int i = 0; i < (two ? 2 : 1); ++i)
                for (int z = lane; z < Z; z += 32) p.noise_out[((size_t)(s0 + i) * B + b) * Z + z] = nzw[i * Z + z];
        }
        double lpl[2] = {0.0, 0.0}, lpx[2] = {0.0, 0.0};
        float pn[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int l = (c << 5) + lane;
            if (c >= nch || l >= L) continue;
            float acc0, acc1;
            small_nr_pair(Rs + (size_t)l * Z, nzw, Z, acc0, acc1);
            float pl = 0.f, px = 0.f;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (s0 + i >= S) continue;
                const float nr = i == 0 ? acc0 : acc1;
                const CellFwd cl = cell_forward<STABLE, LW>(nr + fev[c], yv[c], LW ? w0v[c] : 1.f, LW ? w1v[c] : 1.f);   // mpvae.py:168,177
                const CellFwd cx = cell_forward<STABLE, LW>(nr + fxv[c], yv[c], LW ? w0v[c] : 1.f, LW ? w1v[c] : 1.f);   // mpvae.py:170,180
                if (!MASKED || ov[c]) {
                    lpl[i] += (double)cl.ll; lpx[i] += (double)cx.ll;
                    pn[i][0] += cl.epos; pn[i][1] += cl.eneg; pn[i][2] += cx.epos; pn[i][3] += cx.eneg;
                }
                pl += cl.E; px += cx.E;
                if (p.nr_out) {   // kept for the backward (training)
                    const size_t o = row_of(a, s0 + i, b) * a.ldn + l;
                    p.nr_out[o] = nr; a.E_l[o] = cl.E; a.E_x[o] = cx.E;
                }
            }
            ps[((size_t)pair * 2 + 0) * L + l] = pl;
            ps[((size_t)pair * 2 + 1) * L + l] = px;
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            if (s0 + i >= S) continue;
            lpl[i] = warp_sum(lpl[i]); lpx[i] = warp_sum(lpx[i]);
#pragma unroll
            for (int q = 0; q < 4; ++q) pn[i][q] = warp_sum(pn[i][q]);
            if (lane == 0) {
                const size_t o = (size_t)b * S + s0 + i;
                a.lp[o * 2 + 0] = lpl[i]; a.lp[o * 2 + 1] = lpx[i];
                reinterpret_cast<float4*>(a.stat)[o] = make_float4(pn[i][0], pn[i][1], pn[i][2], pn[i][3]);
            }
        }
        __syncwarp();   // nzw is rewritten by the next pair
    }
    __syncthreads();
    // ---- predictions: mean over samples (mpvae.py:203-204), pairs added in order ----
    const float fS = (float)S;
    for (int l = tid; l < L; l += kSmallThreads) {
        float sl = 0.f, sx = 0.f;
        for (int q = 0; q < npairs; ++q) { sl += ps[((size_t)q * 2 + 0) * L + l]; sx += ps[((size_t)q * 2 + 1) * L + l]; }
        a.indiv_prob_label[(size_t)b * L + l] = sl / fS;
        a.indiv_prob[(size_t)b * L + l] = sx / fS;
    }
    row_tail<kSmallThreads, MASKED>(a, b);
}

// MASKED, LW: unobserved cells and label weights as in probit_row_bwd_saved_kernel.
template <bool MASKED, bool LW>
__global__ void __launch_bounds__(kThreads)
probit_small_bwd_kernel(const SmallArgs p) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    const RowArgs& a = p.a;
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.L, S = a.S, Z = p.Z, B = a.B;
    const int npairs = (S + 1) >> 1;
    float* coef = reinterpret_cast<float*>(s_raw);         // [S][6]
    float* gxs = coef + (size_t)S * 6;                      // [S][L]
    float* nzs = gxs + (size_t)S * L;                       // [S][Z]
    float* gsum = nzs + (size_t)S * Z;                      // [kWarps][2][L]
    const RowCoeffs rc = row_coeffs(a, b);
    for (int s = tid; s < S; s += kThreads) {
        const size_t o = (size_t)b * S + s;
        const float4 st = reinterpret_cast<const float4*>(a.stat)[o];
        const float2 w = reinterpret_cast<const float2*>(a.wts)[o];
        float* c = coef + s * 6;
        c[0] = rc.cnb[0] * w.x;           c[1] = rc.cnb[1] * w.y;
        c[2] = -5.0f * rc.kb[0] * st.y;   c[3] = -5.0f * rc.kb[1] * st.w;
        c[4] = 5.0f * rc.kb[0] * st.x;    c[5] = 5.0f * rc.kb[1] * st.z;
    }
    const float* nsrc = p.noise_ext ? p.noise_ext : p.noise_out;
    for (int i = tid; i < S * Z; i += kThreads) nzs[i] = nsrc[((size_t)(i / Z) * B + b) * Z + (i % Z)];
    for (int i = tid; i < kWarps * 2 * L; i += kThreads) gsum[i] = 0.f;
    __syncthreads();
    const float fS = (float)S, fB = mean_div(a);
    const int nch = (L + 31) >> 5;
    for (int pair = warp; pair < npairs; pair += kWarps) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int l = (c << 5) + lane;
            if (c >= nch || l >= L) continue;
            const bool ob = !MASKED || a.mask[(size_t)b * L + l] != 0;
            const float y = ob ? a.y[(size_t)b * L + l] : 0.f, fe = a.fe_out[(size_t)b * L + l], fx = a.fx_out[(size_t)b * L + l];
            const float gpl = a.g_indiv_prob_label ? a.g_indiv_prob_label[(size_t)b * L + l] / fS : 0.f;
            const float gpx = a.g_indiv_prob ? a.g_indiv_prob[(size_t)b * L + l] / fS : 0.f;
            const float w0 = LW ? a.label_weight[l] : 1.f, w1 = LW ? a.label_weight[L + l] : 1.f;
            float gl = 0.f, gx = 0.f;
            for (int i = 0; i < 2; ++i) {
                const int s = (pair << 1) + i;
                if (s >= S) break;
                const size_t o = row_of(a, s, b) * a.ldn + l;
                const float nr = a.nr[o];
                const float* cf = coef + s * 6;
                float dl, dx;
                if (ob) {
                    dl = cell_backward_saved<LW>(nr + fe, a.E_l[o], y, cf[0], cf[2], cf[4], gpl, w0, w1);
                    dx = cell_backward_saved<LW>(nr + fx, a.E_x[o], y, cf[1], cf[3], cf[5], gpx, w0, w1);
                } else {
                    dl = cell_backward_saved(nr + fe, a.E_l[o], 0.f, 0.f, 0.f, 0.f, gpl);
                    dx = cell_backward_saved(nr + fx, a.E_x[o], 0.f, 0.f, 0.f, 0.f, gpx);
                }
                gl += dl; gx += dx;
                gxs[(size_t)s * L + l] = dl + dx;
            }
            gsum[((size_t)warp * 2 + 0) * L + l] += gl;     // a warp's lane is the only writer of its entries
            gsum[((size_t)warp * 2 + 1) * L + l] += gx;
        }
    }
    __syncthreads();
    for (int l = tid; l < L; l += kThreads) {
        float sl = 0.f, sx = 0.f;
        for (int w = 0; w < kWarps; ++w) { sl += gsum[((size_t)w * 2 + 0) * L + l]; sx += gsum[((size_t)w * 2 + 1) * L + l]; }
        a.g_fe_out[(size_t)b * L + l] = sl;
        a.g_fx_out[(size_t)b * L + l] = sx;
    }
    // this row's contribution to g_R[l, z] = sum_s gxs[s, l] noise[s, z]
    if (p.partial) {
        float* out = p.partial + (size_t)b * L * Z;
        for (int e = tid; e < L * Z; e += kThreads) {
            const int l = e / Z, z = e - l * Z;
            float acc = 0.f;
            for (int s = 0; s < S; ++s) acc = fmaf(gxs[(size_t)s * L + l], nzs[(size_t)s * Z + z], acc);
            out[e] = acc;
        }
    }
    const float kc = rc.a_kl * 0.5f / fB;
    const size_t o = (size_t)b * a.D;
    for (int d = tid; d < a.D; d += kThreads) {
        const KlCell k = kl_cell(a.fe_mu[o + d], a.fe_logvar[o + d], a.fx_mu[o + d], a.fx_logvar[o + d]);
        a.g_fe_mu[o + d] = kc * k.d_fe_mu;
        a.g_fe_logvar[o + d] = kc * k.d_fe_lv;
        a.g_fx_mu[o + d] = kc * k.d_fx_mu;
        a.g_fx_logvar[o + d] = kc * k.d_fx_lv;
    }
}

// g_R[e] = sum_b partial[b][e], rows added in order (deterministic)
__global__ void __launch_bounds__(256)
small_gr_reduce_kernel(const float* __restrict__ partial, float* __restrict__ g_r, int B, int n) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += partial[(size_t)b * n + e];
    g_r[e] = acc;
}

__global__ void log_normal_probe_kernel(const float* __restrict__ in, float* __restrict__ out, float* __restrict__ ref, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        out[i] = MPV_LOG_NORMAL(in[i]);
        ref[i] = logf(in[i]);
    }
}

__global__ void erf_probe_kernel(const float* __restrict__ in, float* __restrict__ out, float* __restrict__ ref, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        out[i] = MPV_ERF(in[i]);
        ref[i] = erff(in[i]);
    }
}

// in: groups of 32 lanes x N values (value k of lane l at in[(g * 32 + l) * N + k]); out[g * N + k]: the total of value k
// from warp_sum_transposed (written by the lane that holds it), ref[g * N + k]: warp_sum's total from lane 0
template <int N, typename T>
__global__ void warp_sum_probe_kernel(const T* __restrict__ in, T* __restrict__ out, T* __restrict__ ref, int groups) {
    const int lane = threadIdx.x & 31;
    for (int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < groups; g += gridDim.x * (blockDim.x >> 5)) {
        T v[N];
#pragma unroll
        for (int k = 0; k < N; ++k) {
            v[k] = in[((size_t)g * 32 + lane) * N + k];
            const T r = warp_sum(v[k]);
            if (lane == 0) ref[(size_t)g * N + k] = r;
        }
        warp_sum_transposed(v, lane);
        constexpr int shift = N == 1 ? 5 : N == 2 ? 4 : N == 4 ? 3 : N == 8 ? 2 : N == 16 ? 1 : 0;
        if ((lane & ((1 << shift) - 1)) == 0) out[(size_t)g * N + (lane >> shift)] = v[0];
    }
}

// f(std::true_type / std::false_type): a run-time choice as a kernel's template flag (decltype(flag)::value)
template <typename F>
void with_flag(bool v, F&& f) {
    if (v) f(std::true_type{});
    else f(std::false_type{});
}
template <typename F>
void for_both(F&& f) {
    f(std::false_type{});
    f(std::true_type{});
}

int pick_nwl(int L) {
    const int nchunks = (L + 31) / 32;
    int nwl = 1;
    while (nwl < nchunks && nwl < kWarps) nwl <<= 1;
    return nwl;
}

}  // namespace

size_t row_smem_bytes(int L) {
    const int nwl = pick_nwl(L);
    return (size_t)(kWarps / nwl) * 2 * (size_t)L * sizeof(float);
}

int device_slot() {
    int d = 0;
    cudaGetDevice(&d);
    return (d >= 0 && d < kMaxDevices) ? d : 0;
}

// ---- small regime (see probit_small_fwd_kernel) ----
static size_t small_fwd_smem(int S, int L, int Z) {
    return ((((size_t)L * Z + 3) & ~(size_t)3) + (size_t)kSmallWarps * 2 * Z + (size_t)((S + 1) / 2) * 2 * L) * sizeof(float);
}
static size_t small_bwd_smem(int S, int L, int Z) {
    return ((size_t)S * 6 + (size_t)S * L + (size_t)S * Z + (size_t)kWarps * 2 * L) * sizeof(float);
}
bool small_regime_fits(int S, int B, int L, int Z) {
    if (L > 128 || Z > 128 || L < 1 || Z < 1 || (long long)L * Z > 8192) return false;
    return small_fwd_smem(S, L, Z) <= 160 * 1024 && small_bwd_smem(S, L, Z) <= 160 * 1024;
}
size_t small_partial_bytes(int B, int L, int Z) { return (size_t)B * L * Z * sizeof(float); }

int launch_small_forward(RowArgs a, const SmallNoise& n, cudaStream_t stream) {
    const size_t smem = small_fwd_smem(a.S, a.L, n.Z);
    static bool configured[kMaxDevices] = {};
    const int dev = device_slot();
    if (!configured[dev]) {
        cudaError_t e = cudaSuccess;
        auto allow = [&](const void* k) {
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        };
        for_both([&](auto m) {
            for_both([&](auto lw) {
                constexpr bool M = decltype(m)::value, LW = decltype(lw)::value;
                allow((const void*)probit_small_fwd_kernel<false, M, LW>);
                allow((const void*)probit_small_fwd_kernel<true, M, LW>);
                allow((const void*)probit_small_bwd_kernel<M, LW>);
            });
        });
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(small): %s", cudaGetErrorString(e)); return 4; }
        configured[dev] = true;
    }
    const SmallArgs p = small_args(a, n);
    with_flag(a.stable, [&](auto st) {
        with_flag(a.mask != nullptr, [&](auto m) {
            with_flag(a.label_weight != nullptr, [&](auto lw) {
                probit_small_fwd_kernel<decltype(st)::value, decltype(m)::value, decltype(lw)::value>
                    <<<a.B, kSmallThreads, smem, stream>>>(p);
            });
        });
    });
    return check_launch("probit_small_fwd_kernel");
}

int launch_small_backward(RowArgs a, const SmallNoise& n, float* g_r, cudaStream_t stream) {
    const SmallArgs p = small_args(a, n);
    with_flag(a.mask != nullptr, [&](auto m) {
        with_flag(a.label_weight != nullptr, [&](auto lw) {
            probit_small_bwd_kernel<decltype(m)::value, decltype(lw)::value>
                <<<a.B, kThreads, small_bwd_smem(a.S, a.L, n.Z), stream>>>(p);
        });
    });
    if (int rc = check_launch("probit_small_bwd_kernel")) return rc;
    if (g_r == nullptr) return 0;
    const int cnt = a.L * n.Z;
    small_gr_reduce_kernel<<<ceil_div(cnt, 256), 256, 0, stream>>>(n.partial, g_r, a.B, cnt);
    return check_launch("small_gr_reduce_kernel");
}

int launch_log_normal_probe(const float* in, float* out, float* ref, size_t n, cudaStream_t stream) {
    log_normal_probe_kernel<<<4 * kNumSMs, 256, 0, stream>>>(in, out, ref, n);
    return check_launch("log_normal_probe_kernel");
}

int launch_erf_probe(const float* in, float* out, float* ref, size_t n, cudaStream_t stream) {
    erf_probe_kernel<<<4 * kNumSMs, 256, 0, stream>>>(in, out, ref, n);
    return check_launch("erf_probe_kernel");
}

// the two shapes the tiled forward reduces: eight float sums and four double sums per (sample pair, chunk)
int launch_warp_sum_probe(const void* in, void* out, void* ref, int groups, bool fp64, cudaStream_t stream) {
    const int grid = ceil_div(groups, kWarps) < 4 * kNumSMs ? ceil_div(groups, kWarps) : 4 * kNumSMs;
    if (fp64)
        warp_sum_probe_kernel<4, double><<<grid, kThreads, 0, stream>>>(static_cast<const double*>(in), static_cast<double*>(out),
                                                                        static_cast<double*>(ref), groups);
    else
        warp_sum_probe_kernel<8, float><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(in), static_cast<float*>(out),
                                                                       static_cast<float*>(ref), groups);
    return check_launch("warp_sum_probe_kernel");
}

int row_chunks(int L) { return (L + kChunk - 1) / kChunk; }

// Forward = cell work tiled over (row, 128-label chunk) + the per-row tail over the chunk partials.  a.part must hold
// B * S * row_chunks(L) FusePart records.
int launch_row_forward(RowArgs a, cudaStream_t stream) {
    if (a.part == nullptr) { set_error("row forward: no scratch for the chunk partials"); return 1; }
    const int nchunks = row_chunks(a.L);
    // enough CTAs for ~2 waves of 4 resident CTAs per SM, at most one CTA per 8 chunks (a warp each)
    int gy = ceil_div(2 * 2 * kNumSMs, a.B);
    if (gy > ceil_div(nchunks, kWarps)) gy = ceil_div(nchunks, kWarps);
    if (gy < 1) gy = 1;
    FusePart* part = const_cast<FusePart*>(a.part);
    // two CTAs of 256 threads per SM (<= 128 registers: sixteen cells in flight per lane, no spills); measured equal
    // to or faster than three (80 registers, spills) and four (64) on B200
    const dim3 grid(a.B, gy);
    with_flag(a.stable, [&](auto st) {
        with_flag(a.mask != nullptr, [&](auto m) {
            with_flag(a.label_weight != nullptr, [&](auto lw) {
                probit_row_fwd_tiled_kernel<decltype(st)::value, 2, decltype(m)::value, decltype(lw)::value>
                    <<<grid, kThreads, 0, stream>>>(a, part, nchunks);
            });
        });
    });
    if (int rc = check_launch("probit_row_fwd_tiled_kernel")) return rc;
    a.part_tiles = nchunks;
    return launch_row_finalize(a, stream);
}

int launch_row_finalize(RowArgs a, cudaStream_t stream) {
    if (a.part == nullptr || a.part_tiles <= 0) { set_error("row finalize: no partials"); return 1; }
    if (a.mask) probit_row_finalize_kernel<true><<<a.B, kThreads, 0, stream>>>(a);
    else probit_row_finalize_kernel<false><<<a.B, kThreads, 0, stream>>>(a);
    return check_launch("probit_row_finalize_kernel");
}

int launch_gxs_bound(RowArgs a, const unsigned int* gp_absmax, unsigned int* out_bits, const unsigned int* lw_absmax,
                     cudaStream_t stream) {
    with_flag(a.mask != nullptr, [&](auto m) {
        with_flag(a.label_weight != nullptr, [&](auto lw) {
            gxs_bound_kernel<decltype(m)::value, decltype(lw)::value>
                <<<ceil_div(a.B * a.S, 256), 256, 0, stream>>>(a, gp_absmax, out_bits, lw_absmax);
        });
    });
    return check_launch("gxs_bound_kernel");
}

int launch_row_backward(RowArgs a, cudaStream_t stream) {
    if (a.E_l != nullptr && a.E_x != nullptr && !a.stable) {
        const size_t smem = (size_t)a.S * 6 * sizeof(float);
        if (smem > 48 * 1024) { set_error("n_sample %d: per-sample coefficients exceed 48 KiB of shared memory", a.S); return 3; }
        const int nchunks = a.gxs_planes ? a.gxs_pitch / 64 : (a.L + 63) / 64;
        // enough CTAs for ~2 waves of 4 resident CTAs per SM, at most one CTA per 8 chunks (a warp each)
        int gy = ceil_div(2 * 4 * kNumSMs, a.B);
        if (gy > ceil_div(nchunks, kWarps)) gy = ceil_div(nchunks, kWarps);
        if (gy < 1) gy = 1;
        with_flag(a.mask != nullptr, [&](auto m) {
            with_flag(a.label_weight != nullptr, [&](auto lw) {
                probit_row_bwd_saved_kernel<decltype(m)::value, decltype(lw)::value><<<dim3(a.B, gy), kThreads, smem, stream>>>(a);
            });
        });
        return check_launch("probit_row_bwd_saved_kernel");
    }
    a.nwl = pick_nwl(a.L);
    const size_t smem = row_smem_bytes(a.L);
    if (smem > 200 * 1024) { set_error("label_dim %d needs %zu B of shared memory per row (limit 200 KiB)", a.L, smem); return 3; }
    static bool configured[kMaxDevices] = {};
    const int dev = device_slot();
    if (smem > 48 * 1024 && !configured[dev]) {
        cudaError_t e = cudaSuccess;
        for_both([&](auto st) {
            for_both([&](auto m) {
                for_both([&](auto lw) {
                    const void* k = (const void*)probit_row_bwd_kernel<decltype(st)::value, decltype(m)::value, decltype(lw)::value>;
                    if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
                });
            });
        });
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(bwd): %s", cudaGetErrorString(e)); return 4; }
        configured[dev] = true;
    }
    with_flag(a.stable, [&](auto st) {
        with_flag(a.mask != nullptr, [&](auto m) {
            with_flag(a.label_weight != nullptr, [&](auto lw) {
                probit_row_bwd_kernel<decltype(st)::value, decltype(m)::value, decltype(lw)::value><<<a.B, kThreads, smem, stream>>>(a);
            });
        });
    });
    return check_launch("probit_row_bwd_kernel");
}

}  // namespace mpv
