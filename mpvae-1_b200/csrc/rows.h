// Internal launch interfaces shared by the .cu translation units of libmpvae_b200.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace mpv {

struct FusePart;   // fused_rows.cuh

// Arguments of the per-row kernels (probit_rows.cu).  Pointers are device pointers.
struct RowArgs {
    int S, B, L, D;
    // row of (sample s, batch row b) in the (S*B)-row scratch matrices nr / gxs / gxs planes = b * row_sb + s * row_ss:
    // s-major (1, B) behind the CUDA-core contraction, b-major (S, 1) behind the tensor engine
    int row_sb, row_ss;
    int nwl;        // warps along the label axis (filled by the launcher)
    int sanitize;   // MPVAE_FLAG_SANITIZE_DEGENERATE
    int stable;     // MPVAE_FLAG_STABLE_CDF
    float nll_coeff, c_coeff;
    const float *y, *fe_out, *fx_out, *fe_mu, *fe_logvar, *fx_mu, *fx_logvar;
    int ldn;           // row pitch (floats) of nr and gxs: L rounded up to a multiple of 4 (16-byte aligned rows)
    const float* nr;   // (S*B,ldn) noise.R^T
    // fused forward (tensor engine): per-(sample-row, tile) partial sums left by the product kernel's math warps; the
    // finalize kernel adds them over the part_tiles column tiles in a fixed order
    const FusePart* part;
    int part_tiles;
    // training forward: the clamped probabilities of both branches, (S*B, ldn) each, kept for the backward (which then
    // needs no erf); nullptr on the inference path
    float *E_l, *E_x;
    // saved statistics (workspace)
    double* lp;        // (B,S,2)  Bernoulli log-likelihood per sample: label branch, feature branch
    float* stat;       // (B,S,4)  pos_l, neg_l, pos_x, neg_x ranking factors
    float* wts;        // (B,S,2)  softmax_s(lp)
    float* rowaux;     // (B,2)    n_pos, n_neg
    double* rowout;    // (B,8)    per-row nll_l, nll_x, c_l, c_x, kl
    unsigned int* counter;
    // forward outputs
    float* scalars[6];
    float *indiv_prob, *indiv_prob_label;
    // backward
    const float* g_scalars[6];
    const float *g_indiv_prob, *g_indiv_prob_label;
    float *g_fe_out, *g_fx_out, *g_fe_mu, *g_fe_logvar, *g_fx_mu, *g_fx_logvar;
    float* gxs;        // (S,B,L) gx_l + gx_x, or nullptr when R needs no gradient
    unsigned int* gxs_absmax;   // max |gxs| as fp32 bits (atomicMax), or nullptr; feeds the fp16 operand scale
    // tensor engine, fp16 kind: gxs is written straight as the hi|lo operand planes of the g_R product
    // ([2][S*B][gxs_pitch] halves, scale from the bound launch_gxs_bound left in *gxs_scale) instead of as fp32
    __half* gxs_planes;
    size_t gxs_plane_elems;     // distance between the hi and the lo plane
    int gxs_pitch;
    const unsigned int* gxs_scale;
    // partially labelled rows: (B, L) bytes, nonzero = the label is observed; nullptr = every label is observed.  The
    // launchers pick the kernels' MASKED instantiation from it: an unobserved cell keeps E and the predictions but adds
    // nothing to the log-likelihood, the ranking sums or the label counts, and its logit gradient is the cotangent of
    // indiv_prob / indiv_prob_label alone.  Whatever y holds there is never read into the arithmetic.
    const uint8_t* mask;
};

size_t row_smem_bytes(int L);
// cudaFuncAttributeMaxDynamicSharedMemorySize is per device: launchers set it once per device (device_slot() <
// kMaxDevices), so that later launches (e.g. under CUDA-graph capture) make no driver calls
constexpr int kMaxDevices = 64;
int device_slot();
// Small regime (L, Z <= 128, L * Z <= 8192): the whole forward of a batch row in one CTA of one launch (probit_rows.cu).
struct SmallNoise {
    const float* r;            // (L, Z) fp32
    int Z;
    const float* noise_ext;    // caller's (S, B, Z) noise, or nullptr: Philox inside the kernel
    float* noise_out;          // fp32 (S, B, Z) copy kept for the backward (training), or nullptr
    float* nr_out;             // (S*B, ldn) noise.R^T kept for the backward (training), or nullptr
    int Bg, row0;
    uint64_t seed, offset;
    const uint64_t* offset_dev;
    float* partial;            // backward: (B, L*Z) scratch for the per-row contributions to g_R, or nullptr
};
bool small_regime_fits(int S, int B, int L, int Z);
size_t small_partial_bytes(int B, int L, int Z);
int launch_small_forward(RowArgs a, const SmallNoise& n, cudaStream_t stream);
// g_r may be nullptr (R frozen); needs the forward's kept nr / E / noise
int launch_small_backward(RowArgs a, const SmallNoise& n, float* g_r, cudaStream_t stream);
int launch_log_normal_probe(const float* in, float* out, float* ref, size_t n, cudaStream_t stream);   // test hook
int row_chunks(int L);   // 64-label chunks of a row: launch_row_forward needs B * S * row_chunks(L) FusePart records in a.part
int launch_row_forward(RowArgs a, cudaStream_t stream);
// the tail of the forward when the product kernel has already done the cell work (a.part != nullptr)
int launch_row_finalize(RowArgs a, cudaStream_t stream);
int launch_row_backward(RowArgs a, cudaStream_t stream);
// *out_bits = fp32 bits of an upper bound of max |gxs| over the whole batch (NaN for non-sanitised degenerate rows),
// from the saved per-(row, sample) statistics and the upstream cotangents; gp_absmax: two slots holding max |g_indiv_prob|
// and max |g_indiv_prob_label| as fp32 bits (zero when absent)
int launch_gxs_bound(RowArgs a, const unsigned int* gp_absmax, unsigned int* out_bits, cudaStream_t stream);

// Prediction only (predict.cu): a.indiv_prob = mean_s E(nr + fx_out), the feature branch alone -- no labels, no
// log-likelihoods, no ranking factors, no per-row tail.  Same E and the same sample order as the forward kernels.
int launch_predict_rows(RowArgs a, cudaStream_t stream);                           // after the nt product (a.nr)
int launch_small_predict(RowArgs a, const SmallNoise& n, cudaStream_t stream);     // small regime, one launch

// Conditional prediction (predict.cu), after the nt product (a.nr): a.indiv_prob = the importance-weighted mean of E
// over the samples, weighted by the likelihood of the row's observed labels (observed (B, L) int8: 0 / 1 observed, any
// other value unobserved); log_evidence (B), ess (B).  Uses part (B * S * row_chunks(L) records), a.lp, a.wts, a.rowaux.
int launch_conditional_rows(RowArgs a, const int8_t* observed, FusePart* part, float* log_evidence, float* ess,
                            cudaStream_t stream);
// Its last two passes: the per-row log-mean-exp of lp_s (the sum of part_chunks FusePart records per sample from part,
// or a.lp itself when part is nullptr), then the weighted mean of E over the samples of a.nr.
int launch_conditional_tail(RowArgs a, const int8_t* observed, const FusePart* part, int part_chunks, float* log_evidence,
                            float* ess, cudaStream_t stream);

// Conditional prediction by a GHK sampler (conditional_ghk.cu), after the nt product (a.nr, overwritten with the
// conditioned samples).  Its own scratch block: G = R R^T (L, L) fp32, the G product's scratch, per row the observed
// count and index list, the fp64 Cholesky factor (mo x mo) and two fp64 (S, mo) vectors.
struct GhkLayout { size_t gram, gram_scratch, nobs, idx, fac, eta, wv, total; };
GhkLayout ghk_layout(int S, int B, int L, int mo, size_t gram_scratch);
struct GhkInputs {
    GhkLayout layout;
    void* ws;
    int max_observed;
    const int8_t* observed;
    const float* gram;                 // (L, L), read at [o_i, o_j] with o_i >= o_j and at rows o
    const float *zeta, *uniform;       // (S, B, L) or nullptr (the library's Philox draws)
    int noise_b_global, noise_row0;
    uint64_t noise_seed, noise_offset;
    const uint64_t* noise_offset_dev;
    float *log_evidence, *ess;
};
int launch_ghk_rows(RowArgs a, const GhkInputs& in, cudaStream_t stream);

// Set prediction (sets.cu).  The sampler, after the nt product (a.nr): bits (B, S, ceil(L / 32)) words of y = (U < E),
// E = predict_E(nr + fx_out), U the caller's (S, B, L) uniforms or the library's Philox stream with its own key.
struct SampleInputs {
    const float* uniform;              // (S, B, L) in (0, 1), or nullptr
    int32_t* bits;
    int noise_b_global, noise_row0;
    uint64_t noise_seed, noise_offset;
    const uint64_t* noise_offset_dev;
};
int launch_sample_labels(RowArgs a, const SampleInputs& in, cudaStream_t stream);
// The F-measure-optimal decoder, one CTA per row, and its scratch: per row the sample cardinalities and weights (S each)
// and the labels set in any sample with their Delta (L each).
struct F1Layout { size_t card, wsmp, ulist, delta, total; };
F1Layout f1_layout(int B, int S, int L);
int launch_f1_sets(const int32_t* bits, int B, int S, int L, double beta, int max_size, uint8_t* sets, double* expected_f,
                   int32_t* set_size, void* ws, cudaStream_t stream);

// Closed-form predictive distribution (predictive.cu), the S -> infinity limit of the above: per-label scales
// 1 / sqrt(1 + |R_l|^2), pair correlations, exact marginals and pair co-occurrence probabilities.  pairs: P int32 pairs
// (i, j); an index outside [0, L) gives NaN.
int launch_predictive_scale(const float* r, int L, int Z, double* scale, cudaStream_t stream);
int launch_predictive_rho(const float* r, int L, int Z, const double* scale, const int* pairs, int P, double* rho,
                          cudaStream_t stream);
int launch_predict_exact(const float* fx_out, int B, int L, const double* scale, bool stable, float* out,
                         cudaStream_t stream);
int launch_predict_pairs(const float* fx_out, int B, int L, const double* scale, const int* pairs, const double* rho, int P,
                         bool stable, float* out, cudaStream_t stream);

// CUDA-core contraction (contract_fma.cu)
//   nt: C[M,N] = A[M,K] . B[N,K]^T
//   tn: C[N1,N2] = A[M,N1]^T . B[M,N2]   (split over M, partials reduced in a fixed order)
int launch_contract_nt_fma(const float* A, const float* Bm, float* C, int M, int N, int K, cudaStream_t stream,
                           int ldc = 0);   // ldc: row pitch of C in floats (0 = N)
size_t contract_tn_fma_workspace(int M, int N1, int N2);
int launch_contract_tn_fma(const float* A, const float* Bm, float* C, int M, int N1, int N2, void* ws, size_t ws_bytes,
                           cudaStream_t stream, int lda = 0);   // lda: row pitch of A in floats (0 = N1)

// per-step metrics (metrics.cu)
size_t batch_metrics_workspace(int B, int L);
int launch_batch_metrics(const float* prob, const float* y, int B, int L, float thr, double* out, void* ws, cudaStream_t stream);
int launch_label_curves(const float* sorted_scores, const float* sorted_targets, int N, int L, double cutoff, double* out,
                        cudaStream_t stream);

// g_R summed over ranks through peer memory (peer_reduce.cu)
struct PeerCtx {
    int world, rank;
    uint32_t step;             // flag value of this exchange (strictly increasing, the same on every rank)
    uint32_t* step_dev;        // optional device counter added to `step` and advanced by step_stride after the exchange
    uint32_t step_stride;      //   (a captured CUDA graph replays the same launch arguments)
    uint32_t* epoch_dev;       // optional: the tile-counter epoch of this rank, advanced by one after the exchange
    long long timeout_cycles;  // a flag wait gives up after this many SM cycles and records the failure (peer_error_word)
    float* part[8];     // every rank's partial g_R (the rank's own product output)
    float* g_r[8];      // every rank's final g_R
    uint32_t* flags[8];
};
size_t peer_flag_bytes();
int peer_error_word();   // index of the error word inside a rank's flag block (0 = no wait has timed out)
int launch_peer_reduce(const PeerCtx& ctx, size_t n, cudaStream_t stream, size_t first = 0);   // elements [first, first + n)
// the same sum for the first n_slabs 256-row slabs of g_R, slab by slab as the product (running beside it) publishes
// them in the per-tile counters `tile_done` (peer memory); `ctas` CTAs, one per SM
int launch_peer_reduce_slabs(const PeerCtx& ctx, void* const* tile_done, int tiles_n, int n_slabs, size_t slab_elems, int ctas,
                             cudaStream_t stream);
int launch_peer_reduce_nvls(const PeerCtx& ctx, const float* mc_part, float* mc_gr, size_t n, cudaStream_t stream);

// clip_grad_norm_ + Adam over flat buffers (optim.cu)
size_t grad_norm_workspace();
int launch_grad_norm(const float* g, size_t n, void* ws, double max_norm, double grad_scale, const float* lr_dev, double lr_host,
                     double beta1, double beta2, double* state, cudaStream_t stream);
int launch_adam(void* p, int p_is_f64, const float* g, void* m, void* v, float* shadow, size_t n, const double* state,
                double beta1, double beta2, double eps, double weight_decay, cudaStream_t stream);

// Philox noise (philox.cu)
int launch_philox_normal(float* noise, int S, int B, int Z, int B_global, int row0, uint64_t seed, uint64_t offset,
                         const uint64_t* offset_dev, cudaStream_t stream);

}  // namespace mpv
