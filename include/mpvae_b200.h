/*
 * mpvae_b200.h -- C-ABI of the B200-native probit-ELBO hot path.
 *
 * Drop-in boundary for lliutianc/MPVAE-1's `compute_loss` (reference mpvae.py:145-210) and its
 * autograd backward.  The reference has no FFI (pure Python/torch), so the entry points below are what
 * a binding for this path would call; the Python mirror in mpvae-1_b200/ binds them with ctypes
 * (INTEGRATION.md shows the stub a reference maintainer would add to mpvae.py).
 *
 * Conventions
 *   - plain C types only: device pointers, sizes, a cudaStream_t passed as void*.
 *   - every buffer is owned by the caller (PyTorch's caching allocator in practice); the library
 *     never allocates or frees device memory, never synchronises the device and launches only on the
 *     given stream.
 *   - all matrices are dense row-major fp32 unless noted.  S = n_sample, B = batch rows, L = label_dim,
 *     Z = z_dim, D = latent_dim.
 *   - return value 0 = success; otherwise an error code, text via mpvae_last_error() (thread-local).
 *   - there is no CPU implementation behind this header.
 */
#ifndef MPVAE_B200_H_
#define MPVAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPVAE_ABI_VERSION 13

/* flags */
#define MPVAE_FLAG_SANITIZE_DEGENERATE 0x1u /* rows with n_pos*n_neg == 0 get zero ranking gradient instead of
                                               the reference's NaN (mpvae.py:118-121); default off = faithful */
#define MPVAE_FLAG_CONTRACT_TENSOR     0x2u /* noise.R^T and g_R on tcgen05 (split-precision fp16 pieces); default: chosen by shape */
#define MPVAE_FLAG_CONTRACT_FMA        0x4u /* force the CUDA-core FMA contraction */
#define MPVAE_FLAG_STABLE_CDF          0x8u /* opt-in: Phi and 1 - Phi from erfc(|x| / sqrt 2) (no cancellation in the tails)
                                               instead of the reference's 0.5 (1 + erf) and 1 - E.  More accurate than the
                                               reference, hence NOT within 1e-5 of it in saturated cells. */
#define MPVAE_FLAG_FUSED_FORWARD        0x10u /* dense regime, opt-in: run the row forward on extra "math" warps INSIDE the tcgen05
                                               product kernel (csrc/fused_rows.cuh) instead of as its own kernel after it.
                                               Same results bit for bit; measured slower on B200 (the product's register
                                               accumulators leave room for 8 math warps per SM, a quarter of what the row
                                               math needs to hide its latencies: profiles/r02_fused_forward.md) */

#define MPVAE_FLAG_SEPARATE_NOISE       0x20u /* dense regime, library-side noise: draw the Philox normals with a kernel of their own
                                               before the product instead of on the product kernel's math warps, just
                                               ahead of the tiles that read them (A/B measurements; same numbers) */

#define MPVAE_FLAG_SERIAL_EXCHANGE      0x80u /* data-parallel dense regime: sum g_R over the ranks only AFTER the g_R product (the
                                               stand-alone reduce kernel) instead of slab by slab on a few reserved SMs beside
                                               it (A/B measurements; same sums) */
#define MPVAE_FLAG_FUSED_EXCHANGE       0x40u /* data-parallel dense regime, opt-in: sum g_R over the ranks tile by tile INSIDE the
                                               g_R product kernel (peer_tile_done must be given) instead of with the
                                               stand-alone reduce kernel after it; same sums */

/* order of the six scalar outputs (first six entries of the 8-tuple at mpvae.py:210) */
enum { MPVAE_TOTAL = 0, MPVAE_NLL = 1, MPVAE_NLL_X = 2, MPVAE_C = 3, MPVAE_C_X = 4, MPVAE_KL = 5 };

typedef struct mpvae_probit_params {
    uint32_t struct_bytes; /* = sizeof(mpvae_probit_params), or MPVAE_PARAMS_BASE_BYTES for a caller that stops before
                              the peer_* fields (single-GPU bindings: the rest then defaults to "off"); ABI guard */
    uint32_t flags;
    int32_t S, B, L, Z, D;
    float nll_coeff; /* args.nll_coeff, mpvae.py:207 */
    float c_coeff;   /* args.c_coeff,   mpvae.py:208 */

    /* ---- inputs (device) ---- */
    const float *y;         /* (B,L) labels, input_label                      mpvae.py:145 */
    const float *fe_out;    /* (B,L) label-branch decoder logits                            */
    const float *fx_out;    /* (B,L) feature-branch decoder logits                          */
    const float *fe_mu;     /* (B,D) */
    const float *fe_logvar; /* (B,D) */
    const float *fx_mu;     /* (B,D) */
    const float *fx_logvar; /* (B,D) */
    const float *r;         /* (L,Z) r_sqrt_sigma cast to fp32                mpvae.py:165 */
    const float *noise;     /* (S,B,Z) standard normal samples                mpvae.py:162
                               NULL = draw them inside the library (Philox, fields at the end of this struct) */

    /* ---- forward outputs (device) ---- */
    float *scalars[6];       /* six 1-element outputs: total, nll, nll_x, c, c_x, kl   mpvae.py:207-210
                                (separate buffers so the host can hand them out as independent 0-dim tensors) */
    float *indiv_prob;       /* (B,L) mean_s E_x                              mpvae.py:203 */
    float *indiv_prob_label; /* (B,L) mean_s E                                mpvae.py:204 */

    /* ---- backward: upstream cotangents (device; a NULL entry = zero cotangent) ---- */
    const float *g_scalars[6];       /* d objective / d (total, nll, nll_x, c, c_x, kl), 1 element each */
    const float *g_indiv_prob;       /* (B,L) or NULL */
    const float *g_indiv_prob_label; /* (B,L) or NULL */

    /* ---- backward outputs (device; g_r may be NULL when R needs no gradient) ---- */
    float *g_fe_out, *g_fx_out;                           /* (B,L) */
    float *g_fe_mu, *g_fe_logvar, *g_fx_mu, *g_fx_logvar; /* (B,D) */
    float *g_r;                                           /* (L,Z) */

    /* ---- scratch (device), >= mpvae_workspace_bytes(); forward fills it, backward reads it ---- */
    void *workspace;
    uint64_t workspace_bytes;

    /* ---- library-side noise (noise == NULL): the numbers of mpvae_philox_normal(seed, offset, B_global, row0),
       generated straight into the layout the contraction engine wants (never materialised as fp32 in the dense
       regime).  These normals lie on the fp16 grid (Box-Muller in fp32, rounded to nearest fp16), which lets the
       tensor engine treat them as a single operand piece.  The backward must be given the same values. ---- */
    uint64_t noise_seed, noise_offset;
    int32_t noise_b_global, noise_row0;
    const uint64_t *noise_offset_dev; /* optional DEVICE counter added to noise_offset inside the kernel, so that a
                                         captured CUDA graph draws fresh noise on every replay; NULL = unused */

    /* ---- data-parallel g_R over NVLink peer memory (optional; peer_world <= 1: off).
       One process per GPU on one node: each rank allocates a partial buffer and a g_R buffer (L*Z floats each) and a
       flag block (mpvae_peer_flag_bytes) with mpvae_peer_alloc, exchanges the IPC handles and opens the others' with
       mpvae_peer_open.  With the tables filled in, mpvae_probit_backward leaves in g_r (which must be
       peer_g_r[peer_rank]) the SUM of g_R over all ranks, bit-identical on every rank: each rank's product goes to its
       own partial buffer, g_R is cut into peer_world chunks, a chunk's owner pulls it from every rank over NVLink, adds
       in rank order and stores the result to every rank (csrc/peer_reduce.cu).  peer_step must increase by one per
       call, the same number on every rank, starting at 1. ---- */
    int32_t peer_world, peer_rank;
    uint32_t peer_step, peer_reserved;
    void *peer_part[8];
    void *peer_g_r[8];
    void *peer_flags[8];
    /* optional MULTICAST addresses of the same part / g_R buffers (both or neither): the chunk owners then reduce inside
       the NVSwitch (multimem.ld_reduce / multimem.st) instead of pulling from every peer */
    void *peer_mc_part;
    void *peer_mc_g_r;
    /* optional DEVICE counter added to peer_step inside the exchange kernels and advanced by them after every exchange,
       so that a captured CUDA graph (which replays the same peer_step) keeps the flag values increasing; NULL = unused */
    uint32_t *peer_step_dev;
    /* optional: every rank's per-tile completion counters (mpvae_peer_alloc'ed, MPVAE_PEER_TILE_BYTES each, zeroed once,
       never reset: the library keeps the exchange's epoch in the buffer's last word, on the device, so captured CUDA graphs
       replay correctly).  With them the g_R product of the dense regime publishes every finished
       256 x 256 tile there and leaves a few SMs idle; an exchange kernel on those SMs (csrc/peer_reduce.cu, a side
       stream forked from and joined to the caller's) sums finished 256-row slabs of g_R over the ranks through NVLink
       while the tensor pipe computes later tiles.  MPVAE_FLAG_FUSED_EXCHANGE moves the sums onto the product kernel's
       own math warps instead (csrc/fused_rows.cuh; slower), MPVAE_FLAG_SERIAL_EXCHANGE or NULL = the stand-alone
       reduce kernel after the product.  Products of fewer than 8192 rows (S * B) always take the latter. */
    void *peer_tile_done[8];
} mpvae_probit_params;
#define MPVAE_PEER_TILE_BYTES 65536u

/* size of the struct up to (not including) peer_world: what a binding without the multi-GPU fields fills in */
#define MPVAE_PARAMS_BASE_BYTES ((uint32_t)offsetof(mpvae_probit_params, peer_world))

/* Peer-memory plumbing for the fields above (CUDA IPC; same node).  handle = 64 opaque bytes + the offset word. */
uint64_t mpvae_peer_flag_bytes(void);
/* The same exchange stand-alone: g_r[r][0..n) = sum over ranks s of part[s][0..n), on every rank r (tables of `world`
 * device pointers, this process being `rank`; `step` as peer_step above, shared with the backward's counter). */
int mpvae_peer_allreduce(void *const *part, void *const *g_r, void *const *flags, int32_t world, int32_t rank,
                         uint32_t step, uint64_t n, void *cuda_stream);
/* The same with the optional DEVICE step counter of peer_step_dev (CUDA-graph replay: flag value = step + *step_dev, the
 * exchange advances *step_dev by one).  g_r[r] may equal part[r] on every rank: the sum then replaces the partials in
 * place (an element is read and written by its owner rank only).  Table entries must be 16-byte aligned. */
int mpvae_peer_allreduce_dev(void *const *part, void *const *g_r, void *const *flags, int32_t world, int32_t rank,
                             uint32_t step, uint32_t *step_dev, uint64_t n, void *cuda_stream);
/* ... with the in-switch reduction when mc_part / mc_g_r (multicast addresses of the same buffers) are given. */
int mpvae_peer_allreduce_nvls(void *const *part, void *const *g_r, void *const *flags, void *mc_part, void *mc_g_r,
                              int32_t world, int32_t rank, uint32_t step, uint64_t n, void *cuda_stream);
/* 0 while no flag wait of this rank has timed out; otherwise the step number that was given up on (the sums of that
 * step are invalid; fall back to an NCCL all-reduce).  Waits give up after MPVAE_PEER_TIMEOUT_S seconds (default 120)
 * instead of trapping, so a slow peer (checkpoint, evaluation, data-loader stall) cannot poison the other contexts.
 * flags = this rank's own flag block; synchronises the stream it reads on. */
int mpvae_peer_error(const void *flags, uint32_t *out_step, void *cuda_stream);
int mpvae_peer_alloc(uint64_t bytes, void **ptr, unsigned char handle[64]);
int mpvae_peer_open(const unsigned char handle[64], void **ptr);
int mpvae_peer_close(void *ptr);
int mpvae_peer_free(void *ptr);

/* Bytes of scratch for one forward(+backward) call.  want_backward=0 sizes the inference path. */
uint64_t mpvae_workspace_bytes(int32_t S, int32_t B, int32_t L, int32_t Z, int32_t want_backward, uint32_t flags);

/* Forward: replaces the body of compute_loss (mpvae.py:145-210) given the noise tensor. */
int mpvae_probit_forward(const mpvae_probit_params *p, void *cuda_stream);

/* Prediction only: indiv_prob (B,L) = mean_s clamp(Phi(fx_out + noise.R^T)) (mpvae.py:170,180,203), the feature branch
 * alone -- what scoring rows without labels needs.  Reads struct_bytes, flags, S, B, L, Z, fx_out, r, noise (or the
 * library-noise fields noise_seed / noise_offset / noise_b_global / noise_row0 / noise_offset_dev), workspace /
 * workspace_bytes (mpvae_workspace_bytes(S, B, L, Z, 0, flags) suffices) and writes indiv_prob only; every other field is
 * ignored and may be NULL.  Takes the regime mpvae_probit_forward takes for the same (S, B, L, Z, flags) and returns
 * the bits of its indiv_prob for the same fx_out, R and noise. */
int mpvae_probit_predict(const mpvae_probit_params *p, void *cuda_stream);

/* Backward: the autograd backward of compute_loss (implicit in the reference, train.py:125),
 * closed form in SURVEY.md 8(a-12).  Must follow a forward on the same workspace. */
int mpvae_probit_backward(const mpvae_probit_params *p, void *cuda_stream);

/* Counter-based standard-normal noise, replaces torch.normal(0,1,(S,B,Z)) of mpvae.py:162.
 * Element (s, b_global, z) depends only on (seed, offset, s, b_global, z): a rank holding rows
 * [row0, row0+B) of a B_global-row batch draws the same numbers a single GPU would. */
int mpvae_philox_normal(float *noise, int32_t S, int32_t B, int32_t Z, int32_t B_global, int32_t row0,
                        uint64_t seed, uint64_t offset, void *cuda_stream);

/* C[M,N] = A[M,K] . B[N,K]^T (fp32).  The contraction of mpvae.py:168 as a stand-alone entry
 * (A = noise viewed (S*B, Z), B = R).  engine: 0 = auto, 1 = CUDA-core FMA, 2 = tcgen05 split-precision,
 * 3 = tcgen05 reusing the operand planes an engine-2 call left in the same workspace (GEMM kernel alone),
 * 4 = tcgen05 with the NOISE operand (A here, B of mpvae_contract_tn) promised to lie on the fp16 grid, as the
 * library's own Philox noise does: that operand is one piece and the product takes two MMA passes instead of three;
 * 5 = engine 4 reusing the planes of a previous engine-2/4 call.
 * MPVAE_ENGINE_KSPLIT or-ed into a tcgen05 engine code lets mpvae_contract_nt cut the tiles of a partial wave of its
 * persistent grid into K slices (few output tiles, long K: the MLP layers).  The loss path never sets it: there the
 * summation order of an output element must not depend on how many rows the call holds. */
#define MPVAE_ENGINE_KSPLIT 0x100
int mpvae_contract_nt(const float *A, const float *Bm, float *C, int32_t M, int32_t N, int32_t K, int32_t engine,
                      void *workspace, uint64_t workspace_bytes, void *cuda_stream);
/* Same with a row pitch of ldc >= N floats for C.  The loss kernels keep noise.R^T in rows padded to 16 bytes
 * (ldc = N rounded up to 4) so that the GEMM epilogue can use 16-byte stores; this entry times exactly that variant. */
int mpvae_contract_nt_pitched(const float *A, const float *Bm, float *C, int32_t M, int32_t N, int32_t K, int32_t ldc,
                              int32_t engine, void *workspace, uint64_t workspace_bytes, void *cuda_stream);

/* The tcgen05 engine in stages, for callers that use an operand more than once (mpvae_b200/dense.py: a layer's input
 * planes serve its forward and its weight gradient, the output-gradient planes both backward products):
 *   mpvae_tc_split      fp32 [rows][cols] -> operand planes [hi|lo][rows][pitch] (mpvae_tc_planes_bytes) + the max |x|
 *                       slot (4 bytes, device) that fixes the power-of-two scale of the fp16 pieces
 *   mpvae_tc_gemm_nt    C[M,N] (pitch ldc) = A[M,K] . B[N,K]^T from planes;  ksplit != 0 allows K-sliced partial waves
 *   mpvae_tc_gemm_tn    C[N1,N2] = A[M,N1]^T . B[M,N2] from planes
 * tail_scratch: mpvae_tc_tail_scratch_bytes() of device memory (may be NULL: no K-slicing). */
uint64_t mpvae_tc_planes_bytes(int32_t rows, int32_t cols);
uint64_t mpvae_tc_tail_scratch_bytes(void);
int mpvae_tc_split(const float *src, int32_t rows, int32_t cols, void *planes, uint32_t *absmax_slot, void *cuda_stream);
int mpvae_tc_gemm_nt(const void *a_planes, const void *b_planes, float *C, int32_t M, int32_t N, int32_t K, int32_t ldc,
                     const uint32_t *absmax_a, const uint32_t *absmax_b, int32_t ksplit, void *tail_scratch,
                     uint64_t tail_scratch_bytes, void *cuda_stream);
int mpvae_tc_gemm_tn(const void *a_planes, const void *b_planes, float *C, int32_t M, int32_t N1, int32_t N2,
                     const uint32_t *absmax_a, const uint32_t *absmax_b, void *tail_scratch, uint64_t tail_scratch_bytes,
                     void *cuda_stream);

/* C[N1,N2] = A[M,N1]^T . B[M,N2] (fp32): g_R = gx^T . noise of SURVEY 8(a-12). Same engine codes. */
int mpvae_contract_tn(const float *A, const float *Bm, float *C, int32_t M, int32_t N1, int32_t N2, int32_t engine,
                      void *workspace, uint64_t workspace_bytes, void *cuda_stream);
uint64_t mpvae_contract_workspace_bytes(int32_t M, int32_t N, int32_t K, int32_t engine);

/* Per-step metrics on the device: replaces evals.compute_metrics(indiv_prob.cpu(), input_label.cpu(), threshold,
 * all_metrics=False) of train.py:131 / fairsoft_train.py:149 (reference evals.py:178-239).
 * out[8] (device, fp64) = ACC, HA, ebF1, miF1, maF1, p@1, p@3, p@5.  workspace >= mpvae_batch_metrics_workspace. */
enum { MPVAE_M_ACC = 0, MPVAE_M_HA, MPVAE_M_EBF1, MPVAE_M_MIF1, MPVAE_M_MAF1, MPVAE_M_P1, MPVAE_M_P3, MPVAE_M_P5 };
uint64_t mpvae_batch_metrics_workspace(int32_t B, int32_t L);
int mpvae_batch_metrics(const float *indiv_prob, const float *input_label, int32_t B, int32_t L, float threshold,
                        double *out, void *workspace, uint64_t workspace_bytes, void *cuda_stream);

/* Closed-form prediction: the S -> infinity limit of mpvae_probit_predict, and the pairwise label co-occurrence of the
 * same predictive distribution.  The noise n = R eps enters linearly, so with h_l = fx_out[b, l] * scale_l,
 * scale_l = 1 / sqrt(1 + sum_z R[l, z]^2) and rho_ij = R_i . R_j * scale_i * scale_j:
 *   P(y_l = 1)          = c + k Phi(h_l)
 *   P(y_i = 1, y_j = 1) = c^2 + c k (Phi(h_i) + Phi(h_j)) + k^2 Phi2(h_i, h_j; rho_ij)
 * where E = c + k Phi is the clamp of mpvae.py:177 (c = eps1 / 2, k = 1 - eps1, eps1 = fp32(1e-6)) and Phi2 the standard
 * bivariate normal CDF (Genz's BVND, fp64).  r = (L, Z) fp32 R; pairs = (P, 2) int32, 8-byte aligned; scale (L) and rho
 * (P) are fp64 buffers the caller keeps between calls.  A pair index outside [0, L) yields NaN.
 *   mpvae_predictive_scale  scale_out[l] = scale_l (fp64 sums over z in a fixed order)
 *   mpvae_predictive_rho    rho_out[p] = rho of pair p
 *   mpvae_predict_exact     indiv_prob (B, L) = E(x') with x' = fp32(fx_out * scale) rounded once, through the same
 *                           probit_E (probit_E_stable under MPVAE_FLAG_STABLE_CDF) as every other entry point
 *   mpvae_predict_pairs     out (B, P) = P(y_i = 1, y_j = 1) in fp64, rounded once to fp32; a pair (i, i) gives the bits
 *                           of mpvae_predict_exact's P(y_i = 1) under the same flags
 * Flags other than MPVAE_FLAG_STABLE_CDF are ignored.  B = 0 or P = 0 launches nothing. */
int mpvae_predictive_scale(const float *r, int32_t L, int32_t Z, double *scale_out, void *cuda_stream);
int mpvae_predictive_rho(const float *r, int32_t L, int32_t Z, const double *scale, const int32_t *pairs, int32_t P,
                         double *rho_out, void *cuda_stream);
int mpvae_predict_exact(const float *fx_out, int32_t B, int32_t L, const double *scale, uint32_t flags, float *indiv_prob,
                        void *cuda_stream);
int mpvae_predict_pairs(const float *fx_out, int32_t B, int32_t L, const double *scale, const int32_t *pairs,
                        const double *rho, int32_t P, uint32_t flags, float *out, void *cuda_stream);

/* The tail of the training step, train.py:126-128 (clip_grad_norm_(params, max_norm); optimizer.step() with
 * torch.optim.Adam(lr, weight_decay)), over flat device buffers.
 * mpvae_grad_norm: L2 norm of g[0..n) times grad_scale (1 / world size when g holds the all-reduced SUM), and the
 *   per-step scalars the Adam kernel needs.  state (6 device doubles, persistent across steps):
 *   [0] step count, incremented by this call  [1] the norm  [2] gradient multiplier = grad_scale * min(1, max_norm /
 *   (norm + 1e-6)) (max_norm <= 0: no clipping)  [3] 1 - beta1^t  [4] sqrt(1 - beta2^t)  [5] learning rate
 *   (*lr_dev when lr_dev != NULL, else lr).  workspace >= mpvae_grad_norm_workspace() bytes.
 * mpvae_adam_step: one pass of torch.optim.Adam's update (L2 weight decay) over n elements; p, m, v are fp32 or fp64
 *   (p_is_f64: the reference's r_sqrt_sigma is an fp64 Parameter), g is always fp32; shadow_f32 (optional) receives
 *   the updated parameter as fp32. */
uint64_t mpvae_grad_norm_workspace(void);
int mpvae_grad_norm(const float *g, uint64_t n, double max_norm, double grad_scale, const float *lr_dev, double lr,
                    double beta1, double beta2, double *state, void *workspace, uint64_t workspace_bytes, void *cuda_stream);
int mpvae_adam_step(void *p, int32_t p_is_f64, const float *g, void *m, void *v, float *shadow_f32, uint64_t n,
                    const double *state, double beta1, double beta2, double eps, double weight_decay, void *cuda_stream);

/* Per-label ranking curves of evals.compute_metrics(..., all_metrics=True) (evals.py:129-175; the reference calls
 * scikit-learn's roc_auc_score / precision_recall_curve + auc per label, 27 times per evaluation, train.py:277-289).
 * sorted_scores / sorted_targets: (N, L) row-major, every COLUMN sorted by decreasing score (targets carried along).
 * out[3][L] (device, fp64): ROC AUC (NaN when a class is absent), area under the PR curve, recall at the lowest
 * threshold whose 1 - precision <= fdr_cutoff. */
int mpvae_label_curves(const float *sorted_scores, const float *sorted_targets, int32_t N, int32_t L, double fdr_cutoff,
                       double *out, void *cuda_stream);

/* Per-kernel device times of the loss path, measured with CUDA events recorded on the caller's stream around each
 * launch group inside mpvae_probit_forward / _backward (bench.py's roofline: the dominant kernel timed INSIDE the step).
 * mpvae_profile(1) switches it on and clears the records (not under CUDA-graph capture: it creates events);
 * mpvae_profile_read waits for the recorded events and returns the summed milliseconds and the number of records of
 * one slot; mpvae_profile_name(slot) names it (NULL past the last slot). */
enum { MPVAE_PROF_NOISE = 0, MPVAE_PROF_SPLIT_R, MPVAE_PROF_PRODUCT_NT, MPVAE_PROF_ROW_FORWARD, MPVAE_PROF_GXS_BOUND,
       MPVAE_PROF_ROW_BACKWARD, MPVAE_PROF_PRODUCT_TN, MPVAE_PROF_EXCHANGE, MPVAE_PROF_FUSED_SMALL_FWD,
       MPVAE_PROF_FUSED_SMALL_BWD, MPVAE_PROF_SLOTS };
int mpvae_profile(int32_t enable);
int mpvae_profile_read(int32_t slot, double *total_ms, int32_t *count);
const char *mpvae_profile_name(int32_t slot);

/* Test hook: out[i] = the library's normal-domain logarithm of in[i] (csrc/probit_math.cuh::log_normal, the libdevice logf
 * main path without its special-case blocks) and ref[i] = logf(in[i]), n device floats each; tests assert bit equality
 * over the whole domain the loss uses, [4.7e-7, 1]. */
int mpvae_test_log_normal(const float *in, float *out, float *ref, uint64_t n, void *cuda_stream);

const char *mpvae_last_error(void);
int mpvae_abi_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches claim) */
uint64_t mpvae_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MPVAE_B200_H_ */
