"""Drop-in for the reference's `mpvae.py`: `VAE` and `compute_loss` with the same signatures.

  * `VAE(args)` / `VAE.forward(label, feature)` (reference mpvae.py:10-100) stay plain torch.nn (cuBLAS):
    they are the boundary producer, not the hot path.  Attribute names, parameter shapes/dtypes and
    therefore state_dict keys are those of the reference, so checkpoints interchange (r_sqrt_sigma is a
    float64 (L, Z) Parameter; fd1/fd2 alias fd_x1/fd_x2).
  * `compute_loss(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args)`
    (reference mpvae.py:145-210) returns the same 8-tuple but runs the fused sm_100a kernels.

Noise (reference mpvae.py:162) -- `args.noise_mode` (optional attribute, default 'philox'):
  'philox'     counter-based normals generated on the GPU, keyed by (args.noise_seed or the module seed,
               a per-call offset, the global row index) -- independent of the data-parallel world size;
  'reference'  exactly the reference's draw: torch.normal(0,1,(S,B,Z)) on the CPU default generator,
               then copied to the device (bit-identical to the reference after torch.manual_seed);
  or pass the tensor itself as `compute_loss(..., noise=tensor)` (validation / external mode).
"""
from __future__ import annotations

import math
from collections import namedtuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .dense import linear
from .probit import ProbitELBO, label_pairs, philox_normal, predictive_rho, predictive_scale, probit_predict
from .probit import contract_nt, ghk_workspace_bytes, predict_exact_from_r, probit_predict_conditional
from .probit import _check_label_weight, _check_observed, _check_row_weight, probit_predict_conditional_ghk
from .probit import check_set_args, f1_sets, probit_sample_labels
from .probit import check_max_flips, check_set_bits, probit_predict_mode, probit_score_sets
from .probit import predict_pairs as probit_predict_pairs

_state = {"seed": 0x5EED_B200, "offset": 0}


def set_noise_seed(seed: int, offset: int = 0):
    """Seed of the Philox noise stream used when args carries no `noise_seed`."""
    _state["seed"], _state["offset"] = int(seed), int(offset)


def _xavier_r(label_dim, z_dim):
    bound = np.sqrt(6.0 / (label_dim + z_dim))
    return torch.from_numpy(np.random.uniform(-bound, bound, (label_dim, z_dim)))


class VAE(nn.Module):
    """Two encoders + a shared decoder trunk around the probit layer (reference mpvae.py:10-100)."""

    def __init__(self, args):
        super().__init__()
        F_, L, D = args.feature_dim, args.label_dim, args.latent_dim
        # registration order follows the reference so that seeded initialisation matches it
        for name, (n_in, n_out) in (("fx1", (F_, 256)), ("fx2", (256, 512)), ("fx3", (512, 256)),
                                    ("fx_mu", (256, D)), ("fx_logvar", (256, D)),
                                    ("fd_x1", (F_ + D, 256)), ("fd_x2", (256, 512)), ("feat_mp_mu", (512, L)),
                                    ("fe1", (F_ + L, 512)), ("fe2", (512, 256)),
                                    ("fe_mu", (256, D)), ("fe_logvar", (256, D))):
            setattr(self, name, nn.Linear(n_in, n_out))
        self.fd1, self.fd2 = self.fd_x1, self.fd_x2          # shared decoder trunk (mpvae.py:30-31)
        self.label_mp_mu = nn.Linear(512, L)
        self.dropout = nn.Dropout(p=args.keep_prob)           # the reference uses keep_prob as p (mpvae.py:38)
        self.scale_coeff = args.scale_coeff
        kind = getattr(args, "residue_sigma", "")
        if kind == "zero":
            r = nn.Parameter(torch.zeros((L, args.z_dim)), requires_grad=False)
        else:
            r = nn.Parameter(_xavier_r(L, args.z_dim), requires_grad=(kind != "random"))
        self.register_parameter("r_sqrt_sigma", r)

    # -- encoders (mpvae.py:51-64) --
    def _heads(self, h, mu, logvar):
        return mu(h) * self.scale_coeff, logvar(h) * self.scale_coeff

    def label_encode(self, x):
        h = x
        for layer in (self.fe1, self.fe2):
            h = self.dropout(F.relu(linear(layer, h)))
        return self._heads(h, self.fe_mu, self.fe_logvar)

    def feat_encode(self, x):
        h = x
        for layer in (self.fx1, self.fx2, self.fx3):
            h = self.dropout(F.relu(linear(layer, h)))
        return self._heads(h, self.fx_mu, self.fx_logvar)

    # -- reparameterisation (mpvae.py:66-74) --
    @staticmethod
    def _reparameterize(mu, logvar):
        std = torch.exp(0.5 * logvar)
        return mu + torch.randn_like(std) * std

    label_reparameterize = _reparameterize
    feat_reparameterize = _reparameterize

    # -- decoders (mpvae.py:76-84) --
    def _decode(self, z, head):
        return linear(head, F.relu(linear(self.fd_x2, F.relu(linear(self.fd_x1, z)))))

    def label_decode(self, z):
        return self._decode(z, self.label_mp_mu)

    def feat_decode(self, z):
        return self._decode(z, self.feat_mp_mu)

    def label_forward(self, x, feat):
        mu, logvar = self.label_encode(torch.cat((feat, x), 1))
        z = self._reparameterize(mu, logvar)
        return self.label_decode(torch.cat((feat, z), 1)), mu, logvar

    def feat_forward(self, x):
        mu, logvar = self.feat_encode(x)
        z = self._reparameterize(mu, logvar)
        return self.feat_decode(torch.cat((x, z), 1)), mu, logvar

    def forward(self, label, feature):
        label_out, label_mu, label_logvar = self.label_forward(label, feature)
        feat_out, feat_mu, feat_logvar = self.feat_forward(feature)
        return label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar


def noise_plan(args, n_sample, n_batch, device, noise=None):
    """How the (S, B, Z) standard-normal tensor of mpvae.py:162 is obtained: returns (tensor | None, spec | None).
    A spec (S, seed, offset, B_global, row0) means the library draws the Philox normals itself."""
    if noise is not None:
        return noise.to(device=device, dtype=torch.float32), None
    mode = getattr(args, "noise_mode", "philox")
    if mode == "reference":
        return torch.normal(0, 1, size=(n_sample, n_batch, args.z_dim)).to(device), None
    if mode != "philox":
        raise ValueError(f"args.noise_mode={mode!r}: expected 'philox' or 'reference'")
    seed = getattr(args, "noise_seed", None)
    if seed is None:
        seed = _state["seed"]
    offset = getattr(args, "noise_offset", None)
    if offset is None:
        offset = _state["offset"]
        _state["offset"] += 1
    return None, (n_sample, seed, offset, getattr(args, "dp_global_batch", None), getattr(args, "dp_row0", 0),
                  getattr(args, "noise_offset_tensor", None))


def draw_noise(args, n_sample, n_batch, device, noise=None):
    """The noise tensor itself (materialised; the loss path normally never needs it in Philox mode)."""
    tensor, spec = noise_plan(args, n_sample, n_batch, device, noise)
    if tensor is not None:
        return tensor
    _, seed, offset, b_global, row0, counter = spec
    if counter is not None:
        offset = int(offset) + int(counter.item())
    return philox_normal(n_sample, n_batch, args.z_dim, seed=seed, offset=offset, device=device,
                         global_batch=b_global, row0=row0)


def compute_loss(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args, noise=None,
                 label_mask=None, row_weight=None, pos_weight=None, neg_weight=None, reduction="mean"):
    """Reference signature (mpvae.py:145) -> (total_loss, nll_loss, nll_loss_x, c_loss, c_loss_x, kl_loss,
    indiv_prob, indiv_prob_label) (mpvae.py:210).

    `label_mask` (B, L) bool or uint8 on the batch's device, or None (every label known): partially labelled rows.
    Nonzero = the label is observed.  Per row, with O the observed labels:
      - both log-likelihoods sum over O only; the log-mean-exp over samples and the mean over all B rows are unchanged,
        so a row with nothing observed adds exactly 0 to nll_loss / nll_loss_x;
      - the ranking losses take pos = observed and y == 1, neg = observed and y == 0, and count only observed cells;
        a row whose observed labels lack a positive or a negative adds 0 (its observed cells get NaN gradients, as an
        unmasked degenerate row does, unless MPVAE_FLAG_SANITIZE_DEGENERATE; unobserved cells never do);
      - kl_loss, indiv_prob and indiv_prob_label (every cell) are unchanged;
      - an unobserved cell's logit gradient is only the cotangent of indiv_prob / indiv_prob_label.
    Whatever input_label holds in an unobserved cell, NaN included, has no effect here.  (The label encoder still reads
    input_label as the caller gives it: filling unknown labels with 0 there is the caller's choice.)  A mask of all ones
    gives the unmasked results bit for bit.  With one row in test mode, -predict_conditional(...,
    observed=torch.where(mask, y.to(torch.int8), -1)).log_evidence equals nll_loss_x on the same noise.

    `row_weight` (B,) floating tensor on the batch's device, or None (every row weighs 1): weighted rows, e.g. importance
    weights, down-weighted noisy rows, or one weighted row for several duplicates.  It can be combined with label_mask.
    With t_b the row's terms -- its negative log-mean-exp over samples of each branch, its ranking sum over samples / S
    in each branch, its KL term -- the five loss scalars become sum_b w_b t_b / B, and total_loss is formed from them as
    before:
      - the divisor is B, not sum(w): a weight of 1 on every row gives the bits of row_weight=None on all 8 outputs and
        every gradient, and data-parallel shards combine as before (for sum(w) normalisation pass w * B / w.sum());
      - indiv_prob and indiv_prob_label do not depend on the weights;
      - a row with weight 0 is removed from the loss: its terms (inf / NaN included) are skipped, and its loss gradients
        are exactly 0 -- a degenerate row gets no NaN, even without MPVAE_FLAG_SANITIZE_DEGENERATE; with finite inputs
        its logit gradient is the cotangent of the predictions alone;
      - other values are used as given (negatives included; NaN propagates); they are not checked on the host.
    The weights are converted to contiguous fp32 and receive no gradient: a weight that requires grad is refused, as are
    a wrong shape, device or a non-floating dtype, before any noise offset is consumed.

    `pos_weight`, `neg_weight` (L,) floating tensors on the batch's device, or None (all ones): label weights inside each
    row's log-likelihood, e.g. pos_weight = n_neg / n_pos (clamped) so that rare labels are predicted, or propensity or
    inverse-frequency weights.  Per cell of both branches the log-likelihood becomes pos_weight[l] * log E (y = 1),
    neg_weight[l] * log(1 - E) (y = 0), or pos_weight[l] * y * log E + neg_weight[l] * (1 - y) * log(1 - E) for a soft
    label, before the log-mean-exp over samples: t_b = -log mean_s exp(sum over the observed l of the weighted ll).  So
    the weights also shift which samples dominate a row.  They can be combined with label_mask and row_weight (the row
    weight multiplies the row term formed from the label-weighted likelihood):
      - weights of 1 give the bits of pos_weight=neg_weight=None on all 8 outputs and every gradient;
      - the ranking losses (c_loss, c_loss_x, normalised per row by n_pos * n_neg already), kl_loss, indiv_prob and
        indiv_prob_label do not depend on them;
      - a zero weight drops the cell's term (it is not multiplied by 0) and its log-likelihood gradient is exactly 0;
      - other values are used as given (negatives included); they are not checked on the host.
    The weights receive no gradient: a weight that requires grad is refused, as are a wrong shape, device or a
    non-floating dtype, before any noise offset is consumed.

    `reduction` 'mean' (the default: the batch means above) or 'none': per-row losses, e.g. to select or reweight rows
    by their own loss (small-loss selection, group DRO, CVaR) or to score rows one by one.  The same 8-tuple comes back,
    with total_loss, nll_loss, nll_loss_x, c_loss, c_loss_x and kl_loss as (B,) fp32 tensors of every row's values:
      - with t_b the row's fp64 terms (above; label_mask and the label weights act inside them), the five terms are
        w_b t_b (w_b = 1 without row_weight), rounded once to fp32, and total_loss[b] is formed from them with the
        operations of the batch total; so the mean over the rows of each output is the 'mean' output up to summation
        order, and with B = 1 the two reductions give the same bits on all 8 outputs and every gradient;
      - a zero-weight row returns exactly 0 on all six outputs, inf / NaN terms included;
      - indiv_prob and indiv_prob_label are unchanged;
      - backward: each of the six takes a (B,) cotangent; row b's gradients are those of the 'mean' call with row b's
        cotangents and the divisor 1 in place of B, so `total.sum() / B` gives the 'mean' gradients up to rounding;
      - a row whose six cotangents are all 0 gets no loss gradient at all, as a zero-weight row: selecting rows by
        indexing (`total[keep].sum()`) leaves an unselected degenerate row without NaN, even without
        MPVAE_FLAG_SANITIZE_DEGENERATE; a selected degenerate row gets NaN gradients as with 'mean'.
    Any other value is refused before any noise offset is consumed."""
    device = input_label.device
    if reduction not in ("mean", "none"):
        raise ValueError(f"reduction must be 'mean' or 'none', got {reduction!r}")
    if row_weight is not None:
        row_weight = _check_row_weight(row_weight, fe_out.shape[0], device)
    label_weight = _check_label_weight(pos_weight, neg_weight, fe_out.shape[1], device)
    if device.type != "cuda":
        raise RuntimeError("mpvae_b200.compute_loss needs CUDA tensors: the probit ELBO is implemented as sm_100a "
                           "kernels only (no CPU fallback)")
    n_sample = args.n_train_sample if args.mode == "train" else args.n_test_sample   # mpvae.py:158
    n_batch = fe_out.shape[0]
    if n_batch == 0:
        # train.py:102 runs int(N/bs)+1 steps, so an empty last batch reaches the loss: every mean is NaN
        nan = (fe_out.sum() + fx_out.sum() + fe_mu.sum() + fe_logvar.sum() + fx_mu.sum() + fx_logvar.sum()) * math.nan
        empty = fx_out.new_empty((0, fx_out.shape[1]))
        if reduction == "none":     # no rows, no per-row values
            z = (fe_out.sum() + fx_out.sum() + fe_mu.sum() + fe_logvar.sum() + fx_mu.sum() + fx_logvar.sum()).reshape(1)[:0]
            return (z, z.clone(), z.clone(), z.clone(), z.clone(), z.clone(), empty, empty.clone())
        return (nan, nan.clone(), nan.clone(), nan.clone(), nan.clone(), nan.clone(), empty, empty.clone())
    r32 = r_sqrt_sigma.to(device).float()                # mpvae.py:165 -- outside the Function: grad returns as fp64
    noise, spec = noise_plan(args, n_sample, n_batch, device, noise)
    flags = int(getattr(args, "mpvae_flags", 0))
    # args.peer_ring (peer.PeerRing, data-parallel runs): g_R comes back already summed over the ranks
    return ProbitELBO.apply(input_label.float(), fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise,
                            float(args.nll_coeff), float(args.c_coeff), flags, spec, getattr(args, "peer_ring", None),
                            label_mask, row_weight, label_weight, reduction == "none")


def predict(fx_out, r_sqrt_sigma, args, noise=None):
    """The prediction `indiv_prob` (B, L) of compute_loss in test mode (mpvae.py:170,180,203) from the feature branch
    alone (`VAE.feat_forward(feature)[0]`): no labels, no label branch, no loss.  Same S (args.n_test_sample), same
    noise (`noise_plan`: a call without args.noise_offset consumes one offset, as compute_loss does), same flags, and
    bit for bit the indiv_prob compute_loss returns for the same fx_out.  Inference only: it builds no autograd graph."""
    n_sample, r32, noise, spec, flags = _sample_plan("predict", fx_out, r_sqrt_sigma, args, noise)
    return probit_predict(fx_out, r32, n_sample, noise=noise, noise_spec=spec, flags=flags)


_UNCONDITIONAL = object()     # _sample_plan's `observed` for predict, which conditions on none


def _sample_plan(name, fx_out, r_sqrt_sigma, args, noise, observed=_UNCONDITIONAL):
    """The start of every sampled predictor: the refusals, in this order, then (n_sample, r32, noise, noise_spec, flags)
    as compute_loss plans them in test mode.  An empty batch gets an (S, 0, Z) noise tensor and consumes no noise
    offset; the probit wrappers return its empty outputs without calling the library."""
    _inference_only(name, fx_out, r_sqrt_sigma)
    device = fx_out.device
    if device.type != "cuda":
        raise RuntimeError(f"mpvae_b200.{name} needs CUDA tensors: the probit prediction is implemented as sm_100a "
                           "kernels only (no CPU fallback)")
    if observed is not _UNCONDITIONAL:
        _check_observed(observed, fx_out.shape, device)
    n_sample = args.n_test_sample
    r32 = r_sqrt_sigma.to(device).float()
    if fx_out.shape[0] == 0:
        noise, spec = torch.empty((n_sample, 0, r32.shape[1]), dtype=torch.float32, device=device), None
    else:
        noise, spec = noise_plan(args, n_sample, fx_out.shape[0], device, noise)
    return n_sample, r32, noise, spec, int(getattr(args, "mpvae_flags", 0))


ConditionalPrediction = namedtuple("ConditionalPrediction", ["prob", "log_evidence", "ess"])


def predict_conditional(fx_out, r_sqrt_sigma, observed, args, noise=None):
    """P(y_l = 1 | the row's observed labels, x) for the labels a row does not have, given the ones it has.

    The probit model's residual label correlation I + R R^T makes the labels of a row dependent; this conditions on
    the known ones.  Each of `predict`'s S samples (args.n_test_sample, the same noise: `noise_plan`, so a call without
    args.noise_offset consumes one offset, and with the same offset it uses predict's noise) is weighted by the
    likelihood of the observed labels, u_s = prod_o E_o^y_o (1 - E_o)^(1 - y_o), and the unobserved cells take the
    weighted mean of E instead of the plain mean.  Returns ConditionalPrediction(prob, log_evidence, ess):
      prob          (B, L) fp32: the conditional probability of each unobserved label; observed cells hold their value
      log_evidence  (B,): the Monte Carlo estimate of log P(observed labels | x); 0 with nothing observed, and with
                    everything observed the row's nll_loss_x of compute_loss, negated
      ess           (B,): the effective sample size of the weights, in [1, S].  It drops towards 1 as more labels are
                    observed; a small ess means few samples carry the estimate.
    With nothing observed, prob is predict's indiv_prob bit for bit.

    `observed` is an int8 (B, L) tensor on fx_out's device: 0 or 1 = observed with that value, any other value (use -1)
    = unobserved.  From labels y and a boolean mask of the known ones:
        observed = torch.where(mask, y.to(torch.int8), -1)
    Its values are not checked (no host synchronisation).  Inference only, CUDA only; args.mpvae_flags as for predict."""
    n_sample, r32, noise, spec, flags = _sample_plan("predict_conditional", fx_out, r_sqrt_sigma, args, noise, observed)
    return ConditionalPrediction(*probit_predict_conditional(fx_out, r32, observed, n_sample, noise=noise, noise_spec=spec,
                                                             flags=flags))


# The GHK sampler's scratch (its per-row Cholesky factors and per-sample vectors grow as B * max|O|^2 and B * S * max|O|)
# is kept under this many bytes by splitting the batch into row groups.
GHK_WORKSPACE_BOUND = 8 << 30


def label_gram(r_sqrt_sigma, args=None):
    """G = R R^T (L, L) fp32, the label covariance of the probit noise, for predict_conditional_ghk(..., gram=G): the
    product the library runs when no gram is passed (the CUDA-core product under MPVAE_FLAG_CONTRACT_FMA in
    args.mpvae_flags, else the engine G's own shape selects), so a prepared G gives the same bits.  Prepare it once per R
    for repeated calls, as PairPredictor prepares rho.  Inference only."""
    _inference_only("label_gram", r_sqrt_sigma)
    _cuda_only("label_gram", r_sqrt_sigma)
    flags = int(getattr(args, "mpvae_flags", 0)) if args is not None else 0
    r32 = r_sqrt_sigma.float()
    return contract_nt(r32, r32, engine=1 if flags & FLAG_CONTRACT_FMA else 0)


def predict_conditional_ghk(fx_out, r_sqrt_sigma, observed, args, noise=None, gram=None):
    """predict_conditional's ConditionalPrediction(prob, log_evidence, ess) from a GHK sampler of the probit posterior,
    whose effective sample size stays usable when many labels are observed (where the importance weights of
    predict_conditional collapse onto one sample).

    In the model's latent form u = fx + R eps + w, each of predict's S samples (same noise, same offset consumption)
    draws the observed latents label by label, each from its clamped truncated conditional given the ones before, and
    takes the product of the observed labels' conditional probabilities as its weight; the sample's R eps is then
    conditioned on those latents (Matheron's rule) before E is averaged.  prob, log_evidence and ess mean what they mean
    for predict_conditional; with nothing observed in a row, its prob is predict's bits, log_evidence 0 and ess S.  The
    two are different estimators of the same quantities: this one costs a Cholesky factor of I + G[O, O] per row and a
    (S x |O|) . (|O| x L) product per row, and is the one to use when rows carry more than a handful of labels.

    `observed`: int8 (B, L) as for predict_conditional.  `gram`: label_gram(r_sqrt_sigma, args), or None to compute it
    here.  The call reads max_b |O_b| on the host (one synchronisation) to size its scratch, and runs the batch in row
    groups that keep that scratch under GHK_WORKSPACE_BOUND bytes; rows are keyed by their global row, so the split
    changes no bits.  The sampler's own uniforms and normals come from a Philox stream separate from the noise.
    Inference only, CUDA only; args.mpvae_flags as for predict."""
    n_sample, r32, noise, spec, flags = _sample_plan("predict_conditional_ghk", fx_out, r_sqrt_sigma, args, noise,
                                                     observed)
    n_batch, L = fx_out.shape
    Z = r32.shape[1]
    # the one host synchronisation (none for an empty batch, which runs as one empty group)
    max_obs = int(((observed == 0) | (observed == 1)).sum(1).max().item()) if n_batch else 0
    one = ghk_workspace_bytes(n_sample, 1, L, Z, max_obs, flags)
    per_row = max(ghk_workspace_bytes(n_sample, 2, L, Z, max_obs, flags) - one, 1)
    rows = max(1, (GHK_WORKSPACE_BOUND - (one - per_row)) // per_row)
    n_groups = max(-(-n_batch // rows), 1)
    rows = max(-(-n_batch // n_groups), 1)
    if gram is None and n_groups > 1 and max_obs > 0:
        gram = label_gram(r32, args)
    if spec is not None:
        b_global = spec[3] if spec[3] is not None else n_batch
    out = []
    for a in range(0, max(n_batch, 1), rows):
        b = min(n_batch, a + rows)
        if spec is not None:
            group_noise, group_spec = None, (spec[0], spec[1], spec[2], b_global, spec[4] + a) + tuple(spec[5:])
        else:
            group_noise, group_spec = noise[:, a:b], (n_sample, 0, 0, n_batch, a)
        out.append(probit_predict_conditional_ghk(fx_out[a:b], r32, observed[a:b], n_sample, max_obs, noise=group_noise,
                                                  noise_spec=group_spec, flags=flags, gram=gram))
    if len(out) == 1:
        return ConditionalPrediction(*out[0])
    return ConditionalPrediction(*(torch.cat(t, 0) for t in zip(*out)))


def sample_labels(fx_out, r_sqrt_sigma, args, noise=None, uniform=None):
    """Joint label samples of the probit predictive distribution: (B, S, ceil(L / 32)) int32 bits, S =
    args.n_test_sample, label l of sample s of row b at bit l % 32 of word [b, s, l // 32] (unpack_label_samples gives
    the (B, S, L) bool tensor).  Sample s is the whole label vector y = (U < E_s), E_s the clamped probit of predict's
    sample s: same noise (`noise_plan`: a call without args.noise_offset consumes one offset, and with the same offset it
    uses predict's noise), so the mean of the samples over s estimates predict's indiv_prob without bias, and the
    samples keep the joint structure of I + R R^T that the marginals lose.  `uniform`: optional (S, B, L) fp32 draws in
    (0, 1); None = the library's own Philox stream, keyed by global row (args.dp_row0), so a row's samples do not depend
    on batching.  Inference only, CUDA only; args.mpvae_flags as for predict."""
    n_sample, r32, noise, spec, flags = _sample_plan("sample_labels", fx_out, r_sqrt_sigma, args, noise)
    return probit_sample_labels(fx_out, r32, n_sample, noise=noise, noise_spec=spec, flags=flags, uniform=uniform)


def unpack_label_samples(bits, label_dim):
    """(B, S, L) bool from sample_labels' (B, S, ceil(L / 32)) int32 bits, on the tensor's device."""
    shifts = torch.arange(32, dtype=torch.int32, device=bits.device)
    y = torch.bitwise_and(torch.bitwise_right_shift(bits.unsqueeze(-1), shifts), 1)
    return y.reshape(bits.shape[0], bits.shape[1], -1)[:, :, :label_dim].bool()


SetPrediction = namedtuple("SetPrediction", ["sets", "expected_f", "size"])


def f1_optimal_sets(bits, label_dim, beta=1.0, max_size=None):
    """The F_beta-optimal label set of each row for the empirical distribution of its label samples (sample_labels'
    bits, or any bits in that layout), by the GFM algorithm (Dembczynski et al., NIPS 2011).  Per row, with s_i the size
    of sample i, Delta_{l,k} = mean_i y_{i,l} (1 + beta^2) / (beta^2 s_i + k): the best set of size k is the top k labels
    of Delta_{., k}, its expected F is their sum, and the empty set scores the share of empty samples.  The result is
    the exact optimum over every set of at most `max_size` labels (None: no bound); ties go to the smaller set and the
    lower label index.  Returns SetPrediction(sets (B, L) bool, expected_f (B,) float64, size (B,) int32).  The cost
    per row grows as min(|U|, max_size) * |U| * S, |U| the number of labels set in any sample: bound max_size when rows
    are dense.  CUDA only; no host synchronisation."""
    if isinstance(bits, torch.Tensor) and not bits.is_cuda:
        raise RuntimeError("mpvae_b200.f1_optimal_sets needs CUDA tensors: the F-measure decoder is implemented as sm_100a "
                           "kernels only (no CPU fallback)")
    return SetPrediction(*f1_sets(bits, label_dim, beta, max_size))


def predict_sets(fx_out, r_sqrt_sigma, args, beta=1.0, max_size=None, noise=None):
    """Per row, the label set with the largest expected F_beta under the model: sample_labels' S joint draws, then
    f1_optimal_sets on them.  Thresholding predict's marginals is the best decision for the Hamming loss, not for the
    example-based F1; this uses the joint distribution of the row's labels.  Returns SetPrediction(sets (B, L) bool,
    expected_f (B,) float64: the expected F_beta of the set on the samples, size (B,) int32).  Same noise and offset
    consumption as predict.  Inference only, CUDA only."""
    check_set_args(beta, max_size)          # before the plan: a refused call consumes no noise offset
    n_sample, r32, noise, spec, flags = _sample_plan("predict_sets", fx_out, r_sqrt_sigma, args, noise)
    bits = probit_sample_labels(fx_out, r32, n_sample, noise=noise, noise_spec=spec, flags=flags)
    return SetPrediction(*f1_sets(bits, fx_out.shape[1], beta, max_size))


SetScores = namedtuple("SetScores", ["log_prob", "ess"])


def score_sets(fx_out, r_sqrt_sigma, bits, args, noise=None):
    """The model's log-probability of given label sets: C sets per row in `bits`, an int32 (B, C, ceil(L / 32)) tensor
    in sample_labels' layout (label l of set c of row b at bit l % 32 of word [b, c, l // 32]; bits at and above L are
    ignored).  On predict's S samples (same noise, same offset consumption: a call without args.noise_offset consumes
    one offset, and with the same offset it uses predict's noise), sample s gives every label its own Bernoulli(E_s),
    and the set's probability is the mean over s of the product, in logs:
        lp_s = sum_l log(y_l ? E_sl : 1 - E_sl)      (the loss's fp32 cell logs, summed in fp64)
        log_prob = log mean_s exp(lp_s),   ess = (sum_s w_s)^2 / sum_s w_s^2,  w_s = exp(lp_s - max lp)
    exp(log_prob) is the model's expected exact-match accuracy of the set; ess says how many samples carry the estimate
    (it falls towards 1 when L is large).  With the row's true labels, log_prob is the row's -nll_loss_x of
    compute_loss up to that path's fp32 rounding.  Returns SetScores(log_prob (B, C) float64, ess (B, C) float64).
    Inference only, CUDA only; args.mpvae_flags as for predict."""
    n_batch, label_dim = fx_out.shape
    check_set_bits(bits, n_batch, label_dim, fx_out.device)
    n_sample, r32, noise, spec, flags = _sample_plan("score_sets", fx_out, r_sqrt_sigma, args, noise)
    return SetScores(*probit_score_sets(fx_out, r32, bits, n_sample, noise=noise, noise_spec=spec, flags=flags))


ModePrediction = namedtuple("ModePrediction", ["sets", "log_prob", "ess", "size", "flips"])


def predict_mode(fx_out, r_sqrt_sigma, args, max_flips=None, noise=None):
    """Per row, the label set the model finds most probable: the decision that maximises the expected exact-match
    (subset) accuracy, where thresholding predict's marginals maximises the Hamming accuracy and predict_sets the F1.
    The search is deterministic: the best of the candidates 1[predict >= 0.5], the empty set and each sample's own mode
    (ties to the earliest), then steepest single-label flips while one raises score_sets' log_prob, at most `max_flips`
    of them (None: no bound; one flip costs S * L per row).  With flips < max_flips the set is a local maximum: no
    single flip scores higher.  Returns ModePrediction(sets (B, L) bool, log_prob (B,) float64, ess (B,) float64 --
    score_sets of the set, bit for bit --, size (B,) int32, flips (B,) int32).  Same noise and offset consumption as
    predict.  Inference only, CUDA only; args.mpvae_flags as for predict."""
    check_max_flips(max_flips)              # before the plan: a refused call consumes no noise offset
    n_sample, r32, noise, spec, flags = _sample_plan("predict_mode", fx_out, r_sqrt_sigma, args, noise)
    return ModePrediction(*probit_predict_mode(fx_out, r32, n_sample, max_flips, noise=noise, noise_spec=spec,
                                               flags=flags))


def _inference_only(name, *tensors):
    if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
        raise RuntimeError(f"mpvae_b200.{name} is inference only and returns no gradient: call it under torch.no_grad() "
                           "(or detach its inputs); compute_loss is the differentiable path")


def _cuda_only(name, t):
    if t.device.type != "cuda":
        raise RuntimeError(f"mpvae_b200.{name} needs CUDA tensors: the closed-form prediction is implemented as sm_100a "
                           "kernels only (no CPU fallback)")


def predict_exact(fx_out, r_sqrt_sigma, args):
    """The exact limit as S -> infinity of `predict`'s indiv_prob (B, L): with n = R eps the noise of mpvae.py:162-170,
        indiv_prob[b, l] = c + k Phi(fx_out[b, l] / sqrt(1 + |R_l|^2))      (E = c + k Phi: the clamp of mpvae.py:177)
    without samples, noise or product, so it consumes no noise offset and does not depend on args.n_test_sample.  Each
    call computes the per-label scale from R first (one read of R, fp64 sums) and then one elementwise pass over fx_out.
    args.mpvae_flags may carry MPVAE_FLAG_STABLE_CDF; other flags do not apply.  Same arguments as `predict`, so it
    serves as `infer.predict_proba(..., predict_fn=predict_exact)`.
    fx_out itself is still random: `VAE.feat_forward` samples the latent through `_reparameterize` (randn_like).  Like
    predict's Monte Carlo, the closed form integrates out the probit noise only.  Inference only."""
    _inference_only("predict_exact", fx_out, r_sqrt_sigma)
    _cuda_only("predict_exact", fx_out)
    if fx_out.shape[0] == 0:
        return fx_out.new_empty((0, fx_out.shape[1]))
    r32 = r_sqrt_sigma.to(fx_out.device).float()
    return predict_exact_from_r(fx_out, r32, int(getattr(args, "mpvae_flags", 0)))


def all_pairs(label_dim):
    """The (L (L - 1) / 2, 2) int64 label pairs (i, j), i < j, in row-major upper-triangle order."""
    return torch.triu_indices(label_dim, label_dim, 1).T.contiguous()


class PairPredictor:
    """P(y_i = 1, y_j = 1 | x) for a fixed list of label pairs: the pairwise co-occurrence of the probit predictive
    distribution in closed form,
        c^2 + c k (Phi(h_i) + Phi(h_j)) + k^2 Phi2(h_i, h_j; rho_ij),   h = fx_out / sqrt(1 + |R_l|^2),
        rho_ij = R_i . R_j / sqrt((1 + |R_i|^2)(1 + |R_j|^2))
    (Phi2: the bivariate normal CDF).  The scale and rho (P * Z fp64 FMAs) are prepared once here, from R as it is now;
    a call with fx_out (B, L) returns (B, P) in one launch.  A pair (i, i) returns predict_exact's P(y_i = 1) bit for bit.
    As for predict_exact, only the probit noise is integrated out; fx_out stays random through feat_forward.
    Inference only; build a new one after R changes."""

    def __init__(self, r_sqrt_sigma, pairs, args):
        _inference_only("PairPredictor", r_sqrt_sigma)
        r32 = r_sqrt_sigma.float()
        self.label_dim = r32.shape[0]
        self.pairs = label_pairs(pairs, self.label_dim, r32.device)
        _cuda_only("PairPredictor", r32)
        self.flags = int(getattr(args, "mpvae_flags", 0))
        self.scale = predictive_scale(r32)
        self.rho = predictive_rho(r32, self.scale, self.pairs)

    def __call__(self, fx_out):
        _inference_only("PairPredictor", fx_out)
        _cuda_only("PairPredictor", fx_out)
        return probit_predict_pairs(fx_out, self.scale, self.pairs, self.rho, self.flags)


probit_elbo = compute_loss
FLAG_SANITIZE_DEGENERATE = _lib.FLAG_SANITIZE_DEGENERATE
FLAG_STABLE_CDF = _lib.FLAG_STABLE_CDF
FLAG_CONTRACT_TENSOR = _lib.FLAG_CONTRACT_TENSOR
FLAG_CONTRACT_FMA = _lib.FLAG_CONTRACT_FMA
FLAG_FUSED_FORWARD = _lib.FLAG_FUSED_FORWARD
FLAG_SEPARATE_NOISE = _lib.FLAG_SEPARATE_NOISE
FLAG_FUSED_EXCHANGE = _lib.FLAG_FUSED_EXCHANGE
FLAG_SERIAL_EXCHANGE = _lib.FLAG_SERIAL_EXCHANGE
