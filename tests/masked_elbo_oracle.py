"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The ELBO of partially labelled rows (compute_loss(..., label_mask=)) restated
with the pinned oracle's pieces: E from `clamped_probit`, the KL from `gaussian_kl`, the Bernoulli cell formula of
`bernoulli_log_mean_exp` and both ranking forms of `ranking_loss_pairwise` / `ranking_loss_factorised`, op for op,
with the mask applied by torch.where BEFORE any arithmetic touches a label:
    y_m = where(mask, y, 0)                      (whatever an unobserved cell holds, NaN included, never reaches a sum)
    lp_{s,b} = -sum_l where(mask, cell, 0)       (cell = -(log E * y_m + log(1 - E) * (1 - y_m)))
    is_pos = (y_m == 1) & mask,  is_neg = (y_m == 0) & mask,  n_pos / n_neg over observed cells only, and the ranking sums read
    where(mask, E, 0), so that an unobserved cell gets no ranking gradient (not the NaN of a degenerate row either)
KL, indiv_prob and indiv_prob_label are probit_elbo's.  With an all-ones mask every torch.where returns its first
argument unchanged, so the terms and the gradients are probit_elbo's bit for bit."""
from __future__ import annotations

import torch

from oracle.probit_elbo_oracle import ElboTerms, clamped_probit, gaussian_kl


def _zero(t):
    return torch.zeros((), dtype=t.dtype, device=t.device)


def masked_bernoulli_log_mean_exp(E, y, mask, accum=None):
    """bernoulli_log_mean_exp over the observed cells: unobserved cells add exactly 0 to a sample's log-likelihood."""
    cell = -(torch.log(E) * y + torch.log(1 - E) * (1 - y))
    if accum is not None:
        cell = cell.to(accum)
    cell = torch.where(mask, cell, _zero(cell))
    logprob = -torch.sum(cell, dim=2)                                                    # (S, B)
    peak = torch.max(logprob, dim=0)[0]
    mean_exp = torch.mean(torch.exp(logprob - peak), dim=0)
    return torch.mean(-torch.log(mean_exp) - peak)


def _pos_neg(E, y, mask):
    """(E, is_pos, is_neg) with E cut off from the graph in unobserved cells: no ranking gradient reaches them, not even
    the NaN of a row whose observed labels lack a positive or a negative (0/0 normaliser)."""
    E = torch.where(mask, E, _zero(E))
    y = y.float() if E.dtype == torch.float32 else y.to(E.dtype)
    is_pos = torch.logical_and(torch.eq(y, torch.ones_like(y)), mask)
    is_neg = torch.logical_and(torch.eq(y, torch.zeros_like(y)), mask)
    return E, is_pos, is_neg


def masked_ranking_loss_pairwise(E, y, mask, accum=None):
    """ranking_loss_pairwise with pos / neg restricted to observed cells."""
    E, is_pos, is_neg = _pos_neg(E, y, mask)
    truth = torch.logical_and(is_pos.unsqueeze(2), is_neg.unsqueeze(1)).to(E.dtype)   # (B, L, L)
    diff = E.unsqueeze(3) - E.unsqueeze(2)                                               # (S, B, L, L)
    masked = torch.exp(-5 * diff) * truth
    if accum is not None:
        masked = masked.to(accum)
    sums = torch.sum(masked, dim=[2, 3])                                                 # (S, B)
    n_pos = torch.sum(is_pos.to(sums.dtype), dim=1)
    n_neg = torch.sum(is_neg.to(sums.dtype), dim=1)
    per_row = torch.div(sums, 5 * (n_pos * n_neg))
    bad = torch.logical_or(torch.isinf(per_row), torch.isnan(per_row))
    per_row = torch.where(bad, torch.zeros_like(per_row), per_row)
    return torch.mean(per_row)


def masked_ranking_loss_factorised(E, y, mask, accum=None):
    """ranking_loss_factorised with pos / neg restricted to observed cells."""
    E, is_pos, is_neg = _pos_neg(E, y, mask)
    is_pos, is_neg = is_pos.to(E.dtype), is_neg.to(E.dtype)
    e_pos = torch.exp(-5 * E) * is_pos
    e_neg = torch.exp(5 * E) * is_neg
    if accum is not None:
        e_pos, e_neg = e_pos.to(accum), e_neg.to(accum)
    sums = torch.sum(e_pos, dim=2) * torch.sum(e_neg, dim=2)                             # (S, B)
    n_pos = torch.sum(is_pos.to(sums.dtype), dim=1)
    n_neg = torch.sum(is_neg.to(sums.dtype), dim=1)
    per_row = torch.div(sums, 5 * (n_pos * n_neg))
    bad = torch.logical_or(torch.isinf(per_row), torch.isnan(per_row))
    per_row = torch.where(bad, torch.zeros_like(per_row), per_row)
    return torch.mean(per_row)


def masked_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise, nll_coeff,
                       c_coeff, label_mask, *, ranking: str = "pairwise", dtype: torch.dtype = torch.float32,
                       accum=None) -> ElboTerms:
    """probit_elbo (oracle/probit_elbo_oracle.py) on the observed labels of `label_mask` (B, L) (nonzero = observed)."""
    dev = input_label.device
    mask = label_mask.to(dev).bool()
    y = input_label.to(dtype)
    y = torch.where(mask, y, _zero(y))                               # before any arithmetic on y
    fe_out, fx_out = fe_out.to(dtype), fx_out.to(dtype)
    kl = gaussian_kl(fe_mu.to(dtype), fe_logvar.to(dtype), fx_mu.to(dtype), fx_logvar.to(dtype), accum)

    eps1 = torch.tensor([1e-6]).float().to(dev).to(dtype)
    noise = noise.to(dev).to(dtype)
    basis = r_sqrt_sigma.T.float().to(dev).to(dtype) if dtype == torch.float32 \
        else r_sqrt_sigma.T.to(dev).to(dtype)
    sample_r = torch.tensordot(noise, basis, dims=1) + fe_out
    sample_r_x = torch.tensordot(noise, basis, dims=1) + fx_out
    E = clamped_probit(sample_r, eps1)
    E_x = clamped_probit(sample_r_x, eps1)

    rank = masked_ranking_loss_pairwise if ranking == "pairwise" else masked_ranking_loss_factorised
    nll = masked_bernoulli_log_mean_exp(E, y, mask, accum)
    c = rank(E, y, mask, accum)
    nll_x = masked_bernoulli_log_mean_exp(E_x, y, mask, accum)
    c_x = rank(E_x, y, mask, accum)

    if accum is not None:
        indiv_prob = torch.mean(E_x.to(accum), dim=0)
        indiv_prob_label = torch.mean(E.to(accum), dim=0)
    else:
        indiv_prob = torch.mean(E_x, dim=0)
        indiv_prob_label = torch.mean(E, dim=0)

    total = (nll + nll_x) * nll_coeff + (c + c_x) * c_coeff + kl * 1.1
    return ElboTerms(total, nll, nll_x, c, c_x, kl, indiv_prob, indiv_prob_label)


_NAMES = ["fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma"]


def masked_probit_elbo_with_grads(inputs: dict, noise, nll_coeff, c_coeff, label_mask, *, upstream=None, **kw):
    """probit_elbo_with_grads for masked_probit_elbo: (terms, {name: gradient}); default cotangent d total_loss = 1."""
    leaves = {k: inputs[k].detach().clone().requires_grad_(True) for k in _NAMES}
    terms = masked_probit_elbo(inputs["y"], *(leaves[k] for k in _NAMES), noise, nll_coeff, c_coeff, label_mask, **kw)
    if upstream is None:
        objective = terms.total_loss
    else:
        objective = sum((getattr(terms, k) * v.to(getattr(terms, k).dtype)).sum() for k, v in upstream.items())
    grads = torch.autograd.grad(objective, [leaves[k] for k in _NAMES], allow_unused=True)
    return terms, {k: g for k, g in zip(_NAMES, grads)}


def masked_loss_fn(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args, noise=None,
                   label_mask=None):
    """compute_loss-shaped wrapper (a `loss_fn` for train.DataParallelStep) on the CPU: needs an explicit noise tensor."""
    if label_mask is None:
        label_mask = torch.ones(input_label.shape, dtype=torch.bool, device=input_label.device)
    return masked_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise,
                              args.nll_coeff, args.c_coeff, label_mask, ranking="factorised")
