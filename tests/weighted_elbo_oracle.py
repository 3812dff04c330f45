"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The ELBO with a weight per row (compute_loss(..., row_weight=)), restated from the
masked oracle (tests/masked_elbo_oracle.py) with every loss term kept per row until the weighted mean:
    nll_b   = -log mean_s exp(lp_{s,b})                      (each branch; lp over the observed cells of the mask)
    c_{s,b} = the row's ranking term of sample s              (each branch; the mean over (S, B) is sum_b w_b c_b / B
                                                               with c_b = sum_s c_{s,b} / S)
    kl_b    = 0.5 * sum_d per_dim_{b,d}
    loss    = mean_b where(w_b != 0, w_b * t_b, 0)            (mean over all B rows: the divisor is B, not sum w)
A zero-weight row is taken out of the loss: its terms are selected away by torch.where (an inf / NaN term does not
reach the mean), and when some weight is 0 the loss-side inputs of those rows (E, E_x, the four encoder outputs) are
cut from the graph, so no NaN of a degenerate row reaches a gradient; indiv_prob and indiv_prob_label still read them.
With all-ones weights w_b * t_b is t_b bit for bit, the graph is the masked oracle's op for op, and so are the terms and
the gradients."""
from __future__ import annotations

import torch

from oracle.probit_elbo_oracle import ElboTerms, clamped_probit
from tests.masked_elbo_oracle import _pos_neg, _zero


def _weighted_mean(t, w, live):
    """mean over every entry of where(live, t * w, 0); w and live broadcast along t's last axis (the batch)"""
    w = w.to(t.dtype)
    return torch.mean(torch.where(live, t * w, _zero(t)))


def weighted_bernoulli_log_mean_exp(E, y, mask, w, live, accum=None):
    cell = -(torch.log(E) * y + torch.log(1 - E) * (1 - y))
    if accum is not None:
        cell = cell.to(accum)
    cell = torch.where(mask, cell, _zero(cell))
    logprob = -torch.sum(cell, dim=2)                                                    # (S, B)
    peak = torch.max(logprob, dim=0)[0]
    mean_exp = torch.mean(torch.exp(logprob - peak), dim=0)
    return _weighted_mean(-torch.log(mean_exp) - peak, w, live)                          # per row (B,)


def _ranking_per_row(sums, is_pos, is_neg):
    n_pos = torch.sum(is_pos.to(sums.dtype), dim=1)
    n_neg = torch.sum(is_neg.to(sums.dtype), dim=1)
    per_row = torch.div(sums, 5 * (n_pos * n_neg))
    bad = torch.logical_or(torch.isinf(per_row), torch.isnan(per_row))
    return torch.where(bad, torch.zeros_like(per_row), per_row)                          # (S, B)


def weighted_ranking_loss_pairwise(E, y, mask, w, live, accum=None):
    E, is_pos, is_neg = _pos_neg(E, y, mask)
    truth = torch.logical_and(is_pos.unsqueeze(2), is_neg.unsqueeze(1)).to(E.dtype)   # (B, L, L)
    diff = E.unsqueeze(3) - E.unsqueeze(2)                                               # (S, B, L, L)
    masked = torch.exp(-5 * diff) * truth
    if accum is not None:
        masked = masked.to(accum)
    sums = torch.sum(masked, dim=[2, 3])                                                 # (S, B)
    return _weighted_mean(_ranking_per_row(sums, is_pos, is_neg), w, live)


def weighted_ranking_loss_factorised(E, y, mask, w, live, accum=None):
    E, is_pos, is_neg = _pos_neg(E, y, mask)
    is_pos_f, is_neg_f = is_pos.to(E.dtype), is_neg.to(E.dtype)
    e_pos = torch.exp(-5 * E) * is_pos_f
    e_neg = torch.exp(5 * E) * is_neg_f
    if accum is not None:
        e_pos, e_neg = e_pos.to(accum), e_neg.to(accum)
    sums = torch.sum(e_pos, dim=2) * torch.sum(e_neg, dim=2)                             # (S, B)
    return _weighted_mean(_ranking_per_row(sums, is_pos_f, is_neg_f), w, live)


def weighted_gaussian_kl(fe_mu, fe_logvar, fx_mu, fx_logvar, w, live, accum=None):
    per_dim = (fx_logvar - fe_logvar) - 1 + torch.exp(fe_logvar - fx_logvar) \
        + torch.square(fx_mu - fe_mu) / (torch.exp(fx_logvar) + 1e-6)
    if accum is not None:
        per_dim = per_dim.to(accum)
    return _weighted_mean(0.5 * torch.sum(per_dim, dim=1), w, live)


def weighted_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise, nll_coeff,
                         c_coeff, row_weight, label_mask=None, *, ranking: str = "pairwise",
                         dtype: torch.dtype = torch.float32, accum=None) -> ElboTerms:
    """The masked oracle's ELBO with the (B,) row weights `row_weight` (label_mask None = every label observed)."""
    dev = input_label.device
    mask = torch.ones(input_label.shape, dtype=torch.bool, device=dev) if label_mask is None else label_mask.to(dev).bool()
    w = row_weight.to(dev).to(dtype)
    live = w != 0
    cut = not bool(live.all())

    def loss_side(t, rows):
        """t itself, or with the zero-weight rows (`rows`: the mask broadcast to t) cut from the graph"""
        return torch.where(rows, t, t.detach()) if cut else t

    y = input_label.to(dtype)
    y = torch.where(mask, y, _zero(y))                               # before any arithmetic on y
    fe_out, fx_out = fe_out.to(dtype), fx_out.to(dtype)
    kl_in = [loss_side(t.to(dtype), live[:, None]) for t in (fe_mu, fe_logvar, fx_mu, fx_logvar)]
    kl = weighted_gaussian_kl(*kl_in, w, live, accum)

    eps1 = torch.tensor([1e-6]).float().to(dev).to(dtype)
    noise = noise.to(dev).to(dtype)
    basis = r_sqrt_sigma.T.float().to(dev).to(dtype) if dtype == torch.float32 \
        else r_sqrt_sigma.T.to(dev).to(dtype)
    sample_r = torch.tensordot(noise, basis, dims=1) + fe_out
    sample_r_x = torch.tensordot(noise, basis, dims=1) + fx_out
    E = clamped_probit(sample_r, eps1)
    E_x = clamped_probit(sample_r_x, eps1)
    E_loss, E_x_loss = loss_side(E, live[None, :, None]), loss_side(E_x, live[None, :, None])

    rank = weighted_ranking_loss_pairwise if ranking == "pairwise" else weighted_ranking_loss_factorised
    nll = weighted_bernoulli_log_mean_exp(E_loss, y, mask, w, live, accum)
    c = rank(E_loss, y, mask, w, live, accum)
    nll_x = weighted_bernoulli_log_mean_exp(E_x_loss, y, mask, w, live, accum)
    c_x = rank(E_x_loss, y, mask, w, live, accum)

    if accum is not None:
        indiv_prob = torch.mean(E_x.to(accum), dim=0)
        indiv_prob_label = torch.mean(E.to(accum), dim=0)
    else:
        indiv_prob = torch.mean(E_x, dim=0)
        indiv_prob_label = torch.mean(E, dim=0)

    total = (nll + nll_x) * nll_coeff + (c + c_x) * c_coeff + kl * 1.1
    return ElboTerms(total, nll, nll_x, c, c_x, kl, indiv_prob, indiv_prob_label)


_NAMES = ["fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma"]


def weighted_probit_elbo_with_grads(inputs: dict, noise, nll_coeff, c_coeff, row_weight, label_mask=None, *, upstream=None,
                                    **kw):
    """(terms, {name: gradient}) of weighted_probit_elbo; default cotangent d total_loss = 1."""
    leaves = {k: inputs[k].detach().clone().requires_grad_(True) for k in _NAMES}
    terms = weighted_probit_elbo(inputs["y"], *(leaves[k] for k in _NAMES), noise, nll_coeff, c_coeff, row_weight,
                                 label_mask, **kw)
    if upstream is None:
        objective = terms.total_loss
    else:
        objective = sum((getattr(terms, k) * v.to(getattr(terms, k).dtype)).sum() for k, v in upstream.items())
    grads = torch.autograd.grad(objective, [leaves[k] for k in _NAMES], allow_unused=True)
    return terms, {k: g for k, g in zip(_NAMES, grads)}


def weighted_loss_fn(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args, noise=None,
                     label_mask=None, row_weight=None):
    """compute_loss-shaped wrapper (a `loss_fn` for train.DataParallelStep) on the CPU: needs an explicit noise tensor."""
    if row_weight is None:
        row_weight = torch.ones(input_label.shape[0], device=input_label.device)
    return weighted_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise,
                                args.nll_coeff, args.c_coeff, row_weight, label_mask, ranking="factorised")
