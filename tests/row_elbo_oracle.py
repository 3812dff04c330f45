"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Per-row losses (compute_loss(..., reduction='none')), restated from the label-weighted
oracle (tests/label_weighted_elbo_oracle.py) with every term kept per row instead of averaged over the batch:
    nll_b = -log mean_s exp(sum over the observed l of ll_{s,b,l})     (each branch; ll label-weighted)
    c_b   = sum_s c_{s,b} / S                                          (each branch; c_{s,b} the row's ranking term)
    kl_b  = 0.5 * sum_d per_dim_{b,d}
    out_b = where(w_b != 0, w_b * t_b, 0)                              (each of the five; w the row weights)
    total_b = (nll_b + nll_x_b) * nll_coeff + (c_b + c_x_b) * c_coeff + kl_b * 1.1
so mean_b out_b is the label-weighted oracle's batch output.  Rows outside `grad_rows` (the rows whose cotangent is not
all zero, and whose weight is not 0) have their loss-side inputs cut from the graph, so a degenerate row left out of the
objective puts no NaN in any gradient; indiv_prob and indiv_prob_label still read them."""
from __future__ import annotations

import torch

from oracle.probit_elbo_oracle import ElboTerms, clamped_probit
from tests.masked_elbo_oracle import _pos_neg, _zero
from tests.weighted_elbo_oracle import _NAMES, _ranking_per_row

ROW_TERMS = ("total_loss", "nll_loss", "nll_loss_x", "c_loss", "c_loss_x", "kl_loss")


def _row_nll(E, y, mask, lw, accum):
    w0, w1 = lw[0].to(E.dtype), lw[1].to(E.dtype)
    pos = torch.log(E) * y * w1
    neg = torch.log(1 - E) * (1 - y) * w0
    cell = -(torch.where(w1 != 0, pos, _zero(pos)) + torch.where(w0 != 0, neg, _zero(neg)))
    if accum is not None:
        cell = cell.to(accum)
    cell = torch.where(mask, cell, _zero(cell))
    logprob = -torch.sum(cell, dim=2)                                                    # (S, B)
    peak = torch.max(logprob, dim=0)[0]
    mean_exp = torch.mean(torch.exp(logprob - peak), dim=0)
    return -torch.log(mean_exp) - peak                                                   # (B,)


def _row_ranking(E, y, mask, ranking, accum):
    E, is_pos, is_neg = _pos_neg(E, y, mask)
    if ranking == "pairwise":
        truth = torch.logical_and(is_pos.unsqueeze(2), is_neg.unsqueeze(1)).to(E.dtype)   # (B, L, L)
        masked = torch.exp(-5 * (E.unsqueeze(3) - E.unsqueeze(2))) * truth
        if accum is not None:
            masked = masked.to(accum)
        sums = torch.sum(masked, dim=[2, 3])                                             # (S, B)
    else:
        is_pos, is_neg = is_pos.to(E.dtype), is_neg.to(E.dtype)
        e_pos, e_neg = torch.exp(-5 * E) * is_pos, torch.exp(5 * E) * is_neg
        if accum is not None:
            e_pos, e_neg = e_pos.to(accum), e_neg.to(accum)
        sums = torch.sum(e_pos, dim=2) * torch.sum(e_neg, dim=2)
    per = _ranking_per_row(sums, is_pos, is_neg)                                         # (S, B)
    return torch.sum(per, dim=0) / per.shape[0]                                          # (B,)


def row_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise, nll_coeff,
                    c_coeff, row_weight=None, label_mask=None, label_weight=None, grad_rows=None, *,
                    ranking: str = "pairwise", dtype: torch.dtype = torch.float32, accum=None) -> ElboTerms:
    """The per-row ELBO terms: six (B,) tensors, then indiv_prob and indiv_prob_label.  label_weight (2, L) [w0; w1] or
    None (ones); grad_rows (B,) bool or None (every row): the rows whose loss terms carry gradients."""
    dev = input_label.device
    B, L = input_label.shape
    mask = torch.ones((B, L), dtype=torch.bool, device=dev) if label_mask is None else label_mask.to(dev).bool()
    w = (torch.ones(B) if row_weight is None else row_weight).to(dev).to(dtype)
    lw = (torch.ones(2, L) if label_weight is None else label_weight).to(dev).to(dtype)
    live = w != 0
    keep = live if grad_rows is None else live & grad_rows.to(dev)
    cut = not bool(keep.all())

    def loss_side(t, rows):
        return torch.where(rows, t, t.detach()) if cut else t

    y = input_label.to(dtype)
    y = torch.where(mask, y, _zero(y))
    fe_out, fx_out = fe_out.to(dtype), fx_out.to(dtype)
    fe_mu, fe_logvar, fx_mu, fx_logvar = (loss_side(t.to(dtype), keep[:, None]) for t in (fe_mu, fe_logvar, fx_mu, fx_logvar))
    per_dim = (fx_logvar - fe_logvar) - 1 + torch.exp(fe_logvar - fx_logvar) \
        + torch.square(fx_mu - fe_mu) / (torch.exp(fx_logvar) + 1e-6)
    if accum is not None:
        per_dim = per_dim.to(accum)
    kl = 0.5 * torch.sum(per_dim, dim=1)

    eps1 = torch.tensor([1e-6]).float().to(dev).to(dtype)
    noise = noise.to(dev).to(dtype)
    basis = r_sqrt_sigma.T.float().to(dev).to(dtype) if dtype == torch.float32 else r_sqrt_sigma.T.to(dev).to(dtype)
    E = clamped_probit(torch.tensordot(noise, basis, dims=1) + fe_out, eps1)
    E_x = clamped_probit(torch.tensordot(noise, basis, dims=1) + fx_out, eps1)
    E_loss, E_x_loss = loss_side(E, keep[None, :, None]), loss_side(E_x, keep[None, :, None])

    terms = [_row_nll(E_loss, y, mask, lw, accum), _row_nll(E_x_loss, y, mask, lw, accum),
             _row_ranking(E_loss, y, mask, ranking, accum), _row_ranking(E_x_loss, y, mask, ranking, accum), kl]
    nll, nll_x, c, c_x, kl = (torch.where(live, t * w.to(t.dtype), _zero(t)) for t in terms)
    total = (nll + nll_x) * nll_coeff + (c + c_x) * c_coeff + kl * 1.1
    src = (E_x, E) if accum is None else (E_x.to(accum), E.to(accum))
    return ElboTerms(total, nll, nll_x, c, c_x, kl, torch.mean(src[0], dim=0), torch.mean(src[1], dim=0))


def row_probit_elbo_with_grads(inputs: dict, noise, nll_coeff, c_coeff, upstream: dict, **kw):
    """(terms, {name: gradient}) of row_probit_elbo for the cotangents `upstream` ({output name: (B,) or (B, L)}).  A
    row whose six per-row cotangents are all 0 (or absent) carries no loss gradient."""
    B = inputs["y"].shape[0]
    grad_rows = torch.zeros(B, dtype=torch.bool)
    for k in ROW_TERMS:
        if k in upstream:
            grad_rows |= upstream[k].cpu() != 0
    leaves = {k: inputs[k].detach().clone().requires_grad_(True) for k in _NAMES}
    terms = row_probit_elbo(inputs["y"], *(leaves[k] for k in _NAMES), noise, nll_coeff, c_coeff, grad_rows=grad_rows,
                            **kw)
    objective = sum((getattr(terms, k) * v.to(getattr(terms, k).dtype)).sum() for k, v in upstream.items())
    grads = torch.autograd.grad(objective, [leaves[k] for k in _NAMES], allow_unused=True)
    return terms, {k: g for k, g in zip(_NAMES, grads)}


def row_loss_fn(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args, noise=None,
                label_mask=None, row_weight=None, reduction="none"):
    """compute_loss(..., reduction='none')-shaped wrapper (a `loss_fn` for train.DataParallelStep(row_objective=)) on the
    CPU: needs an explicit noise tensor."""
    assert reduction == "none"
    return row_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise,
                           args.nll_coeff, args.c_coeff, row_weight, label_mask, ranking="factorised")
