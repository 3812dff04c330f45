"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The ELBO with label weights (compute_loss(..., pos_weight=, neg_weight=)), restated
from the weighted oracle (tests/weighted_elbo_oracle.py) with the (2, L) weights applied to each cell's log-likelihood
before the mask, the log-mean-exp over samples and the row weights:
    ll_{s,b,l} = where(w1_l != 0, log E * y * w1_l, 0) + where(w0_l != 0, log(1 - E) * (1 - y) * w0_l, 0)
    nll_b      = -log mean_s exp(sum over the observed l of ll_{s,b,l})       (each branch)
    loss       = mean_b where(v_b != 0, v_b * t_b, 0)                         (v: the row weights)
w0 (row 0 of label_weight) weighs the y == 0 part, w1 (row 1) the y == 1 part.  A zero weight selects its term away, so
its gradient is exactly 0 whatever the cell holds.  The ranking terms, KL and the predictions are the weighted
oracle's.  With all-ones weights every product with w is the unweighted value bit for bit, so the terms and the
gradients are the weighted oracle's."""
from __future__ import annotations

import torch

from oracle.probit_elbo_oracle import ElboTerms, clamped_probit
from tests.masked_elbo_oracle import _zero
from tests.weighted_elbo_oracle import (_NAMES, _weighted_mean, weighted_gaussian_kl, weighted_ranking_loss_factorised,
                                        weighted_ranking_loss_pairwise)


def label_weighted_bernoulli_log_mean_exp(E, y, mask, lw, w, live, accum=None):
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
    return _weighted_mean(-torch.log(mean_exp) - peak, w, live)


def label_weighted_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise,
                               nll_coeff, c_coeff, label_weight, row_weight=None, label_mask=None, *,
                               ranking: str = "pairwise", dtype: torch.dtype = torch.float32, accum=None) -> ElboTerms:
    """The weighted oracle's ELBO with the (2, L) label weights `label_weight` (row_weight None = every row weighs 1,
    label_mask None = every label observed)."""
    dev = input_label.device
    mask = torch.ones(input_label.shape, dtype=torch.bool, device=dev) if label_mask is None else label_mask.to(dev).bool()
    w = (torch.ones(input_label.shape[0]) if row_weight is None else row_weight).to(dev).to(dtype)
    lw = label_weight.to(dev).to(dtype)
    live = w != 0
    cut = not bool(live.all())

    def loss_side(t, rows):
        return torch.where(rows, t, t.detach()) if cut else t

    y = input_label.to(dtype)
    y = torch.where(mask, y, _zero(y))
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
    nll = label_weighted_bernoulli_log_mean_exp(E_loss, y, mask, lw, w, live, accum)
    c = rank(E_loss, y, mask, w, live, accum)
    nll_x = label_weighted_bernoulli_log_mean_exp(E_x_loss, y, mask, lw, w, live, accum)
    c_x = rank(E_x_loss, y, mask, w, live, accum)

    if accum is not None:
        indiv_prob = torch.mean(E_x.to(accum), dim=0)
        indiv_prob_label = torch.mean(E.to(accum), dim=0)
    else:
        indiv_prob = torch.mean(E_x, dim=0)
        indiv_prob_label = torch.mean(E, dim=0)

    total = (nll + nll_x) * nll_coeff + (c + c_x) * c_coeff + kl * 1.1
    return ElboTerms(total, nll, nll_x, c, c_x, kl, indiv_prob, indiv_prob_label)


def label_weighted_probit_elbo_with_grads(inputs: dict, noise, nll_coeff, c_coeff, label_weight, row_weight=None,
                                          label_mask=None, *, upstream=None, **kw):
    """(terms, {name: gradient}) of label_weighted_probit_elbo; default cotangent d total_loss = 1."""
    leaves = {k: inputs[k].detach().clone().requires_grad_(True) for k in _NAMES}
    terms = label_weighted_probit_elbo(inputs["y"], *(leaves[k] for k in _NAMES), noise, nll_coeff, c_coeff, label_weight,
                                       row_weight, label_mask, **kw)
    if upstream is None:
        objective = terms.total_loss
    else:
        objective = sum((getattr(terms, k) * v.to(getattr(terms, k).dtype)).sum() for k, v in upstream.items())
    grads = torch.autograd.grad(objective, [leaves[k] for k in _NAMES], allow_unused=True)
    return terms, {k: g for k, g in zip(_NAMES, grads)}


def pack(pos_weight, neg_weight, L, dtype=torch.float32):
    """compute_loss's packing: [neg_weight; pos_weight] with None = ones"""
    ones = torch.ones(L, dtype=dtype)
    return torch.stack([ones if neg_weight is None else neg_weight.cpu().to(dtype),
                        ones if pos_weight is None else pos_weight.cpu().to(dtype)])


def label_weighted_loss_fn(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args,
                           noise=None, label_mask=None, row_weight=None, pos_weight=None, neg_weight=None):
    """compute_loss-shaped wrapper (a `loss_fn` for train.DataParallelStep) on the CPU: needs an explicit noise tensor."""
    lw = pack(pos_weight, neg_weight, input_label.shape[1])
    return label_weighted_probit_elbo(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, noise,
                                      args.nll_coeff, args.c_coeff, lw, row_weight, label_mask, ranking="factorised")
