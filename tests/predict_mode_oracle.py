"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Mode prediction in fp64 torch: the probability of a label set under the S-sample
mixture of mpvae_probit_score_sets, its effective sample size, the candidates and the steepest single-flip ascent of
mpvae_probit_predict_mode, and an exhaustive search over every label set.

Inputs are per-sample probabilities E (S, B, L) fp32, the E that predict averages.  The cell logs are the loss's fp32
logs: ll+ = log E, ll- = log(1 - E) with 1 - E rounded to fp32 (the reference's CDF mode).  On a CUDA tensor these are
the library's logs bit for bit (torch's fp32 log is logf there); the host's log may differ in the last bit."""
from __future__ import annotations

import itertools

import torch


def cell_logs(E):
    """(ll+, ll-) (S, B, L) fp64 of the fp32 logs log E and log(1 - E)."""
    E = E.float()
    return torch.log(E).double(), torch.log(1.0 - E).double()


def lp(llp, lln, y):
    """lp_s(y) (B, C, S) fp64 for sets y (B, C, L) 0/1: A_s + sum_{l in y} d_sl."""
    A = lln.sum(2)                                   # (S, B)
    d = llp - lln                                    # (S, B, L)
    return A.T[:, None, :] + torch.einsum("bcl,sbl->bcs", y.double(), d)


def mixture(lps):
    """(log_prob, ess) of lp_s along the last axis: M + log mean_s exp(lp_s - M), (sum w)^2 / sum w^2."""
    m = lps.max(-1, keepdim=True).values
    w = torch.exp(lps - m)
    se = w.sum(-1)
    return m[..., 0] + torch.log(se / lps.shape[-1]), se * se / (w * w).sum(-1)


def score(llp, lln, y):
    """(log_prob (B, C), ess (B, C)) of the sets y (B, C, L)."""
    return mixture(lp(llp, lln, y))


def direct_log_prob(E, y):
    """log of the mean over s of prod_l (y_l ? E : 1 - E), straight from the definition in fp64 (for small L, where the
    product does not underflow)."""
    llp, lln = cell_logs(E)
    p = torch.where(y.bool()[:, :, None, :], llp.permute(1, 0, 2)[:, None], lln.permute(1, 0, 2)[:, None])
    return torch.log(torch.exp(p.sum(-1)).mean(-1))


def indiv_prob(E):
    """predict's indiv_prob from the per-sample E: pair sums E_s + E_{s+1} in fp32, pairs added in order, / S."""
    E = E.float()
    S = E.shape[0]
    acc = torch.zeros_like(E[0])
    for s0 in range(0, S, 2):
        acc = acc + (E[s0] + E[s0 + 1] if s0 + 1 < S else E[s0])
    return acc / float(S)


def candidates(E):
    """(B, S + 2, L) bool: 1[indiv_prob >= 0.5], the empty set, then each sample's mode 1[ll+ > ll-]."""
    llp, lln = cell_logs(E)
    c0 = indiv_prob(E) >= 0.5
    modes = (llp > lln).permute(1, 0, 2)
    return torch.cat([c0[:, None], torch.zeros_like(c0)[:, None], modes], 1)


def mode(E, max_flips=None):
    """(sets (B, L) bool, log_prob (B,), ess (B,), size (B,), flips (B,)) of mpvae_probit_predict_mode: the best candidate
    (ties to the earliest), then while flips < max_flips the label with the largest G_l = sum_s w_s exp(+-d_sl) (ties to
    the lower index) is flipped when G_l > T = sum_s w_s, lp_s updated by +-d_sl."""
    llp, lln = cell_logs(E)
    d = (llp - lln).permute(1, 0, 2)                 # (B, S, L)
    cand = candidates(E)
    cl, _ = score(llp, lln, cand)
    B, L = cand.shape[0], cand.shape[2]
    start = torch.argmax((cl == cl.max(1, keepdim=True).values).to(torch.int8), 1)     # the first of the best
    y = cand[torch.arange(B, device=E.device), start].clone()
    cur = lp(llp, lln, y[:, None])[:, 0]             # (B, S)
    flips = torch.zeros(B, dtype=torch.int64, device=E.device)
    active = torch.ones(B, dtype=torch.bool, device=E.device)
    limit = float("inf") if max_flips is None else int(max_flips)
    while bool(active.any()):
        active &= flips < limit
        if not bool(active.any()):
            break
        m = cur.max(1, keepdim=True).values
        w = torch.exp(cur - m)
        T = w.sum(1)
        sign = torch.where(y, -1.0, 1.0).double()    # (B, L)
        G = (w[:, :, None] * torch.exp(sign[:, None, :] * d)).sum(1)      # (B, L)
        gbest = G.max(1).values
        l = torch.argmax((G == gbest[:, None]).to(torch.int8), 1)
        take = active & (gbest > T)
        rows = torch.nonzero(take)[:, 0]
        if len(rows) == 0:
            break
        cur[rows] += sign[rows, l[rows]][:, None] * d[rows, :, l[rows]]
        y[rows, l[rows]] = ~y[rows, l[rows]]
        flips[rows] += 1
        active = take
    log_prob, ess = score(llp, lln, y[:, None])
    return y, log_prob[:, 0], ess[:, 0], y.sum(1), flips


def all_sets(L):
    """(2^L, L) bool, every label set."""
    return torch.tensor(list(itertools.product((0, 1), repeat=L)), dtype=torch.bool).flip(1)


def exhaustive(E):
    """(log_prob (B, 2^L), sets (2^L, L)): every label set scored for each row."""
    hs = all_sets(E.shape[2]).to(E.device)
    llp, lln = cell_logs(E)
    lpb, _ = score(llp, lln, hs[None].expand(E.shape[1], -1, -1))
    return lpb, hs
