"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The conditional prediction of mpvae.predict_conditional restated with the pinned
oracle's pieces: E from `clamped_probit` (or predict_oracle's `_stable_probit`), the per-sample log-likelihood from the
cell formula of `bernoulli_log_mean_exp` (log E * y + log(1 - E) * (1 - y)) over the observed labels only, given an
explicit (S, B, Z) noise tensor.  Per row:
    lp_s = sum_{o in O} ll_{s,o} (fp64),  m = max_s fp32(lp_s),  u_s = exp(fp32(lp_s) - m),  se = sum_s u_s (fp64)
    prob = sum_s u_s E_s / se   (unobserved),  observed value (observed)
    log_evidence = log(fp32(se) / S) + m,  ess = se^2 / sum_s u_s^2"""
from __future__ import annotations

import torch

from oracle.probit_elbo_oracle import clamped_probit
from tests.predict_oracle import _stable_probit


def samples(fx_out, r_sqrt_sigma, observed, noise, stable=False):
    """(E (S, B, L) fp32, u (S, B) fp32, m (B,) fp32, mask (B, L) bool, y (B, L) fp32) of the estimator."""
    dev = fx_out.device
    fx_out = fx_out.float()
    noise = noise.to(dev).float()
    basis = r_sqrt_sigma.T.float().to(dev)
    x = torch.tensordot(noise, basis, dims=1) + fx_out              # mpvae.py:170
    if stable:
        E, om = _stable_probit(x), _stable_probit(-x)
    else:
        eps1 = torch.tensor([1e-6]).float().to(dev)
        E = clamped_probit(x, eps1)                                  # mpvae.py:180
        om = 1 - E
    observed = observed.to(dev)
    mask = (observed == 0) | (observed == 1)
    y = (observed == 1).float()
    cell = torch.log(E) * y + torch.log(om) * (1 - y)               # bernoulli_log_mean_exp's cell, negated
    lp = torch.where(mask, cell.double(), torch.zeros((), dtype=torch.float64, device=dev)).sum(2)   # (S, B)
    lp32 = lp.float()
    m = lp32.max(0)[0]
    u = torch.exp(lp32 - m)
    return E, u, m, mask, y


def predict_conditional(fx_out, r_sqrt_sigma, observed, noise, stable=False):
    """(prob (B, L) fp32, log_evidence (B,) fp32, ess (B,) fp64).  With nothing observed (u = 1) prob is
    predict_oracle.predict bit for bit: the weighted mean is taken as mean_s(u E) * (S / fse)."""
    E, u, m, mask, y = samples(fx_out, r_sqrt_sigma, observed, noise, stable)
    S = E.shape[0]
    se = u.double().sum(0)
    fse = se.float()
    prob = torch.mean(u[:, :, None] * E, dim=0) * (S / fse)[:, None]
    prob = torch.where(mask, y, prob)
    log_evidence = torch.log(fse / S) + m
    ess = se * se / (u.double() ** 2).sum(0)
    return prob, log_evidence, ess


def stderr(fx_out, r_sqrt_sigma, observed, noise, stable=False):
    """(B, L) fp64 delta-method standard error of the self-normalised mean: sqrt(sum_s u_s^2 (E_s - p)^2) / sum_s u_s."""
    E, u, _, mask, _ = samples(fx_out, r_sqrt_sigma, observed, noise, stable)
    u, E = u.double()[:, :, None], E.double()
    p = (u * E).sum(0) / u.sum(0)
    return torch.sqrt((u * u * (E - p) ** 2).sum(0)) / u.sum(0)
