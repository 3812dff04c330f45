"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The GHK conditional prediction of mpvae.predict_conditional_ghk restated in fp64
torch, given explicit draws: the probit noise xi (S, B, Z), and zeta (S, B, L) and U (S, B, L) at the observed cells.

Latent form: u = fx + R eps + w, P(y = 1 | u) = c + k 1[u > 0].  Per row, O = observed labels in ascending order,
C = chol(I + G[O, O]) with G = R R^T, n_s = R xi_s:
    for k:  m_k = fx_{o_k} + sum_{j<k} C_kj eta_j,  a = -m_k / C_kk,  eta_k = draw(a, y_k, U),  lw += log Z_k
    v = C^-T (eta - C^-1 (n_O + zeta)),  x = n + G[:, O] v
    prob = sum_s u_s E(fx + x_s) / sum_s u_s (unobserved),  log_evidence = log mean exp(lw),  ess = (sum u)^2 / sum u^2
with E = c + k Phi in fp64."""
from __future__ import annotations

import math

import torch

from tests.predict_exact_oracle import C_EPS, K_EPS


def _ndtri(p):
    return torch.special.ndtri(p)


def draw_upper(a, U, V):
    """eta from the density proportional to (c + k 1[eta > a]) phi(eta) at the uniform U (V = 1 - U): (eta, Z)."""
    Qa = 0.5 * torch.special.erfc(a * 0.7071067811865476)
    Z = C_EPS + K_EPS * Qa
    lower = V * Z >= (C_EPS + K_EPS) * Qa
    p = U * Z / C_EPS
    tl = torch.where(p <= 0.5, _ndtri(p.clamp(max=1.0)), -_ndtri((V - U * K_EPS * Qa / C_EPS).clamp(0.0, 1.0)))
    tl = torch.minimum(tl, a)
    q = V * Z / (C_EPS + K_EPS)
    tu = torch.where(q <= 0.5, -_ndtri(q.clamp(max=1.0)), _ndtri(((U * C_EPS + K_EPS * (1.0 - V * Qa)) / (C_EPS + K_EPS))
                                                                  .clamp(0.0, 1.0)))
    tu = torch.maximum(tu, a)
    return torch.where(lower, tl, tu), Z


def draw(a, y, U):
    """The clamped truncated conditional of the observed latent: y = 1 keeps eta > a, y = 0 eta < a (as the
    reflection).  F_y(eta) = U for both.  Returns (eta, Z) with Z = c + k Phi(-+a), the cell probability."""
    a = torch.as_tensor(a, dtype=torch.float64) if not torch.is_tensor(a) else a
    U = torch.as_tensor(U, dtype=a.dtype)
    V = 1.0 - U
    e1, z1 = draw_upper(a, U, V)
    e0, z0 = draw_upper(-a, V, U)
    y = torch.as_tensor(y).bool()
    return torch.where(y, e1, -e0), torch.where(y, z1, z0)


def cdf(eta, a, y):
    """F_y(eta) of the clamped truncated conditional, in fp64 (numpy / scipy), for the sampler's check."""
    import numpy as np
    from scipy.special import ndtr
    eta, a = np.asarray(eta, dtype=np.float64), np.asarray(a, dtype=np.float64)
    if y:
        Z = C_EPS + K_EPS * ndtr(-a)
        return np.where(eta <= a, C_EPS * ndtr(eta) / Z, 1.0 - (C_EPS + K_EPS) * ndtr(-eta) / Z)
    Z = C_EPS + K_EPS * ndtr(a)
    return np.where(eta < a, (C_EPS + K_EPS) * ndtr(eta) / Z, 1.0 - C_EPS * ndtr(-eta) / Z)


def samples(fx_out, r, observed, xi, zeta, U, dtype=torch.float64):
    """(lw (S, B), x (S, B, L)) in fp64 (dtype = float32: the same algorithm restated in fp32, the yardstick of the
    dense regime)."""
    fx = fx_out.detach().cpu().to(dtype)
    R = r.detach().cpu().float().to(dtype)
    G = R @ R.T
    obs = observed.cpu()
    mask = (obs == 0) | (obs == 1)
    xi, zeta, U = (t.detach().cpu().to(dtype) for t in (xi, zeta, U))
    S, B = xi.shape[:2]
    x = torch.tensordot(xi, R.T, dims=1)
    lw = torch.zeros(S, B, dtype=dtype)
    for b in range(B):
        O = torch.nonzero(mask[b]).flatten()
        n = O.numel()
        if n == 0:
            continue
        Cf = torch.linalg.cholesky(torch.eye(n, dtype=dtype) + G[O][:, O])
        eta = torch.zeros(S, n, dtype=dtype)
        for k in range(n):
            m = fx[b, O[k]] + eta[:, :k] @ Cf[k, :k]
            eta[:, k], Zk = draw(-m / Cf[k, k], bool(obs[b, O[k]] == 1), U[:, b, O[k]])
            lw[:, b] += torch.log(Zk)
        w = torch.linalg.solve_triangular(Cf, (x[:, b, O] + zeta[:, b, O]).T, upper=False).T
        v = torch.linalg.solve_triangular(Cf.T, (eta - w).T, upper=True).T
        x[:, b] += v @ G[O]
    return lw, x


def predict_conditional_ghk(fx_out, r, observed, xi, zeta, U, dtype=torch.float64):
    """(prob (B, L), log_evidence (B,), ess (B,)) in fp64 (or the fp32 restatement)."""
    lw, x = samples(fx_out, r, observed, xi, zeta, U, dtype)
    S = lw.shape[0]
    fx = fx_out.detach().cpu().to(dtype)
    E = C_EPS + K_EPS * torch.special.ndtr(fx + x)
    u = torch.exp(lw - lw.max(0)[0])
    prob = (u[:, :, None] * E).sum(0) / u.sum(0)[:, None]
    obs = observed.cpu()
    mask = (obs == 0) | (obs == 1)
    prob = torch.where(mask, (obs == 1).to(dtype), prob)
    log_evidence = torch.logsumexp(lw, 0) - math.log(S)
    ess = u.sum(0) ** 2 / (u * u).sum(0)
    return prob, log_evidence, ess


def stderr(fx_out, r, observed, xi, zeta, U):
    """((B, L) delta-method SE of prob, (B,) SE of log_evidence)."""
    lw, x = samples(fx_out, r, observed, xi, zeta, U)
    S = lw.shape[0]
    E = C_EPS + K_EPS * torch.special.ndtr(fx_out.detach().cpu().double() + x)
    u = torch.exp(lw - lw.max(0)[0])
    p = (u[:, :, None] * E).sum(0) / u.sum(0)[:, None]
    se_p = torch.sqrt((u[:, :, None] ** 2 * (E - p) ** 2).sum(0)) / u.sum(0)[:, None]
    se_le = u.std(0) / (u.mean(0) * math.sqrt(S))
    return se_p, se_le


def quadrature(fx_out, r, observed, nodes=80):
    """(prob (B, L), log_evidence (B,)) by Gauss-Hermite quadrature over eps (Z = 1 or 2): given eps the labels are
    independent with P(y_l = 1 | eps) = c + k Phi(fx_l + R_l eps)."""
    import numpy as np
    t, w = np.polynomial.hermite_e.hermegauss(nodes)
    w = w / math.sqrt(2 * math.pi)
    R = r.detach().cpu().float().double()
    Z = R.shape[1]
    t, w = torch.from_numpy(t), torch.from_numpy(w)
    if Z == 1:
        pts, wts = t[:, None], w
    elif Z == 2:
        pts = torch.stack(torch.meshgrid(t, t, indexing="ij"), -1).reshape(-1, 2)
        wts = (w[:, None] * w[None, :]).reshape(-1)
    else:
        raise ValueError("quadrature: Z must be 1 or 2")
    fx = fx_out.detach().cpu().double()
    obs = observed.cpu()
    mask = (obs == 0) | (obs == 1)
    y = (obs == 1).double()
    P = C_EPS + K_EPS * torch.special.ndtr(fx[None] + (pts @ R.T)[:, None, :])       # (Q, B, L)
    cell = torch.where(mask[None], torch.where(y[None] > 0, P, 1 - P), torch.ones_like(P))
    lik = cell.prod(2)                                                                  # (Q, B)
    ev = (wts[:, None] * lik).sum(0)
    prob = (wts[:, None, None] * lik[:, :, None] * P).sum(0) / ev[:, None]
    return torch.where(mask, y, prob), torch.log(ev)
