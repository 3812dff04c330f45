"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The closed form of the probit predictive distribution in fp64, from formulas
independent of the library's code: Phi from torch.special.ndtr, the bivariate normal CDF from Owen's T function
(scipy.special.owens_t) instead of the kernels' Gauss-Legendre quadrature.

With n = R eps, eps ~ N(0, I_Z), s_l = |R_l|^2 and a = fx_out:
    P(y_l = 1)            = c + k Phi(h_l),                          h_l = a_l / sqrt(1 + s_l)
    P(y_i = 1, y_j = 1)   = c^2 + c k (Phi(h_i) + Phi(h_j)) + k^2 Phi2(h_i, h_j; rho_ij),
                            rho_ij = R_i . R_j / sqrt((1 + s_i)(1 + s_j))
    Var_n(E_l)            = k^2 (Phi2(h_l, h_l; s_l / (1 + s_l)) - Phi(h_l)^2)
with E(x) = c + k Phi(x) the clamped probit of mpvae.py:177, c = eps1 / 2, k = 1 - eps1, eps1 = fp32(1e-6)."""
from __future__ import annotations

import numpy as np
import torch
from scipy.special import ndtr as _ndtr_np
from scipy.special import owens_t

EPS1 = float(np.float32(1e-6))
C_EPS = EPS1 * 0.5
K_EPS = 1.0 - EPS1


def scale(r):
    """(L,) fp64: 1 / sqrt(1 + |R_l|^2) of the fp32 R the kernels read."""
    r64 = r.detach().cpu().float().double()
    return 1.0 / torch.sqrt(1.0 + (r64 * r64).sum(1))


def rho(r, pairs):
    r64 = r.detach().cpu().float().double()
    p = torch.as_tensor(pairs).long().cpu()
    sc = scale(r)
    return (r64[p[:, 0]] * r64[p[:, 1]]).sum(1) * sc[p[:, 0]] * sc[p[:, 1]]


def h_arg(fx_out, r):
    """(B, L) fp64 h = fx_out * scale."""
    return fx_out.detach().cpu().float().double() * scale(r)[None, :]


def marginal_at_t(fx_out, r):
    """(B, L) fp64 c + k Phi at the fp32 argument the kernels' probit_E_stable evaluates: t = fp32(x' * fp32(1 /
    1.41421354)) with x' = fp32(fx_out * scale), then c + k erfc(-t) / 2 in fp64.  Isolates the accuracy of the CDF
    evaluation from the two argument roundings (which move Phi by up to ~2 t^2 * 6e-8 relative in the lower tail)."""
    x = h_arg(fx_out, r).float()
    t = (x * torch.tensor(1.0 / 1.41421354, dtype=torch.float32)).double()
    return C_EPS + K_EPS * 0.5 * torch.special.erfc(-t)


def marginal(fx_out, r):
    """(B, L) fp64 P(y = 1) = c + k Phi(h)."""
    return C_EPS + K_EPS * torch.special.ndtr(h_arg(fx_out, r))


def bvn(h, k, r):
    """Phi2(h, k; rho) elementwise (numpy broadcasting), fp64, by Owen (1956):
        Phi2 = Phi(h)/2 + Phi(k)/2 - T(h, (k - rho h) / (h s)) - T(k, (h - rho k) / (k s)) - beta,   s = sqrt(1 - rho^2)
    beta = 0 when hk > 0 or (hk = 0 and h + k >= 0), else 1/2; T(0, +-inf) = +-1/4; Phi2(0, 0) = 1/4 + asin(rho) / 2 pi;
    |rho| = 1: the degenerate limits."""
    h, k, r = (np.asarray(v, dtype=np.float64) for v in np.broadcast_arrays(h, k, r))
    s = np.sqrt((1.0 - r) * (1.0 + r))
    # k - rho h as (k -+ h) +- (1 -+ rho) h: exact differences, so no cancellation when |rho| is next to 1
    pos = r >= 0.0
    dkh = np.where(pos, (k - h) + (1.0 - r) * h, (k + h) - (1.0 + r) * h)
    dhk = np.where(pos, (h - k) + (1.0 - r) * k, (h + k) - (1.0 + r) * k)
    with np.errstate(divide="ignore", invalid="ignore"):
        ah = dkh / (h * s)
        ak = dhk / (k * s)
        th = np.where(h == 0.0, 0.25 * np.sign(dkh), owens_t(h, np.where(h == 0.0, 0.0, ah)))
        tk = np.where(k == 0.0, 0.25 * np.sign(dhk), owens_t(k, np.where(k == 0.0, 0.0, ak)))
    beta = np.where((h * k > 0.0) | ((h * k == 0.0) & (h + k >= 0.0)), 0.0, 0.5)
    out = 0.5 * _ndtr_np(h) + 0.5 * _ndtr_np(k) - th - tk - beta
    out = np.where((h == 0.0) & (k == 0.0), 0.25 + np.arcsin(r) / (2.0 * np.pi), out)
    out = np.where(r >= 1.0, _ndtr_np(np.minimum(h, k)), out)
    out = np.where(r <= -1.0, np.maximum(0.0, _ndtr_np(h) + _ndtr_np(k) - 1.0), out)
    return np.clip(out, 0.0, 1.0)


def pair_prob(fx_out, r, pairs):
    """(B, P) fp64 P(y_i = 1, y_j = 1) for the (P, 2) label pairs; a pair (i, i) gives the marginal."""
    p = torch.as_tensor(pairs).long().cpu()
    h = h_arg(fx_out, r).numpy()
    hi, hj = h[:, p[:, 0].numpy()], h[:, p[:, 1].numpy()]
    rr = rho(r, p).numpy()[None, :]
    b2 = bvn(hi, hj, rr)
    out = C_EPS * C_EPS + C_EPS * K_EPS * (_ndtr_np(hi) + _ndtr_np(hj)) + K_EPS * K_EPS * b2
    diag = (p[:, 0] == p[:, 1]).numpy()
    out[:, diag] = C_EPS + K_EPS * _ndtr_np(hi[:, diag])
    return torch.from_numpy(out)


def marginal_var(fx_out, r):
    """(B, L) fp64 variance over the probit noise of the sample E(fx_out + n_l) that mpvae.predict averages."""
    r64 = r.detach().cpu().float().double()
    s = (r64 * r64).sum(1)
    h = h_arg(fx_out, r).numpy()
    rr = (s / (1.0 + s)).numpy()[None, :]
    v = K_EPS * K_EPS * (bvn(h, h, rr) - _ndtr_np(h) ** 2)
    return torch.from_numpy(np.maximum(v, 0.0))
