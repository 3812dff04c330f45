"""ORACLE -- TEST INFRASTRUCTURE ONLY.  The prediction of compute_loss alone (reference mpvae.py:170,180,203), restated
with the pinned oracle's own pieces (`oracle/probit_elbo_oracle.py`: `clamped_probit` and the reference's op order), so
that it returns the bits of that oracle's `indiv_prob` -- and hence of the reference -- on the same inputs."""
from __future__ import annotations

import torch

from oracle.probit_elbo_oracle import clamped_probit


def _stable_probit(x):
    """MPVAE_FLAG_STABLE_CDF's E (csrc/probit_math.cuh::probit_E_stable): the smaller tail from erfc(|x| / sqrt 2)."""
    f32 = lambda v: torch.tensor(v, dtype=torch.float32, device=x.device)
    k, h = f32(1.0) - f32(1e-6), f32(1e-6) * f32(0.5)
    t = x * (f32(1.0) / f32(1.41421354))
    u = torch.special.erfc(t.abs())
    small = (f32(0.5) * u) * k + h
    large = (f32(1.0) - f32(0.5) * u) * k + h
    return torch.where(t < 0, small, large)


def predict(fx_out, r_sqrt_sigma, noise, stable=False):
    """indiv_prob (B, L) = mean_s E(noise . R^T + fx_out), noise (S, B, Z) -- the feature branch of
    probit_elbo_oracle.probit_elbo, op for op."""
    dev = fx_out.device
    fx_out = fx_out.float()
    noise = noise.to(dev).float()
    basis = r_sqrt_sigma.T.float().to(dev)                           # :165
    sample_r_x = torch.tensordot(noise, basis, dims=1) + fx_out      # :170
    if stable:
        E_x = _stable_probit(sample_r_x)
    else:
        eps1 = torch.tensor([1e-6]).float().to(dev)                  # :156
        E_x = clamped_probit(sample_r_x, eps1)                       # :180
    return torch.mean(E_x, dim=0)                                    # :203
