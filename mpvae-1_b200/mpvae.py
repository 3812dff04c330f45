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

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .dense import linear
from .probit import ProbitELBO, philox_normal, probit_predict

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


def compute_loss(input_label, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r_sqrt_sigma, args, noise=None):
    """Reference signature (mpvae.py:145) -> (total_loss, nll_loss, nll_loss_x, c_loss, c_loss_x, kl_loss,
    indiv_prob, indiv_prob_label) (mpvae.py:210)."""
    device = input_label.device
    if device.type != "cuda":
        raise RuntimeError("mpvae_b200.compute_loss needs CUDA tensors: the probit ELBO is implemented as sm_100a "
                           "kernels only (no CPU fallback)")
    n_sample = args.n_train_sample if args.mode == "train" else args.n_test_sample   # mpvae.py:158
    n_batch = fe_out.shape[0]
    if n_batch == 0:
        # train.py:102 runs int(N/bs)+1 steps, so an empty last batch reaches the loss: every mean is NaN
        nan = (fe_out.sum() + fx_out.sum() + fe_mu.sum() + fe_logvar.sum() + fx_mu.sum() + fx_logvar.sum()) * math.nan
        empty = fx_out.new_empty((0, fx_out.shape[1]))
        return (nan, nan.clone(), nan.clone(), nan.clone(), nan.clone(), nan.clone(), empty, empty.clone())
    r32 = r_sqrt_sigma.to(device).float()                # mpvae.py:165 -- outside the Function: grad returns as fp64
    noise, spec = noise_plan(args, n_sample, n_batch, device, noise)
    flags = int(getattr(args, "mpvae_flags", 0))
    # args.peer_ring (peer.PeerRing, data-parallel runs): g_R comes back already summed over the ranks
    return ProbitELBO.apply(input_label.float(), fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise,
                            float(args.nll_coeff), float(args.c_coeff), flags, spec, getattr(args, "peer_ring", None))


def predict(fx_out, r_sqrt_sigma, args, noise=None):
    """The prediction `indiv_prob` (B, L) of compute_loss in test mode (mpvae.py:170,180,203) from the feature branch
    alone (`VAE.feat_forward(feature)[0]`): no labels, no label branch, no loss.  Same S (args.n_test_sample), same
    noise (`noise_plan`: a call without args.noise_offset consumes one offset, as compute_loss does), same flags, and
    bit for bit the indiv_prob compute_loss returns for the same fx_out.  Inference only: it builds no autograd graph."""
    if torch.is_grad_enabled() and (fx_out.requires_grad or r_sqrt_sigma.requires_grad):
        raise RuntimeError("mpvae_b200.predict is inference only and returns no gradient: call it under torch.no_grad() "
                           "(or detach its inputs); compute_loss is the differentiable path")
    device = fx_out.device
    if device.type != "cuda":
        raise RuntimeError("mpvae_b200.predict needs CUDA tensors: the probit prediction is implemented as sm_100a "
                           "kernels only (no CPU fallback)")
    n_sample = args.n_test_sample
    n_batch = fx_out.shape[0]
    if n_batch == 0:
        return fx_out.new_empty((0, fx_out.shape[1]))
    r32 = r_sqrt_sigma.to(device).float()
    noise, spec = noise_plan(args, n_sample, n_batch, device, noise)
    flags = int(getattr(args, "mpvae_flags", 0))
    return probit_predict(fx_out, r32, n_sample, noise=noise, noise_spec=spec, flags=flags)


probit_elbo = compute_loss
FLAG_SANITIZE_DEGENERATE = _lib.FLAG_SANITIZE_DEGENERATE
FLAG_STABLE_CDF = _lib.FLAG_STABLE_CDF
FLAG_CONTRACT_TENSOR = _lib.FLAG_CONTRACT_TENSOR
FLAG_CONTRACT_FMA = _lib.FLAG_CONTRACT_FMA
FLAG_FUSED_FORWARD = _lib.FLAG_FUSED_FORWARD
FLAG_SEPARATE_NOISE = _lib.FLAG_SEPARATE_NOISE
FLAG_FUSED_EXCHANGE = _lib.FLAG_FUSED_EXCHANGE
FLAG_SERIAL_EXCHANGE = _lib.FLAG_SERIAL_EXCHANGE
