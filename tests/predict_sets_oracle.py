"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Set prediction in fp64 torch: the label sampler of mpvae_probit_sample_labels
(y = U < E, E the per-sample clamped probit of tests/predict_oracle.py, U the caller's or the library's Philox stream),
the bit packing, the GFM decoder of mpvae_f1_sets and a brute-force search over every label set."""
from __future__ import annotations

import itertools

import numpy as np
import torch

from oracle.probit_elbo_oracle import clamped_probit
from tests.predict_oracle import _stable_probit

SET_KEY = 0x53455421     # csrc/sets.cu kSetKey


def sample_E(fx_out, r_sqrt_sigma, noise, stable=False):
    """(S, B, L) fp32 E(noise . R^T + fx_out), op for op the E that predict_oracle.predict averages."""
    dev = fx_out.device
    x = torch.tensordot(noise.to(dev).float(), r_sqrt_sigma.T.float().to(dev), dims=1) + fx_out.float()
    return _stable_probit(x) if stable else clamped_probit(x, torch.tensor([1e-6]).float().to(dev))


def probit64(x):
    """E = c + k Phi(x) in fp64 (c = 1e-6 / 2, k = 1 - 1e-6): the clamped probit of exact arithmetic."""
    return 0.5e-6 + (1.0 - 1e-6) * 0.5 * torch.special.erfc(-x.double() / 2 ** 0.5)


def library_uniform(S, B, L, seed, offset, b_global=None, row0=0):
    """(S, B, L) fp64 U of the library's stream: counter (s * B_global + row0 + b) * ceil(L / 4) + l // 4, key = the seed
    xor SET_KEY, U = ((r >> 8) + 1/2) 2^-24 from word l % 4 of the Philox output (exact in fp64)."""
    from tests.test_kernels_gpu import philox4x32_10_numpy
    Bg = B if b_global is None else b_global
    q = (L + 3) // 4
    s, b, c = np.meshgrid(np.arange(S, dtype=np.uint64), np.arange(B, dtype=np.uint64), np.arange(q, dtype=np.uint64),
                          indexing="ij")
    ctr = ((s * np.uint64(Bg) + np.uint64(row0) + b) * np.uint64(q) + c).reshape(-1)
    r = philox4x32_10_numpy(ctr, offset, seed ^ SET_KEY)
    words = np.stack(r, 1).reshape(S, B, q * 4)[:, :, :L]
    return torch.from_numpy(((words >> np.uint64(8)).astype(np.float64) + 0.5) / 16777216.0)


def sample(E, U):
    """(S, B, L) bool y = U < E, compared in fp64 (E fp32, U fp32 or the library's 25-bit values: both exact)."""
    return U.to(E.device).double() < E.double()


def pack(y):
    """(S, B, L) or (B, S, L) 0/1 -> int32 words along the last axis, label l at bit l % 32 of word l // 32."""
    *lead, L = y.shape
    W = (L + 31) // 32
    pad = torch.zeros(*lead, W * 32, dtype=torch.int64, device=y.device)
    pad[..., :L] = y.long()
    w = (pad.reshape(*lead, W, 32) << torch.arange(32, device=y.device)).sum(-1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)


def gfm(y, beta=1.0, max_size=None):
    """y (B, S, L) 0/1 -> (sets (B, L) bool, expected_f (B,) fp64, size (B,) int64), the GFM decoder of mpvae_f1_sets:
    Delta_{l,k} = mean_i y_il (1 + b^2) / (b^2 s_i + k), EF(k) = the k largest over the labels set in any sample,
    EF(0) = P0, the smallest argmax, ties to the lower label index.  Delta is summed over the samples in order, as the
    kernel sums it, so that labels whose Delta ties in exact arithmetic tie here too."""
    y = y.double()
    B, S, L = y.shape
    b2 = float(beta) * float(beta)
    s = y.sum(2)
    nu = (y.sum(1) > 0).sum(1)
    best = (s == 0).double().mean(1)
    size = torch.zeros(B, dtype=torch.int64, device=y.device)
    sets = torch.zeros(B, L, dtype=torch.bool, device=y.device)
    K = L if max_size is None else min(int(max_size), L)
    for k in range(1, K + 1):
        w = (1.0 + b2) / (b2 * s + k)
        delta = torch.zeros(B, L, dtype=torch.float64, device=y.device)
        for i in range(S):
            delta = delta + y[:, i] * w[:, i, None]
        delta = delta / S
        vals, idx = torch.sort(delta, dim=1, descending=True, stable=True)
        ef = vals[:, :k].sum(1)
        up = (nu >= k) & (ef > best)
        best = torch.where(up, ef, best)
        size = torch.where(up, torch.full_like(size, k), size)
        top = torch.zeros_like(sets)
        top.scatter_(1, idx[:, :k], True)
        sets = torch.where(up[:, None], top, sets)
    return sets, best, size


def f_measure(h, y, beta=1.0):
    """F_beta of predicted sets h against label sets y (broadcasting over leading axes), 1 where both are empty."""
    h, y = h.double(), y.double()
    b2 = float(beta) ** 2
    tp = (h * y).sum(-1)
    den = b2 * y.sum(-1) + h.sum(-1)
    return torch.where(den == 0, torch.ones_like(tp), (1 + b2) * tp / den.clamp_min(1e-300))


def brute_force(y, beta=1.0, max_size=None):
    """y (S, L) 0/1 of one row -> (the expected F of every set of at most max_size labels, those sets as bool (n, L)),
    over the 2^L label sets."""
    S, L = y.shape
    K = L if max_size is None else min(int(max_size), L)
    hs = torch.tensor(list(itertools.product((0, 1), repeat=L)), dtype=torch.float64).flip(1)
    hs = hs[hs.sum(1) <= K]
    ef = f_measure(hs[:, None, :], y.double()[None, :, :].cpu(), beta).mean(1)
    return ef, hs.bool()
