"""GPU: partially labelled training (compute_loss(..., label_mask=) -> mpvae_probit_forward_masked / _backward_masked, the
MASKED instantiations of the row kernels).  An all-ones mask against the unmasked call (bits), unobserved label values
(bits), the masked oracle, exact zeros of unobserved cells, the tie to predict_conditional's log-evidence, rows with
nothing observed, repeatability, a planted model trained on half-hidden labels, and DataParallelStep on one GPU."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import helpers as H
from tests import masked_elbo_oracle as MO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

SANITIZE, TENSOR, FMA, STABLE, SEPARATE = 0x1, 0x2, 0x4, 0x8, 0x20
LEAVES = ("fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma")


def _inputs(S, B, L, Z, external, seed, rate=None):
    from mpvae_b200 import synth
    inp = synth.loss_inputs(L, Z, B, S, seed=seed, sigma=1.0, label_rate=rate or max(0.05, 20.0 / L), with_noise=external)
    t = {k: torch.from_numpy(v).to(DEV) for k, v in inp.items()}
    return t, t.pop("noise", None)


def _args(S, L, Z, flags=0, mode="train", **kw):
    return orc.make_args(L, Z, n_train_sample=S, n_test_sample=S, mode=mode, noise_seed=4242, noise_offset=6,
                         mpvae_flags=flags, **kw)


def _run(t, noise, args, mask=None, y=None, upstream=None):
    """(8 outputs, {leaf: gradient}) of compute_loss + backward (default cotangent: total_loss)."""
    from mpvae_b200.mpvae import compute_loss
    leaves = {k: t[k].detach().clone().requires_grad_(True) for k in LEAVES}
    kw = {} if mask is None else {"label_mask": mask}
    out = compute_loss(t["y"] if y is None else y, *(leaves[k] for k in LEAVES), args, noise=noise, **kw)
    if upstream is None:
        out[0].backward()
    else:
        torch.autograd.backward([out[i] for i in upstream], [upstream[i] for i in upstream])
    torch.cuda.synchronize()
    return [o.detach() for o in out], {k: leaves[k].grad for k in LEAVES}


def _bits(a, b):
    """bit equality, NaN pattern included"""
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0))


def _random_mask(B, L, frac, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(B, L, generator=g) < frac).to(DEV)


# test_predict_gpu.EQUALITY_CASES (S, B, L, Z, flags, external noise): small, CUDA-core and dense regimes, S in
# {1, 3, 10, 100}, ragged B, L not a multiple of 4 or 128; plus SANITIZE with degenerate rows
ALL_ONES_CASES = [
    (10, 16, 38, 38, 0, False), (10, 16, 38, 38, 0, True), (1, 5, 14, 14, 0, False), (3, 33, 14, 14, 0, True),
    (100, 128, 81, 81, 0, False), (100, 37, 81, 81, 0, True),
    (10, 33, 3993, 10, 0, False), (3, 17, 3993, 10, 0, True), (100, 12, 983, 10, 0, False), (1, 9, 983, 10, 0, False),
    (10, 16, 38, 38, STABLE, False), (100, 7, 81, 81, STABLE, True), (10, 70, 983, 983, FMA, False), (3, 9, 130, 64, FMA, True),
    (10, 70, 983, 983, 0, False), (10, 70, 983, 983, 0, True), (3, 77, 130, 256, 0, True), (100, 12, 300, 128, SEPARATE, False),
    (1, 300, 256, 256, 0, False), (7, 5, 130, 64, TENSOR, False), (10, 40, 257, 300, STABLE, False),
    (3, 19, 983, 983, SEPARATE, True), (100, 1024, 3993, 3993, 0, False), (10, 1024, 3993, 3993, 0, False),
    (10, 16, 38, 38, SANITIZE, False), (10, 33, 983, 10, SANITIZE, False), (10, 70, 983, 983, SANITIZE, False),
]


@pytest.mark.parametrize("S,B,L,Z,flags,external", ALL_ONES_CASES)
def test_all_ones_mask_equals_unmasked(S, B, L, Z, flags, external):
    """Training mode (saved-E backward) and, for the small shapes, test mode too: all 8 outputs and every gradient bit
    for bit, including the NaN pattern of degenerate rows (two rows planted: all zeros, all ones)."""
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    t["y"][0] = 0.0
    if B > 1:
        t["y"][1] = 1.0
    ones = torch.ones(B, L, dtype=torch.bool, device=DEV)
    for mode in (("train", "test") if B * L <= 4096 else ("train",)):
        args = _args(S, L, Z, flags, mode)
        o0, g0 = _run(t, noise, args)
        o1, g1 = _run(t, noise, args, mask=ones)
        for i in range(8):
            assert _bits(o0[i], o1[i]), (mode, i)
        for k in LEAVES:
            assert _bits(g0[k], g1[k]), (mode, k)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (100, 37, 81, 81, 0), (10, 33, 983, 10, 0),
                                           (10, 20, 983, 983, 0), (10, 16, 38, 38, STABLE), (10, 12, 257, 300, STABLE)])
@pytest.mark.parametrize("fill", ["random", 0.5, 7.0, float("nan")])
def test_unobserved_label_values_have_no_effect(S, B, L, Z, flags, fill):
    t, noise = _inputs(S, B, L, Z, True, seed=7 * S + L)
    mask = _random_mask(B, L, 0.5, seed=B + L)
    args = _args(S, L, Z, flags)
    o0, g0 = _run(t, noise, args, mask=mask)
    other = (torch.rand(B, L, device=DEV) < 0.5).float() if fill == "random" else torch.full((B, L), fill, device=DEV)
    o1, g1 = _run(t, noise, args, mask=mask, y=torch.where(mask, t["y"], other))
    for i in range(8):
        assert _bits(o0[i], o1[i]), i
    for k in LEAVES:
        assert _bits(g0[k], g1[k]), k


def _oracle_mask(y, pattern, seed):
    """Mixed patterns; every row with something observed has an observed positive and negative (label 0 and 1 are
    planted), so no row is degenerate: the oracle has no SANITIZE, and degenerate rows are test_degenerate_rows'."""
    B, L = y.shape
    y[:, 0], y[:, 1] = 1.0, 0.0
    if pattern == "none":
        return torch.zeros(B, L, dtype=torch.bool, device=DEV)
    if pattern == "all":
        return torch.ones(B, L, dtype=torch.bool, device=DEV)
    m = _random_mask(B, L, pattern, seed)
    m[:, :2] = True
    m[0] = False                                     # a row with nothing observed
    if B > 2:
        m[1] = True                                  # a fully observed row
    return m


ORACLE_CASES = [(10, 16, 38, 38, 0), (1, 5, 14, 14, 0), (100, 37, 81, 81, 0), (10, 33, 983, 10, 0), (3, 17, 3993, 10, 0),
                (10, 20, 983, 983, 0), (7, 19, 130, 64, TENSOR), (10, 12, 257, 300, FMA)]


@pytest.mark.parametrize("S,B,L,Z,flags", ORACLE_CASES)
@pytest.mark.parametrize("pattern", ["none", "all", 0.1, 0.5, 0.9])
def test_against_the_masked_oracle(S, B, L, Z, flags, pattern):
    """The masked oracle in the reference's fp32 arithmetic on the same device: losses within 1e-5, predictions within
    1e-5 and thresholded decisions identical away from ties.  Gradients by the DESIGN section 5 rule against the fp64
    oracle: relative L2 <= max(1e-5, 2x the fp32 oracle's own), or the trimmed form with <= 1e-4; gradients that are
    exactly 0 in the oracle (nothing observed) exactly 0 here."""
    t, noise = _inputs(S, B, L, Z, True, seed=3 * S + L, rate=0.3)
    mask = _oracle_mask(t["y"], pattern, seed=S + B)
    args = _args(S, L, Z, flags)
    out, g = _run(t, noise, args, mask=mask)
    ranking = "factorised" if L > 128 else "pairwise"
    ref, rg32 = MO.masked_probit_elbo_with_grads(t, noise, args.nll_coeff, args.c_coeff, mask, ranking=ranking)
    tc = {k: v.cpu() for k, v in t.items()}
    _, rg = MO.masked_probit_elbo_with_grads(tc, noise.cpu(), args.nll_coeff, args.c_coeff, mask.cpu(), ranking=ranking,
                                             dtype=torch.float64)
    for i in range(6):
        want = float(ref[i])
        assert abs(float(out[i]) - want) <= 1e-5 * max(1.0, abs(want)), (i, float(out[i]), want)
    for i in (6, 7):
        got, want = out[i].cpu().numpy(), ref[i].detach().cpu().numpy()
        dp = float(np.max(np.abs(got.astype(np.float64) - want)))
        assert dp <= 1e-5, (i, dp)
        assert H.threshold_mismatches(got, want, tie=2 * dp + 1e-7) == 0
    for k in LEAVES:
        got, want, theirs = g[k].double().cpu().numpy(), rg[k].numpy(), rg32[k].double().cpu().numpy()
        if not np.any(want):
            assert not np.any(got), k
            continue
        e, et = H.rel_err_l2(got, want), H.rel_err_l2_trimmed(got, want)
        r, rt = H.rel_err_l2(theirs, want), H.rel_err_l2_trimmed(theirs, want)
        assert e <= max(1e-5, 2 * r) or (et <= max(1e-5, 2 * rt) and e <= 1e-4), (k, e, et, r, rt)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (100, 37, 81, 81, 0), (10, 33, 983, 10, 0),
                                           (10, 20, 983, 983, 0), (10, 16, 38, 38, STABLE)])
def test_unobserved_cells_get_exact_zeros(S, B, L, Z, flags):
    """With only total_loss's cotangent an unobserved cell's logit gradients are exactly 0, and so are the rows of g_R
    of labels unobserved in every row (CUDA-core and tcgen05 products)."""
    t, noise = _inputs(S, B, L, Z, True, seed=11 * S + L, rate=0.3)
    mask = _random_mask(B, L, 0.5, seed=L)
    hidden = torch.arange(L, device=DEV) % 7 == 3
    mask[:, hidden] = False
    _, g = _run(t, noise, _args(S, L, Z, flags | SANITIZE), mask=mask)
    for k in ("fe_out", "fx_out"):
        assert torch.equal(g[k][~mask], torch.zeros_like(g[k][~mask])), k
        assert bool(torch.isfinite(g[k]).all()), k
    assert torch.equal(g["r_sqrt_sigma"][hidden], torch.zeros_like(g["r_sqrt_sigma"][hidden]))
    assert bool((g["r_sqrt_sigma"][~hidden] != 0).any())


# the ALL_OBSERVED cases of test_predict_conditional_gpu, where -log_evidence of a one-row batch is already nll_loss_x
TIE_CASES = [(10, 9, 983, 10, 0, False), (3, 5, 3993, 10, 0, True), (10, 6, 983, 983, TENSOR, False),
             (128, 4, 300, 256, 0, False), (100, 8, 81, 81, 0, False), (10, 7, 38, 38, 0, True),
             (10, 6, 257, 300, STABLE, False), (10, 5, 38, 38, STABLE, True)]


@pytest.mark.parametrize("S,B,L,Z,flags,external", TIE_CASES)
def test_one_row_masked_nll_x_is_the_conditional_log_evidence(S, B, L, Z, flags, external):
    from mpvae_b200.mpvae import compute_loss, predict_conditional
    t, noise = _inputs(S, B, L, Z, external, seed=5 * S + L)
    mask = _random_mask(B, L, 0.4, seed=S + L)
    mask[0] = False
    observed = torch.where(mask, t["y"].to(torch.int8), torch.full_like(t["y"], -1, dtype=torch.int8))
    for b in range(B):
        rows = {k: (v if k == "r_sqrt_sigma" else v[b:b + 1]) for k, v in t.items()}
        a1 = _args(S, L, Z, flags, mode="test", dp_global_batch=B, dp_row0=b)
        nz = noise[:, b:b + 1] if noise is not None else None
        with torch.no_grad():
            nll_x = compute_loss(rows["y"], rows["fe_out"], rows["fe_mu"], rows["fe_logvar"], rows["fx_out"], rows["fx_mu"],
                                 rows["fx_logvar"], rows["r_sqrt_sigma"], a1, noise=nz, label_mask=mask[b:b + 1])[2]
            one = predict_conditional(rows["fx_out"], rows["r_sqrt_sigma"], observed[b:b + 1], a1, noise=nz)
        assert torch.equal(-one.log_evidence[0], nll_x), (b, float(-one.log_evidence[0]), float(nll_x))


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 20, 983, 983, 0),
                                           (10, 20, 983, 983, TENSOR), (10, 16, 38, 38, STABLE)])
def test_degenerate_rows(S, B, L, Z, flags):
    """Row 0 has nothing observed, row 1 only observed negatives, row 2 only observed positives.  Without SANITIZE:
    row 0's gradients are finite, rows 1 and 2 have NaN exactly on their observed cells, every other row and g_R's
    finiteness follow the unmasked rules (NaN from the degenerate rows).  With SANITIZE nothing is NaN.  Both
    contribute 0 to the ranking losses."""
    t, noise = _inputs(S, B, L, Z, True, seed=13 * L + S, rate=0.3)
    y = t["y"]
    y[:, 0], y[:, 1] = 1.0, 0.0
    mask = _random_mask(B, L, 0.5, seed=5)
    mask[:, :2] = True
    mask[0] = False
    mask[1] = (y[1] == 0) & mask[1]
    mask[2] = (y[2] == 1) & mask[2]
    out, g = _run(t, noise, _args(S, L, Z, flags), mask=mask)
    assert all(bool(torch.isfinite(o).all()) for o in out)
    for k in ("fe_out", "fx_out"):
        nan = torch.isnan(g[k])
        want = torch.zeros_like(nan)
        want[1], want[2] = mask[1], mask[2]
        assert torch.equal(nan, want), k
    out_s, g_s = _run(t, noise, _args(S, L, Z, flags | SANITIZE), mask=mask)
    for i in range(8):
        assert torch.equal(out_s[i], out[i]), i
    for k in LEAVES:
        assert bool(torch.isfinite(g_s[k]).all()), k
    # only row 0 degenerate (nothing observed): every gradient finite without SANITIZE, g_R included
    t2 = {k: (v if k == "r_sqrt_sigma" else v[[0, 3, 4, 5]]) for k, v in t.items()}
    m2 = mask[[0, 3, 4, 5]]
    _, g2 = _run(t2, noise[:, [0, 3, 4, 5]], _args(S, L, Z, flags), mask=m2)
    for k in LEAVES:
        assert bool(torch.isfinite(g2[k]).all()), k


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 70, 983, 983, 0),
                                           (100, 37, 81, 81, STABLE)])
def test_repeatable_and_independent_of_workspace_contents(S, B, L, Z, flags, monkeypatch):
    t, noise = _inputs(S, B, L, Z, False, seed=S * L)
    mask = _random_mask(B, L, 0.3, seed=1)
    args = _args(S, L, Z, flags)
    o0, g0 = _run(t, noise, args, mask=mask)
    o1, g1 = _run(t, noise, args, mask=mask)
    monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
    o2, g2 = _run(t, noise, args, mask=mask)
    for o in (o1, o2):
        for i in range(8):
            assert _bits(o0[i], o[i]), i
    for g in (g1, g2):
        for k in LEAVES:
            assert _bits(g0[k], g[k]), k


# ---- a planted model: half of the training labels hidden ----

def _vae_args(F, L, Z, S, c_coeff=10.0, flags=0):
    return SimpleNamespace(feature_dim=F, label_dim=L, latent_dim=16, z_dim=Z, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=S, n_test_sample=S, mode="train", nll_coeff=0.5,
                           c_coeff=c_coeff, batch_size=128, noise_seed=99, mpvae_flags=flags)


def _planted(n, F, L, Z, seed):
    """Correlated labels from a probit model: y_l = 1[x . W_l + b_l + (R eps)_l + e_l > 0], eps ~ N(0, I_Z), e ~ N(0, 1)."""
    g = torch.Generator().manual_seed(seed)
    W = torch.randn(F, L, generator=g) * 0.6 / np.sqrt(F) * 3
    b = torch.randn(L, generator=g) * 0.5 - 0.3
    R = torch.randn(L, 3, generator=g)
    R = torch.cat([R, torch.zeros(L, Z - 3)], 1) * 0.9
    x = torch.randn(n, F, generator=g)
    eps = torch.randn(n, Z, generator=g)
    y = ((x @ W + b + eps @ R.T + torch.randn(n, L, generator=g)) > 0).float()
    return x.to(DEV), y.to(DEV)


def _train(x, y, mask, args, epochs):
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    torch.manual_seed(0)
    np.random.seed(0)
    model = VAE(args).to(DEV)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
    step = DataParallelStep(model, opt, None, args, clip_norm=100.0)
    for ep in range(epochs):
        order = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(ep)).to(DEV)
        train_one_epoch(step, x, y, args.batch_size, order=order, masks=mask)
    return model


def _cell_logloss(model, x, y, args):
    from mpvae_b200.mpvae import predict_exact
    model.eval()
    with torch.no_grad():
        p = predict_exact(model.feat_forward(x)[0], model.r_sqrt_sigma, args).double().clamp(1e-7, 1 - 1e-7)
    yd = y.double()
    return -(yd * torch.log(p) + (1 - yd) * torch.log(1 - p)).flatten()


def test_planted_model_masked_training_beats_zero_filling():
    """Yeast-sized problem (F = 103, L = 14), 50 % of the training labels hidden.  On held-out fully labelled rows the
    per-cell log-loss of predict_exact of the model trained with the mask beats the model trained on hidden labels
    written as 0 by more than 5 standard errors of the paired per-cell difference."""
    F, L, Z, S = 103, 14, 14, 10
    # SANITIZE: zero-filling leaves rows without a positive (degenerate, NaN gradients otherwise); a small ranking weight
    # keeps the comparison about the likelihood
    args = _vae_args(F, L, Z, S, c_coeff=0.1, flags=SANITIZE)
    x, y = _planted(6000, F, L, Z, seed=3)
    xt, yt, xv, yv = x[:4000], y[:4000], x[4000:], y[4000:]
    hide = torch.rand(yt.shape, generator=torch.Generator().manual_seed(8)).to(DEV) < 0.5
    mask = ~hide
    y_zero = torch.where(mask, yt, torch.zeros_like(yt))
    epochs = 25
    masked = _train(xt, y_zero, mask, args, epochs)
    zeroed = _train(xt, y_zero, None, args, epochs)
    full = _train(xt, yt, None, args, epochs)
    a_args = copy.copy(args)
    a_args.mode = "test"
    lm, lz, lf = (_cell_logloss(m, xv, yv, a_args) for m in (masked, zeroed, full))
    d = lz - lm
    se = float(d.std() / np.sqrt(d.numel()))
    print(f"[planted] per-cell log-loss: masked {float(lm.mean()):.4f}  zero-filled {float(lz.mean()):.4f}  "
          f"fully labelled {float(lf.mean()):.4f}  (difference {float(d.mean()):.4f} +- {se:.4f})")
    assert float(d.mean()) > 5 * se, (float(d.mean()), se)


def test_one_gpu_data_parallel_step_equals_the_hand_loop():
    """DataParallelStep with a mask on one GPU == compute_loss(label_mask=) + backward + clip + Adam, bit for bit."""
    from mpvae_b200.mpvae import VAE, compute_loss
    from mpvae_b200.train import DataParallelStep
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    x, y = _planted(64, F, L, Z, seed=5)
    mask = _random_mask(64, L, 0.5, seed=2)
    y = torch.where(mask, y, torch.zeros_like(y))

    def build():
        torch.manual_seed(0)
        np.random.seed(0)
        m = VAE(args).to(DEV)
        return m, torch.optim.Adam(m.parameters(), lr=1e-3)

    m1, o1 = build()
    step = DataParallelStep(m1, o1, None, args, clip_norm=100.0)
    m2, o2 = build()
    a2 = copy.copy(args)
    for i in range(3):
        torch.manual_seed(100 + i)
        step.step(y, x, label_mask=mask)
        torch.manual_seed(100 + i)
        a2.noise_offset = i
        o2.zero_grad()
        out = m2(y, x)
        loss = compute_loss(y, *out, m2.r_sqrt_sigma, a2, label_mask=mask)
        loss[0].backward()
        torch.nn.utils.clip_grad_norm_([p for p in m2.parameters() if p.grad is not None], 100.0)
        o2.step()
    torch.cuda.synchronize()
    for (k, p1), (_, p2) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(p1, p2), k
