"""GPU: label-weighted training (compute_loss(..., pos_weight=, neg_weight=) -> mpvae_probit_forward_label_weighted /
_backward_label_weighted) in every regime: small (yeast / mirflickr shapes), CUDA-core (L = 200, Z = 64), dense tensor
(delicious shape, reduced B) and the stable-CDF backward.  All-ones weights against None (bits, with a mask, row weights,
soft labels), the label-weighted oracle (random, zero, negative weights and a mix with a mask and row
weights), weights of 1e4 and 1e-4 against the g_R bar, zero-weight cells, predictions, repeatability,
DataParallelStep and GraphedTrainStep, and a planted model with rare labels trained with pos_weight."""
import copy

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import label_weighted_elbo_oracle as LO
from tests.test_masked_loss_gpu import (DEV, LEAVES, SANITIZE, STABLE, TENSOR, _args, _bits, _inputs, _random_mask,
                                        _vae_args)
from tests.test_weighted_loss_gpu import _UP_NAMES, _upstream

pytestmark = pytest.mark.gpu

# (S, B, L, Z, flags, external noise): small regime (yeast, mirflickr), CUDA-core (tiled forward + saved backward),
# dense tensor (delicious shape, B reduced; a ragged label tile), the stable-CDF backward (small and dense shapes), SANITIZE
REGIME_CASES = [(10, 16, 14, 14, 0, False), (3, 33, 38, 38, 0, True), (10, 40, 200, 64, 0, False), (7, 21, 200, 64, 0, True),
                (10, 70, 983, 983, 0, False), (3, 19, 983, 983, TENSOR, True), (3, 77, 130, 256, 0, True), (10, 16, 38, 38, STABLE, False),
                (10, 40, 257, 300, STABLE, False), (10, 33, 983, 10, SANITIZE, False)]
ORACLE_CASES = [(10, 16, 38, 38, 0), (1, 5, 14, 14, 0), (10, 20, 200, 64, 0), (10, 20, 983, 983, 0), (7, 19, 130, 64, TENSOR),
                (10, 16, 38, 38, STABLE), (10, 12, 257, 300, STABLE)]


def _run(t, noise, args, pos=None, neg=None, weight=None, mask=None, upstream=None):
    """(8 outputs, {leaf: gradient}) of compute_loss + backward (default cotangent: total_loss)."""
    from mpvae_b200.mpvae import compute_loss
    leaves = {k: t[k].detach().clone().requires_grad_(True) for k in LEAVES}
    kw = {k: v for k, v in (("label_mask", mask), ("row_weight", weight), ("pos_weight", pos), ("neg_weight", neg))
          if v is not None}
    out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, noise=noise, **kw)
    if upstream is None:
        out[0].backward()
    else:
        torch.autograd.backward([out[i] for i in upstream], [upstream[i] for i in upstream])
    torch.cuda.synchronize()
    return [o.detach() for o in out], {k: leaves[k].grad for k in LEAVES}


def _label_weights(L, kind, seed):
    g = torch.Generator().manual_seed(seed)
    pos, neg = torch.rand(L, generator=g) * 4.0 + 0.1, torch.rand(L, generator=g) * 1.5 + 0.1
    if kind in ("zeros", "mixed"):
        pos[torch.rand(L, generator=g) < 0.2] = 0.0
        neg[torch.rand(L, generator=g) < 0.2] = 0.0
        pos[2], neg[3] = 0.0, 0.0
    if kind in ("negative", "mixed"):
        pos[torch.rand(L, generator=g) < 0.2] *= -1.0
        neg[torch.rand(L, generator=g) < 0.2] *= -1.0
    return pos.to(DEV), neg.to(DEV)


@pytest.mark.parametrize("S,B,L,Z,flags,external", REGIME_CASES)
@pytest.mark.parametrize("masked,row_weighted,soft", [(False, False, False), (True, False, False), (False, True, True),
                                                      (True, True, True)])
def test_all_ones_label_weights_equal_none(S, B, L, Z, flags, external, masked, row_weighted, soft):
    """All 8 outputs and every gradient bit for bit, degenerate rows (all zeros, all ones) included, with a mask, row
    weights and soft labels on both sides."""
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    t["y"][0] = 0.0
    t["y"][1] = 1.0
    if soft:
        g = torch.Generator().manual_seed(L)
        t["y"][2:, : L // 3] = torch.rand(B - 2, L // 3, generator=g).to(DEV)
    mask = _random_mask(B, L, 0.6, seed=B) if masked else None
    w = (torch.rand(B, generator=torch.Generator().manual_seed(S)) * 2.0).to(DEV) if row_weighted else None
    ones = torch.ones(L, device=DEV)
    args = _args(S, L, Z, flags)
    o0, g0 = _run(t, noise, args, mask=mask, weight=w)
    for pos, neg in ((ones, ones), (ones, None), (None, ones.double())):
        o1, g1 = _run(t, noise, args, pos=pos, neg=neg, mask=mask, weight=w)
        for i in range(8):
            assert _bits(o0[i], o1[i]), i
        for k in LEAVES:
            assert _bits(g0[k], g1[k]), k


def _check_against_oracle(t, noise, args, lw, w, mask, out, g, upstream=None):
    """The weighted tests' bar: losses within 1e-5, predictions within 1e-5 and thresholded decisions identical away from
    ties; gradients against the fp64 oracle by relative L2 <= max(1e-5, 2x the fp32 oracle's own), or the trimmed form
    with <= 1e-4; gradients that are exactly 0 in the oracle exactly 0 here.  STABLE_CDF does not follow the reference's
    fp32 arithmetic (its E has no cancellation in the tails): its losses and predictions are held to the fp64 oracle."""
    L = t["y"].shape[1]
    ranking = "factorised" if L > 128 else "pairwise"
    up = None if upstream is None else {_UP_NAMES[i]: v for i, v in upstream.items()}
    ref, rg32 = LO.label_weighted_probit_elbo_with_grads(t, noise, args.nll_coeff, args.c_coeff, lw.to(DEV), w, mask,
                                                         ranking=ranking, upstream=up)
    tc = {k: v.cpu() for k, v in t.items()}
    up64 = None if up is None else {k: v.cpu().double() for k, v in up.items()}
    ref64, rg = LO.label_weighted_probit_elbo_with_grads(tc, noise.cpu(), args.nll_coeff, args.c_coeff, lw.cpu(),
                                                     None if w is None else w.cpu(), None if mask is None else mask.cpu(),
                                                     ranking=ranking, dtype=torch.float64, upstream=up64)
    if getattr(args, "mpvae_flags", 0) & STABLE:
        ref = ref64
    for i in range(6):
        want = float(ref[i])
        assert abs(float(out[i]) - want) <= 1e-5 * max(1.0, abs(want)), (i, float(out[i]), want)
    for i in (6, 7):
        got, want = out[i].cpu().numpy(), ref[i].detach().cpu().numpy()
        dp = float(np.max(np.abs(got.astype(np.float64) - want)))
        assert dp <= 1e-5, (i, dp)
        assert H.threshold_mismatches(got, want, tie=2 * dp + 1e-7) == 0
    errs = {}
    for k in LEAVES:
        got, want, theirs = g[k].double().cpu().numpy(), rg[k].numpy(), rg32[k].double().cpu().numpy()
        if not np.any(want):
            assert not np.any(got), k
            continue
        e, et = H.rel_err_l2(got, want), H.rel_err_l2_trimmed(got, want)
        r, rt = H.rel_err_l2(theirs, want), H.rel_err_l2_trimmed(theirs, want)
        errs[k] = (e, r)
        assert e <= max(1e-5, 2 * r) or (et <= max(1e-5, 2 * rt) and e <= 1e-4), (k, e, et, r, rt)
    return errs


def _oracle_inputs(S, B, L, Z, seed):
    """No degenerate row (label 0 and 1 planted): the oracle has no SANITIZE."""
    t, noise = _inputs(S, B, L, Z, True, seed=seed, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    return t, noise


@pytest.mark.parametrize("S,B,L,Z,flags", ORACLE_CASES)
@pytest.mark.parametrize("kind", ["positive", "zeros", "negative", "mixed"])
def test_against_the_label_weighted_oracle(S, B, L, Z, flags, kind):
    """Random cotangents on all 8 outputs; "mixed": zero and negative label weights with a mask and row weights."""
    t, noise = _oracle_inputs(S, B, L, Z, 3 * S + L)
    pos, neg = _label_weights(L, kind, seed=B + L)
    mask = w = None
    if kind == "mixed":
        mask = _random_mask(B, L, 0.7, seed=S + B)
        mask[:, :2] = True
        w = (torch.rand(B, generator=torch.Generator().manual_seed(L)) * 2.0).to(DEV)
        w[1] = 0.0
    args = _args(S, L, Z, flags)
    up = _upstream(B, L, seed=S)
    out, g = _run(t, noise, args, pos=pos, neg=neg, weight=w, mask=mask, upstream=up)
    _check_against_oracle(t, noise, args, torch.stack([neg, pos]), w, mask, out, g, upstream=up)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 70, 983, 983, 0), (7, 19, 130, 64, TENSOR), (10, 20, 200, 64, 0),
                                           (10, 16, 38, 38, 0)])
@pytest.mark.parametrize("scale", [1.0e4, 1.0e-4])
def test_extreme_label_weight_keeps_g_r_within_the_oracle_bar(S, B, L, Z, flags, scale):
    """Label 5 weighted 1e4 (or 1e-4) on both values: the bound that scales the fp16 operand planes of the tensor-regime
    g_R product includes max |w|, so g_R stays within the oracle bar."""
    t, noise = _oracle_inputs(S, B, L, Z, 5 * S + L)
    pos, neg = torch.ones(L, device=DEV), torch.ones(L, device=DEV)
    pos[5] = neg[5] = scale
    args = _args(S, L, Z, flags)
    out, g = _run(t, noise, args, pos=pos, neg=neg)
    assert bool(torch.isfinite(g["r_sqrt_sigma"]).all())
    errs = _check_against_oracle(t, noise, args, torch.stack([neg, pos]), None, None, out, g)
    print(f"[label weight {scale:g}] S{S} B{B} L{L} Z{Z}: g_R rel L2 {errs['r_sqrt_sigma'][0]:.2e} "
          f"(fp32 oracle {errs['r_sqrt_sigma'][1]:.2e})")


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 20, 200, 64, 0), (10, 20, 983, 983, 0),
                                           (10, 16, 38, 38, STABLE), (10, 12, 257, 300, STABLE)])
def test_zero_weight_cells_get_the_ranking_and_prediction_gradient(S, B, L, Z, flags):
    """Labels 2 and 3 weighted 0 on both values: their logit gradients are bit for bit those of the same call with
    cotangents on the ranking losses and the predictions alone (no log-likelihood cotangent), and within the oracle
    bar."""
    t, noise = _oracle_inputs(S, B, L, Z, 7 * S + L)
    pos, neg = _label_weights(L, "positive", seed=L)
    pos[2:4] = neg[2:4] = 0.0
    args = _args(S, L, Z, flags)
    up = _upstream(B, L, seed=11)
    up.pop(0)
    out, g = _run(t, noise, args, pos=pos, neg=neg, upstream=up)
    _check_against_oracle(t, noise, args, torch.stack([neg, pos]), None, None, out, g, upstream=up)
    rank_only = {i: v for i, v in up.items() if i in (3, 4, 6, 7)}
    _, gr = _run(t, noise, args, pos=pos, neg=neg, upstream=rank_only)
    for k in ("fe_out", "fx_out"):
        assert torch.equal(g[k][:, 2:4], gr[k][:, 2:4]), k


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 40, 200, 64, 0), (10, 70, 983, 983, 0),
                                           (100, 37, 81, 81, STABLE)])
def test_predictions_independent_of_label_weights_and_repeatable(S, B, L, Z, flags, monkeypatch):
    t, noise = _inputs(S, B, L, Z, False, seed=S * L)
    pos, neg = _label_weights(L, "mixed", seed=3)
    args = _args(S, L, Z, flags)
    o_none, _ = _run(t, noise, args)
    o0, g0 = _run(t, noise, args, pos=pos, neg=neg)
    assert torch.equal(o_none[6], o0[6]) and torch.equal(o_none[7], o0[7])
    assert torch.equal(o_none[3], o0[3]) and torch.equal(o_none[4], o0[4]) and torch.equal(o_none[5], o0[5])
    o1, g1 = _run(t, noise, args, pos=pos, neg=neg)
    monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
    o2, g2 = _run(t, noise, args, pos=pos, neg=neg)
    for o in (o1, o2):
        for i in range(8):
            assert _bits(o0[i], o[i]), i
    for gg in (g1, g2):
        for k in LEAVES:
            assert _bits(g0[k], gg[k]), k


def test_refused_label_weights_consume_no_noise_offset():
    from mpvae_b200 import mpvae
    S, B, L, Z = 10, 16, 38, 38
    t, _ = _inputs(S, B, L, Z, False, seed=1)
    args = _args(S, L, Z)
    del args.noise_offset                                   # the module's own counter
    before = dict(mpvae._state)
    bad = [torch.ones(L, device=DEV, requires_grad=True), torch.ones(L - 1, device=DEV), torch.ones(L),
           torch.ones(L, dtype=torch.int32, device=DEV)]
    for w in bad:
        for name in ("pos_weight", "neg_weight"):
            with pytest.raises((TypeError, ValueError)):
                mpvae.compute_loss(t["y"], *(t[k] for k in LEAVES), args, **{name: w})
    assert mpvae._state == before


def test_one_gpu_data_parallel_step_and_graphed_step():
    """DataParallelStep with label weights (a mask and row weights too) on one GPU == compute_loss + backward + clip +
    Adam, bit for bit; GraphedTrainStep with label weights, and with a label mask, walks the eager step's trajectory."""
    from mpvae_b200.mpvae import VAE, compute_loss
    from mpvae_b200.train import DataParallelStep, GraphedTrainStep
    from tests.test_masked_loss_gpu import _planted
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    x, y = _planted(64, F, L, Z, seed=5)
    mask = _random_mask(64, L, 0.5, seed=2)
    y = torch.where(mask, y, torch.zeros_like(y))
    lws = [_label_weights(L, "zeros", seed=10 + i) for i in range(5)]
    w = (torch.rand(64, generator=torch.Generator().manual_seed(1)) * 2.0).to(DEV)

    def build(capturable=False):
        torch.manual_seed(0)
        np.random.seed(0)
        m = VAE(args).to(DEV)
        lr = torch.tensor(1e-3, device=DEV) if capturable else 1e-3
        return m, torch.optim.Adam(m.parameters(), lr=lr, capturable=capturable)

    m1, o1 = build()
    step = DataParallelStep(m1, o1, None, args, clip_norm=100.0)
    m2, o2 = build()
    a2 = copy.copy(args)
    for i in range(3):
        pos, neg = lws[i]
        torch.manual_seed(100 + i)
        step.step(y, x, label_mask=mask, row_weight=w, pos_weight=pos, neg_weight=neg)
        torch.manual_seed(100 + i)
        a2.noise_offset = i
        o2.zero_grad()
        out = m2(y, x)
        loss = compute_loss(y, *out, m2.r_sqrt_sigma, a2, label_mask=mask, row_weight=w, pos_weight=pos, neg_weight=neg)
        loss[0].backward()
        torch.nn.utils.clip_grad_norm_([p for p in m2.parameters() if p.grad is not None], 100.0)
        o2.step()
    torch.cuda.synchronize()
    for (k, p1), (_, p2) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(p1, p2), k

    # graph replay: no dropout, collapsed posteriors (host-visible randomness removed, as test_train_gpu does)
    gargs = _vae_args(F, L, Z, S)
    gargs.noise_seed = 77

    def build_g():
        m, o = build(capturable=True)
        with torch.no_grad():
            for head in (m.fe_logvar, m.fx_logvar):
                head.weight.zero_(); head.bias.fill_(-30.0)
        return m, DataParallelStep(m, o, None, copy.copy(gargs), clip_norm=100.0)

    # every row keeps an observed positive and negative under the masks: no degenerate row, no NaN gradient
    y = y.clone()
    y[:, 0], y[:, 1] = 1.0, 0.0
    masks = [_random_mask(64, L, 0.5, seed=20 + i) for i in range(5)]
    for m in masks:
        m[:, :2] = True
    for kws in ([{"pos_weight": p, "neg_weight": n} for p, n in lws], [{"label_mask": m} for m in masks]):
        mg, sg = build_g()
        graphed = GraphedTrainStep(sg, warmup=3)
        lg = [float(graphed.step(y, x, **kw).total_loss) for kw in kws]
        me, se = build_g()
        le = [float(se.step(y, x, **kw).total_loss) for kw in kws]
        for a, b in zip(lg, le):
            assert abs(a - b) <= 2e-4 * abs(b), (lg, le)
        for (n, p), (_, q) in zip(mg.named_parameters(), me.named_parameters()):
            assert torch.allclose(p.double(), q.double(), rtol=1e-3, atol=2e-5), n
        assert len(graphed.graphs) == 1


def test_predict_proba_label_weighted_sums():
    """infer.predict_proba(..., pos_weight=, neg_weight=): all-ones weights give the unweighted sums, pos_weight = 2 and
    neg_weight = 2 twice the nll sums; the ranking sums and the predictions do not change."""
    from mpvae_b200 import infer
    from mpvae_b200.mpvae import VAE
    from tests.test_masked_loss_gpu import _planted
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    args.mode = "test"
    x, y = _planted(300, F, L, Z, seed=9)
    torch.manual_seed(0)
    model = VAE(args).to(DEV).eval()
    res = {}
    ones, twos = torch.ones(L, device=DEV), torch.full((L,), 2.0, device=DEV)
    for name, kw in (("none", {}), ("ones", {"pos_weight": ones, "neg_weight": ones}), ("pos2", {"pos_weight": twos})):
        torch.manual_seed(1)
        args.noise_offset = 5
        res[name] = infer.predict_proba(model, x, y, args, batch_size=128, **kw)
    for k in res["none"][1]:
        assert torch.equal(res["none"][1][k], res["ones"][1][k]), k
    assert torch.equal(res["none"][1]["c_loss"], res["pos2"][1]["c_loss"])
    assert not torch.equal(res["none"][1]["nll_loss"], res["pos2"][1]["nll_loss"])
    assert torch.equal(res["none"][0], res["pos2"][0])


# ---- planted model with rare labels ----
RARE = (3, 7, 11)
EPOCHS_RARE = 12


def _planted_rare(n, F, L, Z, seed):
    """The probit model of test_masked_loss_gpu._planted with the biases of labels RARE lowered to about 2 % positives."""
    g = torch.Generator().manual_seed(seed)
    W = torch.randn(F, L, generator=g) * 0.6 / np.sqrt(F) * 3
    b = torch.randn(L, generator=g) * 0.5 - 0.3
    b[list(RARE)] = -4.7
    R = torch.randn(L, 3, generator=g)
    R = torch.cat([R, torch.zeros(L, Z - 3)], 1) * 0.9
    x = torch.randn(n, F, generator=g)
    eps = torch.randn(n, Z, generator=g)
    y = ((x @ W + b + eps @ R.T + torch.randn(n, L, generator=g)) > 0).float()
    return x.to(DEV), y.to(DEV)


def _rare_f1(epochs):
    """Held-out F1 at threshold 0.5 (predict_exact) of the rare labels, per label and pooled, for a model trained without
    label weights and one with pos_weight = n_neg / n_pos (clamped to [1, 50]) on the rare labels; plus per-row
    contributions for a bootstrap standard error."""
    from mpvae_b200.mpvae import VAE, predict_exact
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    F, L, Z, S = 103, 14, 14, 10
    args = _vae_args(F, L, Z, S, c_coeff=0.1, flags=SANITIZE)
    x, y = _planted_rare(12000, F, L, Z, seed=3)
    xt, yt, xv, yv = x[:8000], y[:8000], x[8000:], y[8000:]
    n_pos = yt.sum(0)
    pos_weight = torch.ones(L, device=DEV)
    rare = list(RARE)
    pos_weight[rare] = ((yt.shape[0] - n_pos[rare]) / n_pos[rare].clamp(min=1.0)).clamp(1.0, 50.0)

    def train(pw):
        torch.manual_seed(0)
        np.random.seed(0)
        model = VAE(args).to(DEV)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
        step = DataParallelStep(model, opt, None, args, clip_norm=100.0)
        for ep in range(epochs):
            order = torch.randperm(xt.shape[0], generator=torch.Generator().manual_seed(ep)).to(DEV)
            train_one_epoch(step, xt, yt, args.batch_size, order=order, pos_weight=pw)
        a = copy.copy(args)
        a.mode = "test"
        model.eval()
        with torch.no_grad():
            p = predict_exact(model.feat_forward(xv)[0], model.r_sqrt_sigma, a)
        return (p[:, rare] >= 0.5).double()

    yr = yv[:, rare].double()
    return yr, train(None), train(pos_weight), pos_weight[rare]


def _f1(yr, pred):
    tp = (pred * yr).sum(0)
    return 2 * tp / (pred.sum(0) + yr.sum(0)).clamp(min=1.0)


def test_planted_model_pos_weight_raises_rare_label_f1():
    """Yeast-sized problem (F = 103, L = 14) with labels 3, 7 and 11 at about 2 % positives.  Trained with pos_weight =
    n_neg / n_pos (clamped to 50) on those labels, the held-out F1 at threshold 0.5 of each rare label, and their mean,
    beats the model trained without label weights; the mean gain exceeds 3 bootstrap standard errors (fixed seeds)."""
    yr, p0, p1, pw = _rare_f1(EPOCHS_RARE)
    f0, f1 = _f1(yr, p0), _f1(yr, p1)
    g = torch.Generator().manual_seed(0)
    n = yr.shape[0]
    boot = []
    for _ in range(200):
        idx = torch.randint(0, n, (n,), generator=g).to(DEV)
        boot.append(float((_f1(yr[idx], p1[idx]) - _f1(yr[idx], p0[idx])).mean()))
    se = float(np.std(boot))
    gain = float((f1 - f0).mean())
    print(f"[planted rare labels] positive rate {[round(float(v), 4) for v in yr.mean(0)]}  pos_weight "
          f"{[round(float(v), 1) for v in pw]}  F1 without {[round(float(v), 3) for v in f0]} (mean {float(f0.mean()):.3f})  "
          f"with {[round(float(v), 3) for v in f1]} (mean {float(f1.mean()):.3f})  gain {gain:.3f} +- {se:.3f}")
    assert bool((f1 > f0).all()), (f0, f1)
    assert gain > 3 * se, (gain, se)
