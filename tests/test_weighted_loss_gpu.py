"""GPU: weighted training (compute_loss(..., row_weight=) -> mpvae_probit_forward_weighted / _backward_weighted).  All-ones
weights against row_weight=None (bits, with and without a mask), the weighted oracle (positive,
zero and negative weights, a mask, cotangents on all 8 outputs), duplicated rows, zero-weight rows, a large weight in
the tensor regime, predictions, repeatability, DataParallelStep and GraphedTrainStep, and a planted model with noisy
rows down-weighted."""
import copy

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import weighted_elbo_oracle as WO
from tests.test_masked_loss_gpu import (ALL_ONES_CASES, DEV, LEAVES, ORACLE_CASES, SANITIZE, STABLE, TENSOR, _args,
                                        _bits, _inputs, _planted, _random_mask, _vae_args)

pytestmark = pytest.mark.gpu
# the planted model with noisy rows: every model is near its best held-out log-loss at 6 epochs; longer training
# overfits all three and, from about 15 epochs, the down-weighted model (fewer effective rows) first (DESIGN §5)
EPOCHS_NOISY_ROWS = 6


def _run(t, noise, args, weight=None, mask=None, upstream=None):
    """(8 outputs, {leaf: gradient}) of compute_loss + backward (default cotangent: total_loss)."""
    from mpvae_b200.mpvae import compute_loss
    leaves = {k: t[k].detach().clone().requires_grad_(True) for k in LEAVES}
    kw = {}
    if mask is not None:
        kw["label_mask"] = mask
    if weight is not None:
        kw["row_weight"] = weight
    out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, noise=noise, **kw)
    if upstream is None:
        out[0].backward()
    else:
        torch.autograd.backward([out[i] for i in upstream], [upstream[i] for i in upstream])
    torch.cuda.synchronize()
    return [o.detach() for o in out], {k: leaves[k].grad for k in LEAVES}


def _weights(B, kind, seed):
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(B, generator=g) * 2.0 + 0.1
    if kind == "zeros":
        w[torch.rand(B, generator=g) < 0.3] = 0.0
        w[0] = 0.0
    elif kind == "negative":
        w[torch.rand(B, generator=g) < 0.3] *= -1.0
    return w.to(DEV)


@pytest.mark.parametrize("S,B,L,Z,flags,external", ALL_ONES_CASES)
@pytest.mark.parametrize("masked", [False, True])
def test_all_ones_weights_equal_unweighted(S, B, L, Z, flags, external, masked):
    """Training mode and, for the small shapes, test mode: all 8 outputs and every gradient bit for bit, the NaN pattern
    of degenerate rows (two planted: all zeros, all ones) included; with a random mask on both sides too."""
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    t["y"][0] = 0.0
    if B > 1:
        t["y"][1] = 1.0
    mask = _random_mask(B, L, 0.6, seed=B) if masked else None
    ones = torch.ones(B, device=DEV)
    for mode in (("train", "test") if B * L <= 4096 else ("train",)):
        args = _args(S, L, Z, flags, mode)
        o0, g0 = _run(t, noise, args, mask=mask)
        o1, g1 = _run(t, noise, args, weight=ones, mask=mask)
        for i in range(8):
            assert _bits(o0[i], o1[i]), (mode, i)
        for k in LEAVES:
            assert _bits(g0[k], g1[k]), (mode, k)


def _upstream(B, L, seed):
    g = torch.Generator().manual_seed(seed)
    up = {i: (torch.randn((), generator=g) * 0.5 + (1.0 if i == 0 else 0.0)).to(DEV) for i in range(6)}
    up[6] = (torch.randn(B, L, generator=g) * 0.1).to(DEV)
    up[7] = (torch.randn(B, L, generator=g) * 0.1).to(DEV)
    return up


_UP_NAMES = ("total_loss", "nll_loss", "nll_loss_x", "c_loss", "c_loss_x", "kl_loss", "indiv_prob", "indiv_prob_label")


def _check_against_oracle(t, noise, args, w, mask, out, g, upstream=None):
    """The masked tests' bar: losses within 1e-5, predictions within 1e-5 and thresholded decisions identical away from
    ties; gradients against the fp64 oracle by relative L2 <= max(1e-5, 2x the fp32 oracle's own), or the trimmed form
    with <= 1e-4; gradients that are exactly 0 in the oracle exactly 0 here."""
    L = t["y"].shape[1]
    ranking = "factorised" if L > 128 else "pairwise"
    up = None if upstream is None else {_UP_NAMES[i]: v for i, v in upstream.items()}
    ref, rg32 = WO.weighted_probit_elbo_with_grads(t, noise, args.nll_coeff, args.c_coeff, w, mask, ranking=ranking,
                                                   upstream=up)
    tc = {k: v.cpu() for k, v in t.items()}
    up64 = None if up is None else {k: v.cpu().double() for k, v in up.items()}
    _, rg = WO.weighted_probit_elbo_with_grads(tc, noise.cpu(), args.nll_coeff, args.c_coeff, w.cpu(),
                                               None if mask is None else mask.cpu(), ranking=ranking,
                                               dtype=torch.float64, upstream=up64)
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


def _oracle_inputs(S, B, L, Z, seed, masked):
    """No degenerate row (label 0 and 1 planted and observed): the oracle has no SANITIZE."""
    t, noise = _inputs(S, B, L, Z, True, seed=seed, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    mask = None
    if masked:
        mask = _random_mask(B, L, 0.6, seed=S + B)
        mask[:, :2] = True
    return t, noise, mask


@pytest.mark.parametrize("S,B,L,Z,flags", ORACLE_CASES)
@pytest.mark.parametrize("kind", ["positive", "zeros", "negative"])
def test_against_the_weighted_oracle(S, B, L, Z, flags, kind):
    """With a mask and random cotangents on all 8 outputs."""
    t, noise, mask = _oracle_inputs(S, B, L, Z, 3 * S + L, masked=True)
    w = _weights(B, kind, seed=B + L)
    args = _args(S, L, Z, flags)
    up = _upstream(B, L, seed=S)
    out, g = _run(t, noise, args, weight=w, mask=mask, upstream=up)
    _check_against_oracle(t, noise, args, w, mask, out, g, upstream=up)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 70, 983, 983, 0), (7, 19, 130, 64, TENSOR), (10, 33, 983, 10, 0),
                                           (10, 16, 38, 38, 0)])
def test_large_weight_keeps_g_r_within_the_oracle_bar(S, B, L, Z, flags):
    """One row weighted 1e4: the bound that scales the fp16 operand planes of the tensor-regime g_R product includes the
    weights, so g_R stays within the oracle bar (an unscaled plane would overflow fp16)."""
    t, noise, _ = _oracle_inputs(S, B, L, Z, 5 * S + L, masked=False)
    w = torch.ones(B, device=DEV)
    w[4] = 1.0e4
    args = _args(S, L, Z, flags)
    out, g = _run(t, noise, args, weight=w)
    assert bool(torch.isfinite(g["r_sqrt_sigma"]).all())
    errs = _check_against_oracle(t, noise, args, w, None, out, g)
    print(f"[large weight] S{S} B{B} L{L} Z{Z}: g_R rel L2 {errs['r_sqrt_sigma'][0]:.2e} (fp32 oracle {errs['r_sqrt_sigma'][1]:.2e})")


DUP_CASES = [(10, 16, 38, 38, 0), (100, 37, 81, 81, 0), (10, 33, 983, 10, 0), (10, 70, 983, 983, 0), (7, 19, 130, 64, TENSOR),
             (10, 1024, 3993, 3993, 0)]


@pytest.mark.parametrize("S,B,L,Z,flags", DUP_CASES)
def test_weight_k_equals_k_copies(S, B, L, Z, flags):
    """Row 3 weighted 3, row 5 weighted 2, row 6 weighted 0, against the batch with rows 3 and 5 repeated (row 6 dropped)
    on duplicated external noise: scalars x B agree, each row's gradients (total_loss x B) are the sum over its copies,
    g_R agrees, predictions are bit-equal."""
    t, noise = _inputs(S, B, L, Z, True, seed=2 * S + L)
    counts = torch.ones(B, dtype=torch.long)
    counts[3], counts[5], counts[6] = 3, 2, 0
    idx = torch.repeat_interleave(torch.arange(B), counts).to(DEV)
    Bd = int(counts.sum())
    args = _args(S, L, Z, flags)
    out, g = _run(t, noise, args, weight=counts.float().to(DEV), upstream={0: torch.tensor(float(B), device=DEV)})
    td = {k: (v if k == "r_sqrt_sigma" else v[idx]) for k, v in t.items()}
    outd, gd = _run(td, noise[:, idx], _args(S, L, Z, flags), upstream={0: torch.tensor(float(Bd), device=DEV)})
    for i in range(6):
        a, b = float(out[i]) * B, float(outd[i]) * Bd
        assert abs(a - b) <= 1e-5 * max(1.0, abs(b)), (i, a, b)
    for i in (6, 7):
        assert torch.equal(out[i][idx], outd[i]), i
    errs = {}
    for k in LEAVES:
        want = gd[k] if k == "r_sqrt_sigma" else torch.zeros_like(g[k]).index_add_(0, idx, gd[k])
        errs[k] = H.rel_err_l2(g[k].double().cpu().numpy(), want.double().cpu().numpy())
        assert errs[k] <= (2e-5 if k == "r_sqrt_sigma" else 1e-5), (k, errs[k])
        if k != "r_sqrt_sigma":
            assert torch.equal(g[k][6], torch.zeros_like(g[k][6])), k
    print(f"[duplicates] S{S} B{B} L{L} Z{Z}: rel L2 " + " ".join(f"{k} {v:.1e}" for k, v in errs.items()))


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 20, 983, 983, 0),
                                           (10, 20, 983, 983, TENSOR), (10, 16, 38, 38, STABLE)])
def test_zero_weight_rows(S, B, L, Z, flags):
    """Rows 1 (no positive) and 2 (no negative) are degenerate and weighted 0, without SANITIZE: every gradient is
    finite; their logit gradients are exactly those of a row with nothing observed (the predictions' cotangent alone),
    their KL gradients exactly 0; the loss is that of the batch without them times (B - 2) / B."""
    t, noise = _inputs(S, B, L, Z, True, seed=13 * L + S, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    t["y"][1], t["y"][2] = 0.0, 1.0
    w = torch.ones(B, device=DEV)
    w[1] = w[2] = 0.0
    args = _args(S, L, Z, flags)
    up = _upstream(B, L, seed=7)
    out, g = _run(t, noise, args, weight=w, upstream=up)
    for k in LEAVES:
        assert bool(torch.isfinite(g[k]).all()), k
    hidden = torch.ones(B, L, dtype=torch.bool, device=DEV)
    hidden[1:3] = False
    _, gm = _run(t, noise, args, mask=hidden, upstream=up)
    for k in ("fe_out", "fx_out"):
        assert torch.equal(g[k][1:3], gm[k][1:3]), k
    for k in ("fe_mu", "fe_logvar", "fx_mu", "fx_logvar"):
        assert torch.equal(g[k][1:3], torch.zeros_like(g[k][1:3])), k
    keep = [b for b in range(B) if b not in (1, 2)]
    ts = {k: (v if k == "r_sqrt_sigma" else v[keep]) for k, v in t.items()}
    outs, _ = _run(ts, noise[:, keep], args)
    for i in range(6):
        want = float(outs[i]) * (B - 2) / B
        assert abs(float(out[i]) - want) <= 1e-5 * max(1.0, abs(want)), (i, float(out[i]), want)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 70, 983, 983, 0),
                                           (100, 37, 81, 81, STABLE)])
def test_predictions_independent_of_weights_and_repeatable(S, B, L, Z, flags, monkeypatch):
    t, noise = _inputs(S, B, L, Z, False, seed=S * L)
    w = _weights(B, "zeros", seed=3) * 5.0
    args = _args(S, L, Z, flags)
    o_none, _ = _run(t, noise, args)
    o0, g0 = _run(t, noise, args, weight=w)
    assert torch.equal(o_none[6], o0[6]) and torch.equal(o_none[7], o0[7])
    o1, g1 = _run(t, noise, args, weight=w)
    monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
    o2, g2 = _run(t, noise, args, weight=w)
    for o in (o1, o2):
        for i in range(8):
            assert _bits(o0[i], o[i]), i
    for g in (g1, g2):
        for k in LEAVES:
            assert _bits(g0[k], g[k]), k


def test_refused_weights_consume_no_noise_offset():
    from mpvae_b200 import mpvae
    S, B, L, Z = 10, 16, 38, 38
    t, _ = _inputs(S, B, L, Z, False, seed=1)
    args = _args(S, L, Z)
    del args.noise_offset                                   # the module's own counter
    before = dict(mpvae._state)
    bad = [torch.ones(B, device=DEV, requires_grad=True), torch.ones(B - 1, device=DEV), torch.ones(B),
           torch.ones(B, dtype=torch.int32, device=DEV)]
    for w in bad:
        with pytest.raises((TypeError, ValueError)):
            mpvae.compute_loss(t["y"], *(t[k] for k in LEAVES), args, row_weight=w)
    assert mpvae._state == before


def test_one_gpu_data_parallel_step_and_graphed_step():
    """DataParallelStep with weights (and a mask) on one GPU == compute_loss(row_weight=) + backward + clip + Adam, bit for
    bit; GraphedTrainStep replays with weights that change every step walk the eager step's trajectory."""
    from mpvae_b200.mpvae import VAE, compute_loss
    from mpvae_b200.train import DataParallelStep, GraphedTrainStep
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    x, y = _planted(64, F, L, Z, seed=5)
    mask = _random_mask(64, L, 0.5, seed=2)
    y = torch.where(mask, y, torch.zeros_like(y))
    ws = [_weights(64, "zeros", seed=10 + i) for i in range(5)]

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
        torch.manual_seed(100 + i)
        step.step(y, x, label_mask=mask, row_weight=ws[i])
        torch.manual_seed(100 + i)
        a2.noise_offset = i
        o2.zero_grad()
        out = m2(y, x)
        loss = compute_loss(y, *out, m2.r_sqrt_sigma, a2, label_mask=mask, row_weight=ws[i])
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

    mg, sg = build_g()
    graphed = GraphedTrainStep(sg, warmup=3)
    lg = [float(graphed.step(y, x, row_weight=w).total_loss) for w in ws]
    me, se = build_g()
    le = [float(se.step(y, x, row_weight=w).total_loss) for w in ws]
    for a, b in zip(lg, le):
        assert abs(a - b) <= 2e-4 * abs(b), (lg, le)
    for (n, p), (_, q) in zip(mg.named_parameters(), me.named_parameters()):
        assert torch.allclose(p.double(), q.double(), rtol=1e-3, atol=2e-5), n
    assert len(graphed.graphs) == 1


def _noisy_rows_logloss(epochs):
    """Per-cell held-out log-loss of predict_exact of three models trained on the planted problem whose training rows
    carry, for a random 40 %, the labels of another random row: noisy rows weighted 0.05, all-ones weights, and clean
    rows alone."""
    from mpvae_b200.mpvae import VAE, predict_exact
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    F, L, Z, S = 103, 14, 14, 10
    args = _vae_args(F, L, Z, S, c_coeff=0.1, flags=SANITIZE)
    x, y = _planted(6000, F, L, Z, seed=3)
    xt, yt, xv, yv = x[:4000], y[:4000].clone(), x[4000:], y[4000:]
    g = torch.Generator().manual_seed(8)
    noisy = (torch.rand(4000, generator=g) < 0.4).to(DEV)
    donor = torch.randint(0, 4000, (4000,), generator=g).to(DEV)
    y_noisy = torch.where(noisy[:, None], yt[donor], yt)
    w = torch.where(noisy, 0.05, 1.0).float()

    def train(xs, ys, weights):
        torch.manual_seed(0)
        np.random.seed(0)
        model = VAE(args).to(DEV)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
        step = DataParallelStep(model, opt, None, args, clip_norm=100.0)
        for ep in range(epochs):
            order = torch.randperm(xs.shape[0], generator=torch.Generator().manual_seed(ep)).to(DEV)
            train_one_epoch(step, xs, ys, args.batch_size, order=order, weights=weights)
        return model

    def cell_logloss(model):
        a = copy.copy(args)
        a.mode = "test"
        model.eval()
        with torch.no_grad():
            p = predict_exact(model.feat_forward(xv)[0], model.r_sqrt_sigma, a).double().clamp(1e-7, 1 - 1e-7)
        yd = yv.double()
        return -(yd * torch.log(p) + (1 - yd) * torch.log(1 - p)).flatten()

    return tuple(cell_logloss(m) for m in (train(xt, y_noisy, w), train(xt, y_noisy, None), train(xt[~noisy], yt[~noisy], None)))


def test_planted_model_downweighted_noisy_rows_beat_uniform_weights():
    """Yeast-sized problem (F = 103, L = 14).  The labels of a random 40 % of the training rows are replaced by those of
    another random row; those rows are weighted 0.05.  On held-out clean rows the per-cell log-loss of predict_exact of
    the model trained with the weights beats the model trained with all-ones weights by more than 5 standard errors of
    the paired per-cell difference.  The model trained on the clean rows alone is printed beside them."""
    lw, lu, lc = _noisy_rows_logloss(EPOCHS_NOISY_ROWS)
    d = lu - lw
    se = float(d.std() / np.sqrt(d.numel()))
    print(f"[planted] per-cell log-loss: weighted {float(lw.mean()):.4f}  all-ones {float(lu.mean()):.4f}  "
          f"clean rows only {float(lc.mean()):.4f}  (difference {float(d.mean()):.4f} +- {se:.4f})")
    assert float(d.mean()) > 5 * se, (float(d.mean()), se)


def test_predict_proba_weighted_sums():
    """infer.predict_proba(..., row_weight=): the summed losses are sum_n w_n t_n (all-ones: the unweighted sums), the
    predictions do not change."""
    from mpvae_b200 import infer
    from mpvae_b200.mpvae import VAE
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    args.mode = "test"
    x, y = _planted(300, F, L, Z, seed=9)
    torch.manual_seed(0)
    model = VAE(args).to(DEV).eval()
    res = {}
    for name, w in (("none", None), ("ones", torch.ones(300, device=DEV)), ("twos", torch.full((300,), 2.0, device=DEV))):
        torch.manual_seed(1)
        args.noise_offset = 5
        res[name] = infer.predict_proba(model, x, y, args, batch_size=128, row_weight=w)
    for k in ("total_loss", "nll_loss", "c_loss"):
        assert torch.equal(res["none"][1][k], res["ones"][1][k]), k
        assert torch.equal(res["twos"][1][k], 2.0 * res["none"][1][k]), k
    assert torch.equal(res["none"][0], res["twos"][0])
