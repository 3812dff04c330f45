"""GPU: per-row losses (compute_loss(..., reduction='none') -> mpvae_probit_forward_rows / _backward_rows).  B = 1 against
'mean' (bits, with mask, row weights and label weights), predictions against 'mean', nll_x against the conditional log
evidence row by row, a cotangent on one row against a one-row 'mean' call, row weights, the per-row fp64 oracle with
random cotangents, a large cotangent in the tensor regime, degenerate rows left out by indexing, repeatability,
DataParallelStep(row_objective=), infer.predict_proba(reduction='none'), and a planted model with noisy rows: their
detection by per-row nll_x and small-loss training."""
import copy

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import row_elbo_oracle as RO
from tests.test_masked_loss_gpu import (ALL_ONES_CASES, DEV, FMA, LEAVES, SANITIZE, STABLE, TENSOR, TIE_CASES, _args,
                                        _bits, _inputs, _planted, _random_mask, _vae_args)

pytestmark = pytest.mark.gpu


def _run(t, noise, args, reduction="mean", upstream=None, **kw):
    """(8 outputs, {leaf: gradient}) of compute_loss + backward; upstream {output index: cotangent} (default: total_loss,
    ones per row for 'none')."""
    from mpvae_b200.mpvae import compute_loss
    leaves = {k: t[k].detach().clone().requires_grad_(True) for k in LEAVES}
    out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, noise=noise, reduction=reduction, **kw)
    if upstream is None:
        upstream = {0: torch.ones_like(out[0])}
    torch.autograd.backward([out[i] for i in upstream], [upstream[i] for i in upstream])
    torch.cuda.synchronize()
    return [o.detach() for o in out], {k: leaves[k].grad for k in LEAVES}


def _options(B, L, kind, seed):
    g = torch.Generator().manual_seed(seed)
    kw = {}
    if kind in ("mask", "all"):
        kw["label_mask"] = _random_mask(B, L, 0.6, seed=seed)
    if kind in ("row_weight", "all"):
        kw["row_weight"] = (torch.rand(B, generator=g) * 2.0 + 0.1).to(DEV)
    if kind in ("label_weight", "all"):
        kw["pos_weight"] = (torch.rand(L, generator=g) * 3.0 + 0.2).to(DEV)
        kw["neg_weight"] = (torch.rand(L, generator=g) * 1.5 + 0.2).to(DEV)
    return kw


# one row in every regime: small, CUDA-core (FMA, and Z < 128), dense tensor, stable CDF
B1_CASES = [(10, 1, 38, 38, 0, False), (1, 1, 14, 14, 0, True), (100, 1, 81, 81, 0, False), (10, 1, 983, 10, 0, False),
            (3, 1, 3993, 10, 0, True), (10, 1, 983, 983, FMA, False), (10, 1, 983, 983, TENSOR, False),
            (7, 1, 130, 64, TENSOR, True), (128, 1, 300, 256, 0, False), (10, 1, 38, 38, STABLE, False),
            (10, 1, 257, 300, STABLE, True), (10, 1, 38, 38, SANITIZE, False)]


@pytest.mark.parametrize("S,B,L,Z,flags,external", B1_CASES)
@pytest.mark.parametrize("kind", ["plain", "mask", "row_weight", "label_weight", "all"])
def test_one_row_none_equals_mean(S, B, L, Z, flags, external, kind):
    """B = 1, train and test mode, random cotangents on all 8 outputs: 'none' gives the bits of 'mean' on every output
    and gradient."""
    t, noise = _inputs(S, B, L, Z, external, seed=S + L + Z)
    kw = _options(B, L, kind, seed=L)
    g = torch.Generator().manual_seed(S)
    up = {i: (torch.randn((), generator=g) * 0.5 + (1.0 if i == 0 else 0.0)).to(DEV) for i in range(6)}
    up[6] = (torch.randn(B, L, generator=g) * 0.1).to(DEV)
    up[7] = (torch.randn(B, L, generator=g) * 0.1).to(DEV)
    for mode in ("train", "test"):
        args = _args(S, L, Z, flags, mode)
        o0, g0 = _run(t, noise, args, upstream=up, **kw)
        o1, g1 = _run(t, noise, args, "none", upstream={i: (v.reshape(1) if i < 6 else v) for i, v in up.items()}, **kw)
        for i in range(6):
            assert o1[i].shape == (1,) and _bits(o0[i], o1[i][0]), (mode, i, float(o0[i]), float(o1[i][0]))
        for i in (6, 7):
            assert _bits(o0[i], o1[i]), (mode, i)
        for k in LEAVES:
            assert _bits(g0[k], g1[k]), (mode, k)


@pytest.mark.parametrize("S,B,L,Z,flags,external", ALL_ONES_CASES)
def test_predictions_are_the_mean_bits_and_rows_average_to_the_means(S, B, L, Z, flags, external):
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    kw = _options(B, L, "all", seed=B)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        from mpvae_b200.mpvae import compute_loss
        o0 = compute_loss(t["y"], *(t[k] for k in LEAVES), args, noise=noise, **kw)
        o1 = compute_loss(t["y"], *(t[k] for k in LEAVES), args, noise=noise, reduction="none", **kw)
    torch.cuda.synchronize()
    for i in (6, 7):
        assert _bits(o0[i], o1[i]), i
    for i in range(6):
        assert o1[i].shape == (B,)
        got, want = float(o1[i].double().mean()), float(o0[i])
        assert abs(got - want) <= 1e-5 * max(1.0, abs(want)) or (np.isnan(want) and np.isnan(got)), (i, got, want)


@pytest.mark.parametrize("S,B,L,Z,flags,external", TIE_CASES)
@pytest.mark.parametrize("masked", [False, True])
def test_nll_x_is_the_conditional_log_evidence_row_by_row(S, B, L, Z, flags, external, masked):
    """Test mode, the same noise: nll_x_b = -predict_conditional(observed).log_evidence[b] for every row of the batch,
    observed = y (or y where the mask is set, -1 elsewhere)."""
    from mpvae_b200.mpvae import compute_loss, predict_conditional
    t, noise = _inputs(S, B, L, Z, external, seed=5 * S + L)
    args = _args(S, L, Z, flags, mode="test")
    y8 = t["y"].to(torch.int8)
    kw = {}
    if masked:
        kw["label_mask"] = mask = _random_mask(B, L, 0.4, seed=S + L)
        y8 = torch.where(mask, y8, torch.full_like(y8, -1))
    with torch.no_grad():
        nll_x = compute_loss(t["y"], *(t[k] for k in LEAVES), args, noise=noise, reduction="none", **kw)[2]
        ev = predict_conditional(t["fx_out"], t["r_sqrt_sigma"], y8, args, noise=noise).log_evidence
    assert torch.equal(-ev, nll_x), (-ev - nll_x).abs().max()


# small, CUDA-core (Z < 128; forced FMA), dense tensor (forced, so that one row takes the same product), stable CDF
ONE_ROW_CASES = [(10, 16, 38, 38, 0, "small"), (10, 33, 983, 10, 0, "cuda-core"), (10, 20, 983, 983, FMA, "cuda-core"),
                 (10, 20, 983, 983, TENSOR, "tensor"), (7, 19, 130, 64, TENSOR, "tensor"), (10, 16, 38, 38, STABLE, "stable")]


@pytest.mark.parametrize("S,B,L,Z,flags,regime", ONE_ROW_CASES)
@pytest.mark.parametrize("term", [0, 1, 2, 3, 4, 5])
def test_a_cotangent_on_one_row_is_that_row_alone(S, B, L, Z, flags, regime, term):
    """A cotangent on row b of one output: row b's logit and latent gradients equal those of a 'mean' call on row b
    alone with the same Philox keys, bit for bit; every other row's are exactly 0; g_R bit-equal in the small regime,
    within the fp64 oracle's bar elsewhere (a different M splits the g_R product differently)."""
    t, _ = _inputs(S, B, L, Z, False, seed=7 * S + L, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    b = 3
    for mode in ("train", "test"):
        args = _args(S, L, Z, flags, mode, dp_global_batch=B, dp_row0=0)
        g = torch.zeros(B, device=DEV)
        g[b] = 0.75
        out, grads = _run(t, None, args, "none", upstream={term: g})
        row = {k: (v if k == "r_sqrt_sigma" else v[b:b + 1]) for k, v in t.items()}
        o1, g1 = _run(row, None, _args(S, L, Z, flags, mode, dp_global_batch=B, dp_row0=b),
                      upstream={term: torch.tensor(0.75, device=DEV)})
        assert _bits(out[term][b], o1[term]), (mode, float(out[term][b]), float(o1[term]))
        others = torch.arange(B, device=DEV) != b
        for k in LEAVES[:-1]:
            assert _bits(grads[k][b:b + 1], g1[k]), (mode, k)
            assert not bool(grads[k][others].any()), (mode, k)
        gr, gr1 = grads["r_sqrt_sigma"], g1["r_sqrt_sigma"]
        same = _bits(gr, gr1)
        err = H.rel_err_l2(gr.double().cpu().numpy(), gr1.double().cpu().numpy())
        print(f"[one row] {regime} S{S} B{B} L{L} Z{Z} term {term} {mode}: g_R bit-equal {same}, rel L2 {err:.2e}")
        if regime == "small":
            assert same, (mode, err)
        else:
            assert err <= 2e-5, (mode, err)


def test_row_weights_scale_the_rows():
    """'none' with row weights: w_b * t_b (fp64 product of the fp32 terms, within one rounding), all-ones weights give
    the unweighted bits, zero-weight rows exactly 0 on all six even when degenerate."""
    S, B, L, Z = 10, 16, 38, 38
    for flags in (0, FMA, STABLE):
        t, noise = _inputs(S, B, L, Z, True, seed=11 + flags)
        t["y"][2] = 0.0
        args = _args(S, L, Z, flags)
        w = (torch.rand(B, generator=torch.Generator().manual_seed(4)) * 3.0).to(DEV)
        w[[2, 5]] = 0.0
        o_none, _ = _run(t, noise, args, "none", upstream={0: torch.zeros(B, device=DEV)})
        o_ones, _ = _run(t, noise, args, "none", upstream={0: torch.zeros(B, device=DEV)}, row_weight=torch.ones(B, device=DEV))
        o_w, _ = _run(t, noise, args, "none", upstream={0: torch.zeros(B, device=DEV)}, row_weight=w)
        for i in range(8):
            assert _bits(o_none[i], o_ones[i]), (flags, i)
        for i in range(1, 6):
            want = (w.double() * o_none[i].double()).float()
            live = w != 0
            assert torch.allclose(o_w[i][live], want[live], rtol=1e-6, atol=0), (flags, i)
            assert torch.equal(o_w[i][~live], torch.zeros_like(o_w[i][~live])), (flags, i)
        assert torch.equal(o_w[0][[2, 5]], torch.zeros(2, device=DEV))


def _oracle_check(t, noise, args, up, kw, out, grads):
    """The weighted tests' bar: outputs within 1e-5 of the fp32 oracle (of the fp64 oracle under STABLE_CDF, which does
    not follow the reference's fp32 tails), gradients against the fp64 oracle by relative L2 <= max(1e-5, 2x the fp32
    oracle's own) or the trimmed form with <= 1e-4; gradients exactly 0 in the oracle exactly 0 here."""
    L = t["y"].shape[1]
    names = RO.ROW_TERMS + ("indiv_prob", "indiv_prob_label")
    lw = None
    if "pos_weight" in kw:
        lw = torch.stack([kw["neg_weight"], kw["pos_weight"]])
    okw = dict(row_weight=kw.get("row_weight"), label_mask=kw.get("label_mask"), label_weight=lw,
               ranking="factorised" if L > 128 else "pairwise")
    upn = {names[i]: v for i, v in up.items()}
    ref, rg32 = RO.row_probit_elbo_with_grads(t, noise, args.nll_coeff, args.c_coeff, upn, **okw)
    cpu = lambda v: None if v is None else v.cpu()   # noqa: E731
    okw64 = {k: (cpu(v) if isinstance(v, torch.Tensor) else v) for k, v in okw.items()}
    ref64, rg = RO.row_probit_elbo_with_grads({k: v.cpu() for k, v in t.items()}, noise.cpu(), args.nll_coeff,
                                              args.c_coeff, {k: v.cpu().double() for k, v in upn.items()}, dtype=torch.float64,
                                              **okw64)
    if args.mpvae_flags & STABLE:
        ref = ref64
    for i in range(8):
        got, want = out[i].double().cpu(), ref[i].detach().double().cpu()
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-5), (names[i], float((got - want).abs().max()))
    errs = {}
    for k in LEAVES:
        got, want, theirs = grads[k].double().cpu().numpy(), rg[k].numpy(), rg32[k].double().cpu().numpy()
        if not np.any(want):
            assert not np.any(got), k
            continue
        e, et = H.rel_err_l2(got, want), H.rel_err_l2_trimmed(got, want)
        r, rt = H.rel_err_l2(theirs, want), H.rel_err_l2_trimmed(theirs, want)
        errs[k] = e
        assert e <= max(1e-5, 2 * r) or (et <= max(1e-5, 2 * rt) and e <= 1e-4), (k, e, et, r, rt)
    return errs


ORACLE_CASES = [(10, 16, 38, 38, 0), (1, 5, 14, 14, 0), (100, 37, 81, 81, 0), (10, 33, 983, 10, 0), (3, 17, 3993, 10, 0),
                (10, 20, 983, 983, 0), (7, 19, 130, 64, TENSOR), (10, 12, 257, 300, FMA), (10, 16, 38, 38, STABLE)]


@pytest.mark.parametrize("S,B,L,Z,flags", ORACLE_CASES)
@pytest.mark.parametrize("kind", ["plain", "all"])
def test_against_the_row_oracle(S, B, L, Z, flags, kind):
    """Random per-row cotangents (positive, zero, negative) on all six outputs and (B, L) cotangents on the predictions,
    with and without mask, row weights (one of them 0) and label weights."""
    t, noise = _inputs(S, B, L, Z, True, seed=3 * S + L, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    kw = _options(B, L, kind, seed=S + B)
    if "label_mask" in kw:
        kw["label_mask"][:, :2] = True
    if "row_weight" in kw:
        kw["row_weight"][1] = 0.0
    g = torch.Generator().manual_seed(B)
    up = {}
    for i in range(6):
        v = torch.randn(B, generator=g)
        v[torch.rand(B, generator=g) < 0.25] = 0.0
        up[i] = v.to(DEV)
    up[0][2] = 0.0
    up[6] = (torch.randn(B, L, generator=g) * 0.1).to(DEV)
    up[7] = (torch.randn(B, L, generator=g) * 0.1).to(DEV)
    args = _args(S, L, Z, flags)
    out, grads = _run(t, noise, args, "none", upstream=up, **kw)
    _oracle_check(t, noise, args, up, kw, out, grads)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 70, 983, 983, 0), (7, 19, 130, 64, TENSOR)])
def test_large_row_cotangent_keeps_g_r_within_the_oracle_bar(S, B, L, Z, flags):
    """One row's cotangent 1e4 (the rest 1): the bound that scales the fp16 operand planes of the g_R product reads the
    per-row cotangents, so g_R stays within the oracle bar."""
    t, noise = _inputs(S, B, L, Z, True, seed=5 * S + L, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    g = torch.ones(B, device=DEV)
    g[4] = 1.0e4
    args = _args(S, L, Z, flags)
    out, grads = _run(t, noise, args, "none", upstream={0: g})
    assert bool(torch.isfinite(grads["r_sqrt_sigma"]).all())
    errs = _oracle_check(t, noise, args, {0: g}, {}, out, grads)
    print(f"[large cotangent] S{S} B{B} L{L} Z{Z}: g_R rel L2 {errs['r_sqrt_sigma']:.2e}")


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 20, 983, 983, 0),
                                           (10, 20, 983, 983, TENSOR), (10, 16, 38, 38, STABLE)])
def test_degenerate_rows_left_out_by_indexing(S, B, L, Z, flags):
    """Rows 1 (all labels 0) and 2 (all 1) are degenerate; without SANITIZE, `total[keep].sum()` over the other rows
    leaves every gradient finite and their logit gradients exactly 0; selecting them gives NaN as 'mean' does."""
    from mpvae_b200.mpvae import compute_loss
    t, noise = _inputs(S, B, L, Z, True, seed=13 * L + S, rate=0.3)
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    t["y"][1], t["y"][2] = 0.0, 1.0
    args = _args(S, L, Z, flags)
    keep = torch.tensor([b not in (1, 2) for b in range(B)], device=DEV)
    leaves = {k: t[k].detach().clone().requires_grad_(True) for k in LEAVES}
    out = compute_loss(t["y"], *(leaves[k] for k in LEAVES), args, noise=noise, reduction="none")
    out[0][keep].sum().backward()
    for k in LEAVES:
        assert bool(torch.isfinite(leaves[k].grad).all()), k
    for k in ("fe_out", "fx_out"):
        assert torch.equal(leaves[k].grad[1:3], torch.zeros_like(leaves[k].grad[1:3])), k
    _, g_all = _run(t, noise, args, "none")
    _, g_mean = _run(t, noise, args)
    for g in (g_all, g_mean):
        assert bool(torch.isnan(g["fe_out"][1]).any()) and bool(torch.isnan(g["fe_out"][2]).any())


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 70, 983, 983, 0),
                                           (100, 37, 81, 81, STABLE)])
def test_repeatable_and_poisoned_workspace(S, B, L, Z, flags, monkeypatch):
    t, noise = _inputs(S, B, L, Z, False, seed=S * L)
    kw = _options(B, L, "all", seed=3)
    args = _args(S, L, Z, flags)
    up = {0: torch.linspace(-1.0, 2.0, B, device=DEV), 2: torch.ones(B, device=DEV)}
    o0, g0 = _run(t, noise, args, "none", upstream=up, **kw)
    o1, g1 = _run(t, noise, args, "none", upstream=up, **kw)
    monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
    o2, g2 = _run(t, noise, args, "none", upstream=up, **kw)
    for o, g in ((o1, g1), (o2, g2)):
        for i in range(8):
            assert _bits(o0[i], o[i]), i
        for k in LEAVES:
            assert _bits(g0[k], g[k]), k


def test_empty_batch_and_refusal():
    from mpvae_b200 import mpvae
    S, B, L, Z = 10, 16, 38, 38
    t, _ = _inputs(S, B, L, Z, False, seed=1)
    args = _args(S, L, Z)
    empty = {k: (v if k == "r_sqrt_sigma" else v[:0]) for k, v in t.items()}
    out = mpvae.compute_loss(empty["y"], *(empty[k] for k in LEAVES), args, reduction="none")
    assert all(o.shape == (0,) for o in out[:6]) and out[6].shape == (0, L)
    del args.noise_offset
    before = dict(mpvae._state)
    with pytest.raises(ValueError, match="reduction"):
        mpvae.compute_loss(t["y"], *(t[k] for k in LEAVES), args, reduction="sum")
    assert mpvae._state == before


def _small_loss_objective(q):
    """keep, per batch, the rows whose detached per-row total is below the batch's q-quantile"""
    def f(out, rows):
        total = out[0]
        keep = (total.detach() <= torch.quantile(total.detach(), q)).float()
        return keep * total
    return f


def test_one_gpu_data_parallel_step_with_a_row_objective_is_the_hand_loop():
    """DataParallelStep(row_objective=) on one GPU == compute_loss(reduction='none') + (phi.sum() / B).backward() + clip +
    Adam, bit for bit; the returned scalars are the means of the per-row terms."""
    from mpvae_b200.mpvae import VAE, compute_loss
    from mpvae_b200.train import DataParallelStep
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    x, y = _planted(64, F, L, Z, seed=5)
    objective = _small_loss_objective(0.6)

    def build():
        torch.manual_seed(0)
        np.random.seed(0)
        m = VAE(args).to(DEV)
        return m, torch.optim.Adam(m.parameters(), lr=1e-3)

    m1, o1 = build()
    step = DataParallelStep(m1, o1, None, args, clip_norm=100.0, row_objective=objective)
    m2, o2 = build()
    a2 = copy.copy(args)
    for i in range(3):
        torch.manual_seed(100 + i)
        so = step.step(y, x)
        torch.manual_seed(100 + i)
        a2.noise_offset = i
        o2.zero_grad()
        out = compute_loss(y, *m2(y, x), m2.r_sqrt_sigma, a2, reduction="none")
        (objective(out, slice(0, 64)).sum() * (1.0 / 64)).backward()
        torch.nn.utils.clip_grad_norm_([p for p in m2.parameters() if p.grad is not None], 100.0)
        o2.step()
        for j in range(6):
            assert torch.equal(so[j], out[j].detach().mean()), (i, j)
    torch.cuda.synchronize()
    for (k, p1), (_, p2) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(p1, p2), k


def test_predict_proba_per_rows_agree_with_the_sums():
    from mpvae_b200 import infer
    from mpvae_b200.mpvae import VAE
    F, L, Z, S = 40, 38, 38, 10
    args = _vae_args(F, L, Z, S)
    x, y = _planted(300, F, L, Z, seed=9)
    torch.manual_seed(0)
    model = VAE(args).to(DEV).eval()
    res = {}
    for red in ("mean", "none"):
        torch.manual_seed(1)
        args.noise_offset = 5
        res[red] = infer.predict_proba(model, x, y, args, batch_size=128, reduction=red)
    assert torch.equal(res["mean"][0], res["none"][0])
    rows = res["none"][1]
    assert set(rows) == set(RO.ROW_TERMS) and all(v.shape == (300,) for v in rows.values())
    for k in ("total_loss", "nll_loss", "c_loss"):
        got, want = float(rows[k].double().sum()), float(res["mean"][1][k])
        assert abs(got - want) <= 1e-5 * abs(want), (k, got, want)


# ---- the planted model with noisy rows (test_weighted_loss_gpu): detection and small-loss training ----

EPOCHS = 6                       # test_weighted_loss_gpu.EPOCHS_NOISY_ROWS


def _noisy_problem():
    F, L, Z, S = 103, 14, 14, 10
    args = _vae_args(F, L, Z, S, c_coeff=0.1, flags=SANITIZE)
    x, y = _planted(6000, F, L, Z, seed=3)
    xt, yt, xv, yv = x[:4000], y[:4000].clone(), x[4000:], y[4000:]
    g = torch.Generator().manual_seed(8)
    noisy = (torch.rand(4000, generator=g) < 0.4).to(DEV)
    donor = torch.randint(0, 4000, (4000,), generator=g).to(DEV)
    return args, xt, torch.where(noisy[:, None], yt[donor], yt), noisy, xv, yv


def _train(args, x, y, epochs, weights=None, row_objective=None):
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    torch.manual_seed(0)
    np.random.seed(0)
    model = VAE(args).to(DEV)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
    step = DataParallelStep(model, opt, None, args, clip_norm=100.0, row_objective=row_objective)
    for ep in range(epochs):
        order = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(ep)).to(DEV)
        train_one_epoch(step, x, y, args.batch_size, order=order, weights=weights)
    return model


def _auroc(score, label):
    r = torch.empty_like(score, dtype=torch.float64)
    r[torch.argsort(score)] = torch.arange(1, score.numel() + 1, dtype=torch.float64, device=score.device)
    n1 = int(label.sum())
    n0 = label.numel() - n1
    return (float(r[label].sum()) - n1 * (n1 + 1) / 2) / (n1 * n0)


def _cell_logloss(model, args, xv, yv):
    from mpvae_b200.mpvae import predict_exact
    a = copy.copy(args)
    a.mode = "test"
    model.eval()
    with torch.no_grad():
        p = predict_exact(model.feat_forward(xv)[0], model.r_sqrt_sigma, a).double().clamp(1e-7, 1 - 1e-7)
    yd = yv.double()
    return -(yd * torch.log(p) + (1 - yd) * torch.log(1 - p)).flatten()


AUROC_BAR = 0.80                # measured 0.876 on one B200 (DESIGN §5)


def test_planted_noisy_rows_are_found_by_their_nll_x():
    """Train with uniform weights, then score the training rows: the AUROC of each row's held-out-style nll_x
    (predict_proba(reduction='none'), test mode) for the noisy-row indicator."""
    from mpvae_b200 import infer
    args, xt, yn, noisy, _, _ = _noisy_problem()
    model = _train(args, xt, yn, EPOCHS)
    a = copy.copy(args)
    a.noise_offset = 0
    torch.manual_seed(1)
    _, rows = infer.predict_proba(model, xt, yn, a, batch_size=500, reduction="none")
    auc = {k: _auroc(rows[k], noisy) for k in ("nll_loss_x", "total_loss", "nll_loss")}
    print("[noisy rows] AUROC " + "  ".join(f"{k} {v:.4f}" for k, v in auc.items()))
    assert auc["nll_loss_x"] > AUROC_BAR, auc


def test_planted_small_loss_training():
    """Keep, per batch, the rows below the batch's 0.6-quantile of the detached per-row total (40 % of the rows are
    noisy); held-out per-cell log-loss against uniform weights and the 0.05 weights an oracle of the noisy rows gives.
    Measured on one B200 the selection does not beat uniform weights (DESIGN §5), so only the run itself is asserted."""
    args, xt, yn, noisy, xv, yv = _noisy_problem()
    ls = _cell_logloss(_train(args, xt, yn, EPOCHS, row_objective=_small_loss_objective(0.6)), args, xv, yv)
    lu = _cell_logloss(_train(args, xt, yn, EPOCHS), args, xv, yv)
    lw = _cell_logloss(_train(args, xt, yn, EPOCHS, weights=torch.where(noisy, 0.05, 1.0).float()), args, xv, yv)
    d = lu - ls
    se = float(d.std() / np.sqrt(d.numel()))
    print(f"[small loss] per-cell log-loss: small-loss {float(ls.mean()):.4f}  uniform {float(lu.mean()):.4f}  "
          f"oracle 0.05 weights {float(lw.mean()):.4f}  (uniform - small-loss {float(d.mean()):.4f} +- {se:.4f})")
    assert bool(torch.isfinite(ls).all())
