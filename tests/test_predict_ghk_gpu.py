"""GPU: the GHK conditional prediction (mpvae_probit_predict_conditional_ghk: the nt product, the G product,
ghk_gather_kernel, ghk_factor_kernel, ghk_chain_kernel, ghk_update_kernel, then predict.cu's conditional weights and
predict kernels) against predict with nothing observed, its exact cases (R = 0, one observed label), the fp64 oracle on the same
draws, quadrature, the importance path and PairPredictor; a planted model where it must beat the importance path; and
batching, row groups, repetition, a poisoned workspace, a prepared G, offsets and launch counts."""
import math

import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import predict_exact_oracle as XO
from tests import predict_ghk_oracle as GO
from tests.test_predict_gpu import EQUALITY_CASES, _args, _inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

STABLE, FMA, TENSOR, SEPARATE, FUSED = 0x8, 0x4, 0x2, 0x20, 0x10


def _none(B, L):
    return torch.full((B, L), -1, dtype=torch.int8, device=DEV)


def _random_obs(B, L, seed, frac=0.5, y=None, empty_rows=(0,)):
    """Mixed patterns: the rows in empty_rows observe nothing, row 1 (B > 1) everything, the others a random share."""
    g = torch.Generator().manual_seed(seed)
    vals = (torch.rand(B, L, generator=g) < 0.3).to(torch.int8) if y is None else y.cpu().to(torch.int8)
    keep = torch.rand(B, L, generator=g) < frac
    if B > 1:
        keep[1] = True
    for b in empty_rows:
        if b < B:
            keep[b] = False
    return torch.where(keep, vals, torch.full_like(vals, -1)).to(DEV)


def _ghk(t, obs, args, noise=None, gram=None):
    from mpvae_b200.mpvae import predict_conditional_ghk
    with torch.no_grad():
        out = predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"], obs, args, noise=noise, gram=gram)
    torch.cuda.synchronize()
    return out


def _draws(S, B, L, seed):
    g = torch.Generator().manual_seed(seed)
    zeta = torch.randn(S, B, L, generator=g)
    U = torch.rand(S, B, L, generator=g).clamp(2.0 ** -24, 1 - 2.0 ** -24)
    return zeta.to(DEV), U.to(DEV)


def _ghk_external(t, obs, S, noise, zeta, U, flags=0):
    from mpvae_b200.probit import probit_predict_conditional_ghk
    mo = int(((obs == 0) | (obs == 1)).sum(1).max())
    with torch.no_grad():
        out = probit_predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"].float(), obs, S, mo, noise=noise,
                                             flags=flags, zeta=zeta, uniform=U)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("S,B,L,Z,flags,external", EQUALITY_CASES)
def test_nothing_observed_is_predict(S, B, L, Z, flags, external):
    """No observed label: lw = 0 and no update -- predict's indiv_prob bit for bit, log_evidence = 0, ess = S."""
    from mpvae_b200.mpvae import predict
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        want = predict(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
    got = _ghk(t, _none(B, L), args, noise)
    assert torch.equal(got.prob, want)
    assert torch.equal(got.log_evidence, torch.zeros(B, device=DEV))
    assert torch.equal(got.ess, torch.full((B,), float(S), device=DEV))


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 12, 83, 10, 0), (10, 20, 300, 256, 0), (7, 9, 130, 64, TENSOR)])
def test_empty_rows_in_a_mixed_batch_are_predict(S, B, L, Z, flags):
    from mpvae_b200.mpvae import predict
    t, _ = _inputs(S, B, L, Z, False, seed=3)
    args = _args(S, L, Z, flags)
    obs = _random_obs(B, L, seed=4, frac=0.3, empty_rows=(0, 3, 5))
    with torch.no_grad():
        want = predict(t["fx_out"], t["r_sqrt_sigma"], args)
    got = _ghk(t, obs, args)
    for b in (0, 3, 5):
        assert torch.equal(got.prob[b], want[b])
        assert float(got.log_evidence[b]) == 0.0 and float(got.ess[b]) == S


@pytest.mark.parametrize("S,B,L,Z,flags", [(100, 9, 81, 81, 0), (10, 12, 983, 10, 0), (10, 20, 300, 256, 0),
                                           (10, 8, 257, 300, STABLE)])
def test_zero_r_identities(S, B, L, Z, flags):
    """R = 0: G = 0, C = I, constant weights prod (c + k Phi(+-fx_o)), unobserved cells = predict's bits."""
    from mpvae_b200.mpvae import predict
    t, _ = _inputs(S, B, L, Z, False, seed=11)
    t["r_sqrt_sigma"] = torch.zeros_like(t["r_sqrt_sigma"])
    args = _args(S, L, Z, flags)
    obs = _random_obs(B, L, seed=3, frac=0.4)
    with torch.no_grad():
        want = predict(t["fx_out"], t["r_sqrt_sigma"], args)
    got = _ghk(t, obs, args)
    free = (obs != 0) & (obs != 1)
    assert torch.equal(got.prob[free], want[free])
    assert torch.equal(got.prob[~free], obs[~free].float())
    assert torch.allclose(got.ess, torch.full((B,), float(S), device=DEV), rtol=1e-6, atol=0)
    P = XO.C_EPS + XO.K_EPS * torch.special.ndtr(t["fx_out"].double().cpu())
    ocpu = obs.cpu()
    cell = torch.where(ocpu == 1, P, torch.where(ocpu == 0, 1 - P, torch.ones_like(P)))
    want_le = torch.log(cell).sum(1)
    assert torch.allclose(got.log_evidence.double().cpu(), want_le, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("S,B,L,Z,flags", [(100, 8, 81, 81, 0), (10, 10, 983, 10, 0), (10, 20, 300, 256, 0)])
def test_one_observed_label_identities(S, B, L, Z, flags):
    """|O| = 1: every sample has the weight c + k Phi(+-fx_o / sqrt(1 + |R_o|^2)): ess = S and log_evidence = its log."""
    t, _ = _inputs(S, B, L, Z, False, seed=12)
    args = _args(S, L, Z, flags)
    g = torch.Generator().manual_seed(5)
    obs = torch.full((B, L), -1, dtype=torch.int8)
    cols = torch.randint(0, L, (B,), generator=g)
    ys = torch.randint(0, 2, (B,), generator=g)
    obs[torch.arange(B), cols] = ys.to(torch.int8)
    got = _ghk(t, obs.to(DEV), args)
    marg = XO.marginal(t["fx_out"], t["r_sqrt_sigma"])[torch.arange(B), cols]
    want = torch.where(ys == 1, marg, 1 - marg)
    assert torch.allclose(got.ess, torch.full((B,), float(S), device=DEV), rtol=1e-6, atol=0)
    assert torch.allclose(got.log_evidence.double().cpu(), torch.log(want), rtol=1e-6, atol=0)


# (S, B, L, Z, flags): CUDA-core (incl. S = 1, STABLE, FMA), then dense
ORACLE_FMA = [(10, 9, 83, 10, 0), (1, 7, 130, 64, FMA), (37, 5, 257, 40, 0), (10, 6, 38, 38, STABLE), (3, 4, 983, 10, 0)]
ORACLE_DENSE = [(10, 20, 300, 256, 0), (7, 19, 130, 64, TENSOR)]


def _distances(got, want):
    prob, le, ess = (x.double().cpu() for x in got)
    wp, wl, we = want
    return (float((prob - wp).abs().max()), float(((le - wl).abs() / wl.abs().clamp(min=1e-30)).max()),
            float(((ess - we).abs() / we).max()))


@pytest.mark.parametrize("S,B,L,Z,flags", ORACLE_FMA + ORACLE_DENSE)
def test_against_the_oracle_on_the_same_draws(S, B, L, Z, flags):
    """External xi, zeta, U handed to the fp64 oracle.  CUDA-core regime: prob <= 2e-5 absolute, log_evidence <= 1e-5
    relative, ess <= 1e-4 relative.  Dense regime (G and nr on the split-precision tensor engine): each distance within
    2x that of the fp32 restatement of the same algorithm, or within the CUDA-core bar."""
    t, noise = _inputs(S, B, L, Z, True, seed=7 * L + S)
    obs = _random_obs(B, L, seed=L, frac=0.3, y=t["y"])
    zeta, U = _draws(S, B, L, seed=S + L)
    got = _ghk_external(t, obs, S, noise, zeta, U, flags)
    args = (t["fx_out"], t["r_sqrt_sigma"], obs, noise, zeta, U)
    want = GO.predict_conditional_ghk(*args)
    d = _distances(got, want)
    bars = (2e-5, 1e-5, 1e-4)
    if (S, B, L, Z, flags) in ORACLE_DENSE:
        d32 = _distances(GO.predict_conditional_ghk(*args, dtype=torch.float32), want)
        print("ghk dense distances", (S, B, L, Z, flags), "library", d, "fp32 restatement", d32)
        bars = tuple(max(2 * a, b) for a, b in zip(d32, bars))
    assert all(x <= bar for x, bar in zip(d, bars)), (d, bars)
    assert bool(((got[2] >= 1 - 1e-5) & (got[2] <= S * (1 + 1e-6))).all())


@pytest.mark.parametrize("Z", [1, 2])
def test_converges_to_quadrature_with_most_labels_observed(Z):
    """S = 10 000, L = 20, ~80 % observed: evidence and conditional marginals within 6 SE of Gauss-Hermite quadrature
    (SE from the oracle's spread on its own draws at the same S)."""
    S, B, L = 10000, 4, 20
    g = torch.Generator().manual_seed(40 + Z)
    fx = torch.randn(B, L, generator=g)
    r = torch.randn(L, Z, generator=g) * 1.5 / math.sqrt(Z)
    obs = torch.where(torch.rand(B, L, generator=g) < 0.8, (torch.rand(B, L, generator=g) < 0.4).to(torch.int8),
                      torch.full((B, L), -1, dtype=torch.int8))
    t = {"fx_out": fx.to(DEV), "r_sqrt_sigma": r.to(DEV)}
    args = _args(S, L, Z, 0)
    got = _ghk(t, obs.to(DEV), args)
    qp, qle = GO.quadrature(fx, r, obs)
    xi = torch.randn(S, B, Z, generator=g)
    zeta = torch.randn(S, B, L, generator=g)
    U = torch.rand(S, B, L, generator=g, dtype=torch.float64).clamp(1e-12, 1 - 1e-12)
    se_p, se_le = GO.stderr(fx, r, obs, xi, zeta, U)
    assert bool(((got.log_evidence.double().cpu() - qle).abs() <= 6 * se_le).all()), (got.log_evidence, qle, se_le)
    free = (obs != 0) & (obs != 1)
    err = (got.prob.double().cpu() - qp).abs()
    assert bool((err[free] <= 6 * se_p[free] + 1e-6).all()), float((err / se_p)[free].max())
    assert bool((got.ess > 0.01 * S).all())


def test_few_observed_agree_with_the_importance_path_and_pair_predictor():
    """S = 10 000, one observed label per row: within 6 / sqrt(ess) of PairPredictor's P(y_l, y_o) / P(y_o) and of the
    importance path's estimate."""
    from mpvae_b200.mpvae import PairPredictor, predict_conditional
    S, B, L, Z = 10000, 6, 83, 10
    t, _ = _inputs(S, B, L, Z, False, seed=21)
    args = _args(S, L, Z, 0)
    g = torch.Generator().manual_seed(8)
    cols = torch.randint(0, L, (B,), generator=g)
    obs = torch.full((B, L), -1, dtype=torch.int8)
    obs[torch.arange(B), cols] = 1
    obs = obs.to(DEV)
    got = _ghk(t, obs, args)
    with torch.no_grad():
        imp = predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, args)
    for b in range(B):
        pb = torch.stack([torch.arange(L), torch.full((L,), int(cols[b]))], 1).to(DEV)
        with torch.no_grad():
            pp = PairPredictor(t["r_sqrt_sigma"], pb, args)
            joint = pp(t["fx_out"][b:b + 1])[0].double()
        want = joint / joint[int(cols[b])]
        free = torch.arange(L, device=DEV) != int(cols[b])
        tol = 6 / math.sqrt(float(got.ess[b]))
        assert float((got.prob[b].double() - want)[free].abs().max()) <= tol
        tol2 = 6 * math.sqrt(1 / float(got.ess[b]) + 1 / float(imp.ess[b]))
        assert float((got.prob[b] - imp.prob[b])[free].abs().max()) <= tol2


def test_planted_model_ghk_beats_importance():
    """Labels drawn from a probit model with a rank-4 correlation at delicious width (L = 983), half of each row observed,
    S = 100: the GHK sampler's median ESS exceeds the importance path's, and its log-loss on the hidden labels beats the
    importance path's by more than 5 standard errors (paired over rows)."""
    from mpvae_b200.mpvae import predict_conditional
    S, B, L, Z = 100, 48, 983, 4
    g = torch.Generator().manual_seed(2024)
    r = torch.randn(L, Z, generator=g) * 1.2
    fx = torch.randn(B, L, generator=g) * 0.5 - 0.5
    eps = torch.randn(B, Z, generator=g)
    u = fx + eps @ r.T + torch.randn(B, L, generator=g)
    y = (u > 0).to(torch.int8)
    keep = torch.rand(B, L, generator=g) < 0.5
    obs = torch.where(keep, y, torch.full_like(y, -1)).to(DEV)
    t = {"fx_out": fx.to(DEV), "r_sqrt_sigma": r.to(DEV)}
    args = _args(S, L, Z, 0)
    ghk = _ghk(t, obs, args)
    with torch.no_grad():
        imp = predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, args)
    hidden = (~keep).to(DEV)
    yd = y.to(DEV).double()

    def row_loss(p):
        p = p.double().clamp(1e-7, 1 - 1e-7)
        cell = -(yd * torch.log(p) + (1 - yd) * torch.log(1 - p))
        return (cell * hidden).sum(1) / hidden.sum(1)

    diff = row_loss(imp.prob) - row_loss(ghk.prob)
    se = float(diff.std()) / math.sqrt(B)
    print("planted: median ess ghk", float(ghk.ess.median()), "importance", float(imp.ess.median()),
          "hidden log-loss ghk", float(row_loss(ghk.prob).mean()), "importance", float(row_loss(imp.prob).mean()),
          "diff", float(diff.mean()), "se", se)
    assert float(ghk.ess.median()) > float(imp.ess.median())
    assert float(diff.mean()) > 5 * se


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 9, 83, 10, 0), (7, 6, 130, 64, TENSOR)])
def test_rows_alone_equal_rows_in_a_batch(S, B, L, Z, flags):
    t, _ = _inputs(S, B, L, Z, False, seed=31)
    obs = _random_obs(B, L, seed=2, frac=0.4)
    args = _args(S, L, Z, flags, dp_global_batch=B, dp_row0=0)
    full = _ghk(t, obs, args)
    for b in range(B):
        rows = {k: (v if k == "r_sqrt_sigma" else v[b:b + 1]) for k, v in t.items()}
        one = _ghk(rows, obs[b:b + 1], _args(S, L, Z, flags, dp_global_batch=B, dp_row0=b))
        assert torch.equal(one.prob[0], full.prob[b])
        assert torch.equal(one.log_evidence[0], full.log_evidence[b]) and torch.equal(one.ess[0], full.ess[b])


@pytest.mark.parametrize("S,B,L,Z,flags,external", [(10, 11, 83, 10, 0, False), (7, 9, 130, 64, TENSOR, False),
                                                    (10, 11, 83, 10, 0, True)])
def test_row_groups_change_no_bits(S, B, L, Z, flags, external, monkeypatch):
    from mpvae_b200 import mpvae
    t, noise = _inputs(S, B, L, Z, external, seed=32)
    obs = _random_obs(B, L, seed=5, frac=0.4)
    args = _args(S, L, Z, flags)
    whole = _ghk(t, obs, args, noise)
    monkeypatch.setattr(mpvae, "GHK_WORKSPACE_BOUND", mpvae.ghk_workspace_bytes(S, 3, L, Z, L, flags))
    split = _ghk(t, obs, args, noise)
    for a, b in zip(whole, split):
        assert torch.equal(a, b)


def test_repeat_poison_gram_and_empty(monkeypatch):
    from mpvae_b200 import mpvae
    for (S, B, L, Z, flags) in ((10, 9, 83, 10, 0), (10, 20, 300, 256, 0), (10, 9, 300, 256, FMA)):
        t, _ = _inputs(S, B, L, Z, False, seed=33)
        obs = _random_obs(B, L, seed=6, frac=0.3)
        args = _args(S, L, Z, flags)
        a = _ghk(t, obs, args)
        b = _ghk(t, obs, args)
        with torch.no_grad():
            G = mpvae.label_gram(t["r_sqrt_sigma"], args)
        c = _ghk(t, obs, args, gram=G)
        monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
        d = _ghk(t, obs, args)
        monkeypatch.delenv("MPVAE_POISON_WORKSPACE")
        for x in (b, c, d):
            for u, v in zip(a, x):
                assert torch.equal(u, v)
        assert bool(torch.isfinite(a.prob).all() and torch.isfinite(a.log_evidence).all())
    t, _ = _inputs(10, 4, 83, 10, False, seed=1)
    empty = {"fx_out": t["fx_out"][:0], "r_sqrt_sigma": t["r_sqrt_sigma"]}
    out = _ghk(empty, _none(0, 83), _args(10, 83, 10, 0))
    assert out.prob.shape == (0, 83) and out.log_evidence.shape == (0,) and out.ess.shape == (0,)


def test_offset_consumption_is_predicts():
    from mpvae_b200 import mpvae
    S, B, L, Z = 10, 5, 83, 10
    t, _ = _inputs(S, B, L, Z, False, seed=34)
    args = orc.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=4242)
    obs = _random_obs(B, L, seed=7)
    before = mpvae._state["offset"]
    _ghk(t, obs, args)
    assert mpvae._state["offset"] == before + 1
    with torch.no_grad():
        mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], args)
    assert mpvae._state["offset"] == before + 2


def test_launch_counts():
    """CUDA-core regime: the importance path launches noise, product, loglik, weights, predict; the GHK path replaces
    loglik by gather, factor, chain, update and adds the G product (none of factor, update and G with nothing
    observed)."""
    from mpvae_b200 import _lib, mpvae
    lib = _lib.lib()
    S, B, L, Z = 10, 9, 83, 10
    t, _ = _inputs(S, B, L, Z, False, seed=35)
    args = _args(S, L, Z, 0)
    obs = _random_obs(B, L, seed=8)
    G = mpvae.label_gram(t["r_sqrt_sigma"], args)
    torch.cuda.synchronize()

    def count(fn):
        c0 = lib.mpvae_launch_count()
        with torch.no_grad():
            fn()
        torch.cuda.synchronize()
        return lib.mpvae_launch_count() - c0

    imp = count(lambda: mpvae.predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, args))
    ghk = count(lambda: mpvae.predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"], obs, args))
    ghk_g = count(lambda: mpvae.predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"], obs, args, gram=G))
    none = count(lambda: mpvae.predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"], _none(B, L), args))
    assert (imp, ghk, ghk_g, none) == (5, 9, 8, 6)


def test_infer_predict_conditional_with_the_ghk_predict_fn():
    """infer.predict_conditional(predict_fn=mpvae.predict_conditional_ghk) over a dataset: with nothing observed the
    default path's prob bit for bit (same torch seed); with labels observed, finite and ess in [1, S]."""
    from types import SimpleNamespace
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_conditional
    from mpvae_b200.mpvae import VAE
    args = SimpleNamespace(feature_dim=12, label_dim=40, latent_dim=6, z_dim=8, keep_prob=1.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=16, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=16)
    torch.manual_seed(0)
    model = VAE(args).to(DEV)
    x = torch.randn(37, 12, device=DEV)
    none = _none(37, 40)
    torch.manual_seed(1)
    want = predict_conditional(model, x, none, args)
    torch.manual_seed(1)
    got = predict_conditional(model, x, none, args, predict_fn=mpvae.predict_conditional_ghk)
    assert torch.equal(got[0], want[0])
    obs = _random_obs(37, 40, seed=9, frac=0.5)
    prob, le, ess = predict_conditional(model, x, obs, args, predict_fn=mpvae.predict_conditional_ghk)
    assert bool(torch.isfinite(prob).all() and torch.isfinite(le).all())
    assert bool(((ess >= 1 - 1e-5) & (ess <= 16 * (1 + 1e-6))).all())
