"""GPU: the closed-form prediction (csrc/predictive.cu: predictive_scale / predictive_rho / predict_exact / predict_pairs
kernels) against the fp64 oracle (tests/predict_exact_oracle.py), against mpvae.predict's Monte Carlo (bit for bit where
R = 0, statistically at S = 10 000), and at the model level through infer.predict_proba / infer.predict_pairs."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import predict_exact_oracle as XO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
STABLE = 0x8


def _inputs(B, L, Z, sigma=1.0, seed=0, r_scale=1.0):
    from mpvae_b200 import synth
    inp = synth.loss_inputs(L, Z, B, 1, seed=seed, sigma=sigma, with_noise=False)
    return torch.from_numpy(inp["fx_out"]).to(DEV), torch.from_numpy(inp["r_sqrt_sigma"] * r_scale).to(DEV)


def _args(L, Z, S=100, flags=0, **kw):
    return orc.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=4242, noise_offset=6, mpvae_flags=flags, **kw)


def _ulp_close(got, want, atol):
    """|got - want| <= max(atol, 1 fp32 ulp of want), elementwise (want fp64)."""
    g = got.double().cpu().numpy()
    w = want.double().cpu().numpy()
    ulp = np.spacing(np.abs(w).astype(np.float32)).astype(np.float64)
    return np.abs(g - w) <= np.maximum(atol, ulp)


# the three regime shapes (small 38/38, mid 3993/10, dense 983/983) and odd L for the scalar tail
SHAPES = [(64, 38, 38), (64, 3993, 10), (32, 983, 983), (9, 131, 7), (5, 37, 5), (3, 1, 3)]


@pytest.mark.parametrize("B,L,Z", SHAPES)
@pytest.mark.parametrize("sigma", [1.0, 3.0])
def test_marginals_against_the_oracle(B, L, Z, sigma):
    """Faithful E: within 5e-7 of c + k Phi(h) in fp64.  STABLE_CDF: within 1e-6 relative (tails included) of the fp64
    formula at the fp32 argument probit_E_stable evaluates (x' = fp32(fx_out * scale), then t = fp32(x' / sqrt 2) as the
    reference's op order forms it), and within 3e-6 relative of c + k Phi(h) itself: the two argument roundings move
    Phi by up to ~2 t^2 * 6e-8 relative in the lower tail, where E is not yet the clamp."""
    from mpvae_b200 import mpvae
    fx, r = _inputs(B, L, Z, sigma, seed=B + L)
    with torch.no_grad():
        faithful = mpvae.predict_exact(fx, r, _args(L, Z))
        stable = mpvae.predict_exact(fx, r, _args(L, Z, flags=STABLE))
    assert faithful.shape == (B, L) and faithful.dtype == torch.float32
    err = (faithful.double().cpu() - XO.marginal(fx, r)).abs().max().item()
    assert err <= 5e-7, err
    want = XO.marginal_at_t(fx, r)
    rel = ((stable.double().cpu() - want).abs() / want).max().item()
    assert rel <= 1e-6, rel
    want = XO.marginal(fx, r)
    rel = ((stable.double().cpu() - want).abs() / want).max().item()
    assert rel <= 3e-6, rel


def test_odd_offsets_take_the_scalar_path():
    """A view whose rows do not start on 16 bytes gives the bits of the same rows laid out afresh."""
    from mpvae_b200 import probit
    fx, r = _inputs(17, 40, 8, seed=3)
    with torch.no_grad():
        scale = probit.predictive_scale(r.float())
        full = probit.predict_exact(fx, scale)
        view = torch.empty(17 * 40 + 1, device=DEV)[1:].view(17, 40)
        view.copy_(fx)
        assert torch.equal(probit.predict_exact(view, scale), full)


@pytest.mark.parametrize("B,L,Z,flags", [(128, 38, 38, 0), (128, 3993, 10, 0), (128, 983, 983, 0), (128, 300, 64, STABLE)])
@pytest.mark.parametrize("S", [1, 2, 4])
def test_equals_predict_bit_for_bit_when_r_is_zero(B, L, Z, flags, S):
    """R = 0 (residue_sigma='zero'): the scale is exactly 1, x' = fx_out, and predict's pair sums E + 0, E + E, 2E + 2E
    and the division by S are exact, so the Monte Carlo and the closed form give the same bits (small, CUDA-core and
    dense regime; the stable CDF in the CUDA-core one)."""
    from mpvae_b200 import mpvae
    fx, _ = _inputs(B, L, Z, seed=S + L)
    model_args = _args(L, Z, S, flags, feature_dim=8, latent_dim=4, keep_prob=0.0, scale_coeff=1.0, residue_sigma="zero")
    r = mpvae.VAE(model_args).r_sqrt_sigma.to(DEV)
    assert not bool(r.any())
    with torch.no_grad():
        mc = mpvae.predict(fx, r, model_args)
        exact = mpvae.predict_exact(fx, r, model_args)
    assert torch.equal(mc, exact)


@pytest.mark.parametrize("B,L,Z", [(128, 38, 38), (64, 3993, 10), (32, 983, 983)])
def test_monte_carlo_converges_to_the_closed_form(B, L, Z):
    """mpvae.predict at S = 10 000 against predict_exact: per-cell z-scores with the variance of the fp64 oracle,
    Var(E_l) = k^2 (Phi2(h, h; s / (1 + s)) - Phi(h)^2): max |z| <= 6 and RMS within [0.8, 1.2] over the cells whose
    standard error exceeds 2e-5, 10x the random part of the rounding of predict's fp32 running sum at S = 10 000.  Where
    the noise barely moves E (eurlex-Z10: |R_l|^2 ~ 0.005), that sum adds nearly the same pair sum S / 2 times and its
    rounding no longer averages out: up to ulp(S) / 4 = 2^-12 of bias, so those cells are held to 6 standard errors
    plus 2^-12."""
    from mpvae_b200 import mpvae
    S = 10_000
    fx, r = _inputs(B, L, Z, seed=L)
    with torch.no_grad():
        mc = mpvae.predict(fx, r, _args(L, Z, S))
        exact = mpvae.predict_exact(fx, r, _args(L, Z, S))
    var = XO.marginal_var(fx, r)
    se = torch.sqrt(var / S)
    diff = mc.double().cpu() - exact.double().cpu()
    keep = se > 2e-5
    assert keep.float().mean() > 0.5
    assert bool((diff.abs() <= 6 * se + 2.0 ** -12).all())
    z = (diff / se)[keep]
    zmax, rms = z.abs().max().item(), z.pow(2).mean().sqrt().item()
    assert zmax <= 6.0 and 0.8 <= rms <= 1.2, (zmax, rms)


def _pairs_with_extras(L, n_random=0, seed=0):
    from mpvae_b200.mpvae import all_pairs
    g = torch.Generator().manual_seed(seed)
    if n_random:
        p = torch.randint(0, L, (n_random, 2), generator=g)
    else:
        p = all_pairs(L)
    diag = torch.arange(L)[:, None].repeat(1, 2)[: min(L, 50)]
    return torch.cat([p, p.flip(1)[:200], diag])


@pytest.mark.parametrize("B,L,Z,n_random,flags,r_scale", [
    (16, 38, 38, 0, 0, 1.0), (8, 983, 983, 5000, 0, 1.0), (8, 3993, 10, 5000, 0, 1.0), (8, 81, 81, 0, STABLE, 1.0),
    (8, 200, 2, 5000, 0, 30.0), (8, 200, 3, 5000, 0, 3.0)])
def test_pairs_against_the_oracle(B, L, Z, n_random, flags, r_scale):
    """Within one fp32 ulp or 1.2e-7 of the fp64 formula with Owen's T.  A large R in few dimensions puts correlations
    into every branch of the quadrature, up to |rho| next to 1."""
    from mpvae_b200 import mpvae
    fx, r = _inputs(B, L, Z, sigma=2.0, seed=L + 1, r_scale=r_scale)
    pairs = _pairs_with_extras(L, n_random)
    with torch.no_grad():
        pp = mpvae.PairPredictor(r, pairs, _args(L, Z, flags=flags))
        got = pp(fx)
    assert got.shape == (B, pairs.shape[0])
    off = pairs[:, 0] != pairs[:, 1]
    ok = _ulp_close(got[:, off], XO.pair_prob(fx, r, pairs[off]), 1.2e-7)
    assert ok.all(), (~ok).sum()
    if r_scale >= 30.0:
        a = XO.rho(r, pairs[off]).abs()
        for lo, hi in ((0.0, 0.3), (0.3, 0.75), (0.75, 0.925), (0.925, 0.999)):
            assert bool(((a >= lo) & (a < hi)).any()), (lo, hi)


def test_pairs_against_monte_carlo():
    """All 703 pairs of L = 38: a fp64 torch Monte Carlo of mean_s E_i E_j over the library's Philox noise, S = 20 000."""
    from mpvae_b200 import mpvae
    from mpvae_b200.probit import philox_normal
    B, L, Z, S = 8, 38, 38, 20_000
    fx, r = _inputs(B, L, Z, seed=9)
    pairs = mpvae.all_pairs(L)
    with torch.no_grad():
        got = mpvae.PairPredictor(r, pairs, _args(L, Z))(fx).double()
        noise = philox_normal(S, B, Z, seed=123, offset=0, device=DEV).double()
        E = XO.C_EPS + XO.K_EPS * torch.special.ndtr(fx.double()[None] + noise @ r.float().double().T)   # (S, B, L)
        m = torch.einsum("sbi,sbj->bij", E, E) / S
        m2 = torch.einsum("sbi,sbj->bij", E * E, E * E) / S
    i, j = pairs[:, 0].to(DEV), pairs[:, 1].to(DEV)
    mean, sq = m[:, i, j], m2[:, i, j]
    se = torch.sqrt((sq - mean * mean) / S)
    z = ((mean - got) / se).abs().max().item()
    assert z <= 6.0, z


@pytest.mark.parametrize("flags", [0, STABLE])
def test_pair_symmetry_diagonal_and_bounds(flags):
    """(i, j) and (j, i) give the same bits, (i, i) the bits of predict_exact, and every pair lies within the Frechet
    bounds max(0, P_i + P_j - 1) <= P_ij <= min(P_i, P_j) of the fp64 marginals, to one ulp."""
    from mpvae_b200 import mpvae
    B, L, Z = 12, 81, 81
    fx, r = _inputs(B, L, Z, sigma=2.0, seed=4)
    up = mpvae.all_pairs(L)
    pairs = torch.cat([up, up.flip(1), torch.arange(L)[:, None].repeat(1, 2)])
    args = _args(L, Z, flags=flags)
    with torch.no_grad():
        got = mpvae.PairPredictor(r, pairs, args)(fx)
        marg = mpvae.predict_exact(fx, r, args)
    P = up.shape[0]
    assert torch.equal(got[:, :P], got[:, P:2 * P])
    assert torch.equal(got[:, 2 * P:], marg)
    m64 = XO.marginal(fx, r)
    pi, pj = m64[:, up[:, 0]], m64[:, up[:, 1]]
    g = got[:, :P].double().cpu()
    ulp = torch.from_numpy(np.spacing(g.float().numpy()).astype(np.float64))
    assert bool((g <= torch.minimum(pi, pj) + ulp).all())
    assert bool((g >= torch.clamp(pi + pj - 1.0, min=0.0) - ulp).all())


def test_kernel_returns_nan_for_pairs_out_of_range():
    """The host refuses such pairs; the kernels bounds-check anyway and write NaN instead of reading past R or fx_out."""
    from mpvae_b200 import _lib
    from mpvae_b200.probit import _ptr, predictive_scale
    B, L, Z = 4, 10, 6
    fx, r = _inputs(B, L, Z, seed=2)
    r = r.float().contiguous()
    lib = _lib.lib()
    with torch.no_grad():
        scale = predictive_scale(r)
        pairs = torch.tensor([[0, 1], [0, L], [-1, 2], [3, 3], [1 << 30, 0]], dtype=torch.int32, device=DEV)
        rho = torch.zeros(5, dtype=torch.float64, device=DEV)
        out = torch.zeros(B, 5, device=DEV)
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(lib.mpvae_predictive_rho(_ptr(r), L, Z, _ptr(scale), _ptr(pairs), 5, _ptr(rho), s), "rho")
        _lib.check(lib.mpvae_predict_pairs(_ptr(fx), B, L, _ptr(scale), _ptr(pairs), _ptr(rho), 5, 0, _ptr(out), s), "pairs")
        torch.cuda.synchronize()
    bad = torch.tensor([False, True, True, False, True])
    assert torch.isnan(rho.cpu()[bad]).all() and torch.isfinite(rho.cpu()[~bad]).all()
    assert torch.isnan(out.cpu()[:, bad]).all() and torch.isfinite(out.cpu()[:, ~bad]).all()


@pytest.mark.parametrize("L,Z,flags", [(38, 38, 0), (983, 983, 0), (3993, 10, STABLE), (131, 7, 0)])
def test_results_do_not_depend_on_batching_or_repetition(L, Z, flags, monkeypatch):
    """Rows scored alone, in windows of 7 or all at once give the same bits; so do a second call and a call with
    MPVAE_POISON_WORKSPACE=1 (outputs start as NaN: every element is written)."""
    from mpvae_b200 import mpvae
    N = 40
    fx, r = _inputs(N, L, Z, seed=L)
    pairs = _pairs_with_extras(L, n_random=300, seed=1)
    args = _args(L, Z, flags=flags)
    with torch.no_grad():
        pp = mpvae.PairPredictor(r, pairs, args)
        full, full_p = mpvae.predict_exact(fx, r, args), pp(fx)
        alone = torch.cat([mpvae.predict_exact(fx[i:i + 1], r, args) for i in range(N)])
        alone_p = torch.cat([pp(fx[i:i + 1]) for i in range(N)])
        win = torch.cat([mpvae.predict_exact(fx[i:i + 7], r, args) for i in range(0, N, 7)])
        win_p = torch.cat([pp(fx[i:i + 7]) for i in range(0, N, 7)])
        again, again_p = mpvae.predict_exact(fx, r, args), mpvae.PairPredictor(r, pairs, args)(fx)
        monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
        poisoned, poisoned_p = mpvae.predict_exact(fx, r, args), mpvae.PairPredictor(r, pairs, args)(fx)
    for a in (alone, win, again, poisoned):
        assert torch.equal(a, full)
    for a in (alone_p, win_p, again_p, poisoned_p):
        assert torch.equal(a, full_p)
    assert torch.isfinite(full).all() and torch.isfinite(full_p).all()


def test_launch_counts_and_empty_batches():
    """probit.predict_exact and PairPredictor.__call__: one launch per batch; mpvae.predict_exact: the scale pass plus
    one; PairPredictor(): the scale and rho passes.  B = 0 launches nothing."""
    from mpvae_b200 import _lib, mpvae, probit
    L, Z = 983, 983
    fx, r = _inputs(16, L, Z, seed=1)
    args = _args(L, Z)
    pairs = mpvae.all_pairs(40)
    with torch.no_grad():
        counts = []
        for fn in (lambda: probit.predictive_scale(r.float()),
                   lambda: mpvae.predict_exact(fx, r, args),
                   lambda: mpvae.PairPredictor(r, pairs, args)):
            n0 = _lib.launch_count()
            res = fn()
            counts.append(_lib.launch_count() - n0)
        pp, scale = res, probit.predictive_scale(r.float())
        n0 = _lib.launch_count()
        probit.predict_exact(fx, scale)
        pp(fx)
        counts.append(_lib.launch_count() - n0)
        n0 = _lib.launch_count()
        e0 = mpvae.predict_exact(fx[:0], r, args)
        p0 = pp(fx[:0])
        assert _lib.launch_count() - n0 == 0
        assert e0.shape == (0, L) and p0.shape == (0, pairs.shape[0])
    torch.cuda.synchronize()
    assert counts == [1, 2, 2, 2], counts


def test_does_not_consume_noise_offsets():
    """predict_exact draws no noise: the module's offset counter does not move (predict's does)."""
    from mpvae_b200 import mpvae
    L, Z = 38, 38
    fx, r = _inputs(8, L, Z)
    args = orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9)
    mpvae.set_noise_seed(77, offset=3)
    with torch.no_grad():
        mpvae.predict_exact(fx, r, args)
        assert mpvae._state["offset"] == 3
        mpvae.predict(fx, r, args)
        assert mpvae._state["offset"] == 4


def test_scoring_a_trained_model():
    """The setup of test_predict_gpu.py::test_label_free_scoring_of_a_trained_model.  predict_proba with
    predict_fn=predict_exact and infer.predict_pairs (with the diagonal) agree under the same torch seed, and the metric
    sweep of the exact predictions lies within Monte-Carlo tolerance of that of predict at S = 10 000."""
    from mpvae_b200 import metrics, mpvae
    from mpvae_b200.infer import predict_pairs, predict_proba
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    from tests.test_predict_gpu import _yeast_args, _yeast_data
    args = _yeast_args()
    x, y = _yeast_data(1500)
    n_train, n_valid = int(1500 * 0.7), int(1500 * 0.2)
    np.random.seed(4); torch.manual_seed(0)
    vae = mpvae.VAE(args).to(DEV)
    opt = torch.optim.Adam(vae.parameters(), lr=1e-3, weight_decay=1e-5)
    sched = torch.optim.lr_scheduler.StepLR(opt, 9 * 5, 0.5)
    step = DataParallelStep(vae, opt, sched, args, clip_norm=100.0)
    for _ in range(6):
        train_one_epoch(step, x[:n_train], y[:n_train], 128, torch.randperm(n_train, device=DEV))
    xv, yv = x[n_train:n_train + n_valid], y[n_train:n_train + n_valid]
    vae._reparameterize = lambda mu, logvar: mu       # score on the posterior mean: both paths see the same fx_out
    exact, sums = predict_proba(vae, xv, None, args, batch_size=128, predict_fn=mpvae.predict_exact)
    assert sums is None and exact.shape == (n_valid, 14)
    pairs = torch.cat([mpvae.all_pairs(14), torch.arange(14)[:, None].repeat(1, 2)])
    pp = predict_pairs(vae, xv, pairs, args, batch_size=128)
    assert pp.shape == (n_valid, pairs.shape[0])
    assert torch.equal(pp[:, -14:], exact)
    a_mc = copy.copy(args)
    a_mc.n_test_sample = 10_000
    mc, _ = predict_proba(vae, xv, None, a_mc, batch_size=128)
    assert (mc - exact).abs().max().item() <= 6 * 0.5 / np.sqrt(10_000)
    thresholds = [0.05 * i for i in range(1, 20)]
    for me, mm in zip(metrics.sweep_metrics(exact, yv, thresholds), metrics.sweep_metrics(mc, yv, thresholds)):
        for key, v in me.items():
            if v.dim() != 0:
                continue
            a, b = float(v), float(mm[key])
            if not (np.isnan(a) and np.isnan(b)):      # a label absent from the rows has no AUC either way
                assert abs(a - b) <= 0.02, (key, a, b)
