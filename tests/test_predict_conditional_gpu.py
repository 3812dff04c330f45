"""GPU: conditional prediction (mpvae_probit_predict_conditional: the nt product, then probit_cond_loglik_kernel,
probit_cond_weights_kernel and probit_cond_predict_kernel) against predict with nothing observed or R = 0, against the
loss's nll_x with everything observed, against the oracle and the closed form, on a planted model, under batching,
repetition and a poisoned workspace, by launch count, and at the model level through infer.predict_conditional."""
import copy

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import predict_conditional_oracle as CO
from tests import predict_exact_oracle as XO
from tests.test_predict_gpu import EQUALITY_CASES, _args, _inputs, _yeast_args, _yeast_data

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

STABLE, FMA, TENSOR, SEPARATE, FUSED = 0x8, 0x4, 0x2, 0x20, 0x10


def _none(B, L):
    return torch.full((B, L), -1, dtype=torch.int8, device=DEV)


def _random_obs(B, L, seed, max_obs=16, y=None):
    """Mixed patterns: row 0 observes nothing, row 1 everything (when B > 1), the others up to max_obs labels."""
    g = torch.Generator().manual_seed(seed)
    obs = torch.full((B, L), -1, dtype=torch.int8)
    vals = (torch.rand(B, L, generator=g) < 0.3).to(torch.int8) if y is None else y.cpu().to(torch.int8)
    for b in range(B):
        if b == 0:
            continue
        if b == 1:
            obs[b] = vals[b]
            continue
        k = int(torch.randint(1, max_obs + 1, (1,), generator=g))
        idx = torch.randperm(L, generator=g)[:min(k, L)]
        obs[b, idx] = vals[b, idx]
    return obs.to(DEV)


def _cond(t, obs, args, noise=None):
    from mpvae_b200.mpvae import predict_conditional
    with torch.no_grad():
        out = predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, args, noise=noise)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("S,B,L,Z,flags,external", EQUALITY_CASES)
def test_nothing_observed_is_predict(S, B, L, Z, flags, external):
    """No observed label: lp = 0, u = 1, fse = S -- predict's indiv_prob bit for bit, log_evidence = 0, ess = S."""
    from mpvae_b200.mpvae import predict
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        want = predict(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
    got = _cond(t, _none(B, L), args, noise)
    assert torch.equal(got.prob, want)
    assert torch.equal(got.log_evidence, torch.zeros(B, device=DEV))
    assert torch.equal(got.ess, torch.full((B,), float(S), device=DEV))


@pytest.mark.parametrize("S,B,L,Z,flags,external", [(100, 37, 81, 81, 0, False), (10, 33, 983, 10, 0, True),
                                                    (10, 70, 983, 983, 0, False), (10, 40, 257, 300, STABLE, False)])
def test_zero_r_gives_predict_on_the_unobserved_cells(S, B, L, Z, flags, external):
    """R = 0: all samples are the same, so u = 1 whatever is observed."""
    from mpvae_b200.mpvae import predict
    t, noise = _inputs(S, B, L, Z, external, seed=11)
    t["r_sqrt_sigma"] = torch.zeros_like(t["r_sqrt_sigma"])
    args = _args(S, L, Z, flags)
    obs = _random_obs(B, L, seed=3)
    with torch.no_grad():
        want = predict(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
    got = _cond(t, obs, args, noise)
    free = (obs != 0) & (obs != 1)
    assert torch.equal(got.prob[free], want[free])
    assert torch.equal(got.prob[~free], obs[~free].float())
    assert torch.equal(got.ess, torch.full((B,), float(S), device=DEV))


# (S, B, L, Z, flags, external): CUDA-core, dense (one-row batches need CONTRACT_TENSOR or S >= 128), small shapes, STABLE
ALL_OBSERVED = [(10, 9, 983, 10, 0, False), (3, 5, 3993, 10, 0, True), (10, 6, 983, 983, TENSOR, False),
                (128, 4, 300, 256, 0, False), (100, 8, 81, 81, 0, False), (10, 7, 38, 38, 0, True),
                (10, 6, 257, 300, STABLE, False), (10, 5, 38, 38, STABLE, True)]


@pytest.mark.parametrize("S,B,L,Z,flags,external", ALL_OBSERVED)
def test_everything_observed_is_the_loss_nll_x(S, B, L, Z, flags, external):
    """Every label observed: lp is the loss forward's lp_x, so for a one-row batch -log_evidence is compute_loss's
    nll_loss_x bit for bit (the global-row keys of the batch passed in); over the whole batch the mean of -log_evidence
    is within one fp32 ulp of nll_loss_x.  Observed cells return exactly 0 / 1."""
    from mpvae_b200.mpvae import compute_loss
    t, noise = _inputs(S, B, L, Z, external, seed=5 * S + L)
    y = t["y"]
    obs = y.to(torch.int8)
    args = _args(S, L, Z, flags, dp_global_batch=B, dp_row0=0)
    got = _cond(t, obs, args, noise)
    assert torch.equal(got.prob, y)
    assert bool(((got.ess >= 1) & (got.ess <= S)).all())
    with torch.no_grad():
        full = compute_loss(y, t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                            t["r_sqrt_sigma"], args, noise=noise)[2]
    mean = float((-got.log_evidence.double()).mean())
    assert abs(mean - float(full)) <= float(np.spacing(np.float32(abs(float(full))))), (mean, float(full))
    for b in range(B):
        rows = {k: (v if k == "r_sqrt_sigma" else v[b:b + 1]) for k, v in t.items()}
        a1 = _args(S, L, Z, flags, dp_global_batch=B, dp_row0=b)
        nz = noise[:, b:b + 1] if noise is not None else None
        with torch.no_grad():
            nll_x = compute_loss(rows["y"], rows["fe_out"], rows["fe_mu"], rows["fe_logvar"], rows["fx_out"], rows["fx_mu"],
                                 rows["fx_logvar"], rows["r_sqrt_sigma"], a1, noise=nz)[2]
        one = _cond(rows, obs[b:b + 1], a1, nz)
        assert torch.equal(-one.log_evidence[0], nll_x), (b, float(-one.log_evidence[0]), float(nll_x))
        assert torch.equal(one.log_evidence[0], got.log_evidence[b])


@pytest.mark.parametrize("S,B,L,Z,flags", [(100, 37, 81, 81, 0), (10, 33, 983, 10, 0), (10, 20, 983, 983, 0),
                                           (7, 19, 130, 64, TENSOR), (10, 16, 38, 38, STABLE), (10, 12, 257, 300, STABLE)])
def test_against_the_oracle(S, B, L, Z, flags):
    """External noise, mixed observation patterns (none, all, up to 16 labels), L not a multiple of 4 or 128."""
    t, noise = _inputs(S, B, L, Z, True, seed=2 * S + L)
    obs = _random_obs(B, L, seed=B + L)
    got = _cond(t, obs, _args(S, L, Z, flags), noise)
    with torch.no_grad():
        prob, le, ess = CO.predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, noise, stable=bool(flags & STABLE))
    dp = float((got.prob.double() - prob.double()).abs().max())
    dle = float(((got.log_evidence.double() - le.double()).abs() / le.double().abs().clamp_min(1.0)).max())
    dess = float(((got.ess.double() - ess.to(DEV)).abs() / ess.to(DEV)).max())
    assert dp <= 1e-5 and dle <= 1e-5 and dess <= 1e-4, (dp, dle, dess)


@pytest.mark.parametrize("y_o", [0, 1])
def test_one_observed_label_converges_to_the_closed_form(y_o):
    """S = 10 000, one observed label o: P(y_u = 1 | y_o) from PairPredictor and predict_exact.  Every cell within
    6 / sqrt(ess) (a conservative bound of a self-normalised mean of values in [0, 1]); the mean signed error over all
    cells within 4 standard errors of 0."""
    from mpvae_b200 import mpvae
    S, B, L, Z = 10_000, 64, 40, 8
    t, _ = _inputs(2, B, L, Z, False, seed=21)
    g = torch.Generator().manual_seed(5)
    t["r_sqrt_sigma"] = (torch.randn(L, Z, generator=g, dtype=torch.float64) * 0.6).to(DEV)
    o = 7
    obs = _none(B, L)
    obs[:, o] = y_o
    args = orc.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=31, noise_offset=2)
    got = _cond(t, obs, args)
    with torch.no_grad():
        pairs = torch.tensor([[u, o] for u in range(L)])
        P_uo = mpvae.PairPredictor(t["r_sqrt_sigma"], pairs, args)(t["fx_out"]).double()
        P_u = mpvae.predict_exact(t["fx_out"], t["r_sqrt_sigma"], args).double()
    P_o = P_u[:, o:o + 1]
    want = P_uo / P_o if y_o == 1 else (P_u - P_uo) / (1 - P_o)
    free = [u for u in range(L) if u != o]
    err = (got.prob.double() - want)[:, free]
    bound = 6.0 / torch.sqrt(got.ess.double())[:, None]
    assert bool((err.abs() <= bound).all()), float((err.abs() / bound).max())
    # the cells of a row share its samples, so their errors are correlated: the standard error of a row's summed error
    # is the delta-method one of the self-normalised mean of F_s = sum_u E_{s,u} (the oracle's samples on the same
    # noise); rows are independent
    noise = mpvae.draw_noise(args, S, B, DEV)
    E, u, _, _, _ = CO.samples(t["fx_out"], t["r_sqrt_sigma"], obs, noise)
    F, u = E[:, :, free].double().sum(2), u.double()
    Fbar = (u * F).sum(0) / u.sum(0)
    se_row = torch.sqrt((u * u * (F - Fbar) ** 2).sum(0)) / u.sum(0)
    z = float(err.sum() / torch.sqrt((se_row * se_row).sum()))
    assert abs(z) <= 4.0, z
    assert torch.equal(got.prob[:, o], torch.full((B,), float(y_o), device=DEV))


def test_planted_model_conditional_beats_the_marginals():
    """Labels drawn from the model itself (Z = 2, loadings around +-1.5) and half of each row observed: the log-loss of
    predict_conditional on the hidden labels beats predict_exact's marginals by more than 5 standard errors of the
    paired difference (the true conditional is the Bayes predictor, Gibbs' inequality).  With R = 0 the two agree (mean
    log-loss within 1e-4 relative)."""
    from mpvae_b200 import mpvae
    S, B, L, Z = 1000, 512, 24, 2
    g = torch.Generator().manual_seed(8)
    fx = (torch.randn(B, L, generator=g) * 0.7).to(DEV)
    signs = torch.where(torch.rand(L, Z, generator=g) < 0.5, -1.0, 1.0)
    r = (signs * (1.5 + 0.2 * torch.randn(L, Z, generator=g))).double().to(DEV)
    eps = torch.randn(B, Z, generator=g).to(DEV)
    p_true = XO.C_EPS + XO.K_EPS * torch.special.ndtr((fx + eps @ r.float().T).double())
    y = (torch.rand(B, L, generator=g).to(DEV).double() < p_true).to(torch.int8)
    hide = torch.rand(B, L, generator=g).to(DEV) < 0.5
    obs = torch.where(hide, torch.full_like(y, -1), y)
    args = orc.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=3, noise_offset=1)

    def losses(rr):
        t = {"fx_out": fx, "r_sqrt_sigma": rr}
        pc = _cond(t, obs, args).prob.double().clamp(1e-7, 1 - 1e-7)
        with torch.no_grad():
            pm = mpvae.predict_exact(fx, rr, args).double().clamp(1e-7, 1 - 1e-7)
        yy = y.double()
        ll = lambda p: -(yy * torch.log(p) + (1 - yy) * torch.log(1 - p))
        return ll(pc)[hide], ll(pm)[hide]

    lc, lm = losses(r)
    d = lm - lc
    gain, se = float(d.mean()), float(d.std() / np.sqrt(d.numel()))
    assert gain > 5 * se, (gain, se, float(lc.mean()), float(lm.mean()))
    # R = 0: the weights are all 1, so the conditional is predict's plain mean of S identical E, which carries the fp32
    # running sum's rounding (up to ~1e-4 relative at S = 1000) against the closed form
    lc0, lm0 = losses(torch.zeros_like(r))
    assert abs(float(lc0.mean() - lm0.mean())) <= 1e-4 * float(lm0.mean()), (float(lc0.mean()), float(lm0.mean()))


@pytest.mark.parametrize("S,L,Z,flags,windows", [
    (100, 81, 81, 0, [(0, 1), (1, 64), (64, 100)]),                 # small shapes (CUDA-core product)
    (10, 983, 10, 0, [(0, 37), (37, 38), (38, 100)]),               # CUDA-core regime
    (10, 983, 983, TENSOR, [(0, 5), (5, 61), (61, 100)]),           # dense regime
])
def test_rows_do_not_depend_on_batching(S, L, Z, flags, windows):
    from mpvae_b200.mpvae import predict_conditional
    N = windows[-1][1]
    t, _ = _inputs(S, N, L, Z, False, seed=N + L)
    obs = _random_obs(N, L, seed=4)
    with torch.no_grad():
        full = predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, _args(S, L, Z, flags, dp_global_batch=N, dp_row0=0))
        parts = [predict_conditional(t["fx_out"][lo:hi], t["r_sqrt_sigma"], obs[lo:hi],
                                     _args(S, L, Z, flags, dp_global_batch=N, dp_row0=lo)) for lo, hi in windows]
    for i in range(3):
        assert torch.equal(torch.cat([p[i] for p in parts], 0), full[i])


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (100, 33, 81, 81, 0), (10, 33, 983, 10, 0),
                                           (10, 128, 983, 983, 0), (3, 77, 130, 256, SEPARATE),
                                           (10, 40, 257, 300, STABLE)])
def test_repeatable_poison_proof_and_state_values(S, B, L, Z, flags, monkeypatch):
    """Two runs give the same bits; so does a workspace and output poisoned with 0xFF bytes; and the unobserved states
    2 and -7 give the bits of -1."""
    t, _ = _inputs(S, B, L, Z, False, seed=S + L)
    obs = _random_obs(B, L, seed=9)
    args = _args(S, L, Z, flags)
    a = _cond(t, obs, args)
    b = _cond(t, obs, args)
    odd = obs.clone()
    free = (obs != 0) & (obs != 1)
    odd[free] = torch.where(torch.rand(int(free.sum()), device=DEV) < 0.5, 2, -7).to(torch.int8)
    c = _cond(t, odd, args)
    monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
    d = _cond(t, obs, args)
    for other in (b, c, d):
        for i in range(3):
            assert torch.equal(a[i], other[i])
    assert torch.isfinite(a.prob).all()


def test_empty_batch_and_offset_consumption():
    """B == 0 gives empty outputs; without args.noise_offset a call consumes one offset, as predict does, and with the
    same offset it uses predict's noise."""
    from mpvae_b200 import mpvae
    L, Z = 14, 14
    args = orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9)
    with torch.no_grad():
        out = mpvae.predict_conditional(torch.empty(0, L, device=DEV), torch.zeros(L, Z, dtype=torch.float64, device=DEV),
                                        _none(0, L), args)
    assert out.prob.shape == (0, L) and out.log_evidence.shape == (0,) and out.ess.shape == (0,)
    t, _ = _inputs(10, 8, L, Z, False, seed=1)
    none = _none(8, L)
    mpvae.set_noise_seed(77, offset=3)
    with torch.no_grad():
        a = mpvae.predict_conditional(t["fx_out"], t["r_sqrt_sigma"], none, args).prob
        b = mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], args)
        c = mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9,
                                                                         noise_offset=3))
        d = mpvae.predict_conditional(t["fx_out"], t["r_sqrt_sigma"], none,
                                      orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9, noise_offset=4)).prob
    assert torch.equal(a, c) and torch.equal(b, d) and not torch.equal(a, b)


@pytest.mark.parametrize("S,B,L,Z,flags,external,small", [
    (100, 128, 81, 81, 0, False, True), (10, 16, 38, 38, 0, True, True),
    (10, 33, 3993, 10, 0, False, False), (10, 33, 3993, 10, 0, True, False),
    (10, 70, 983, 983, 0, False, False), (10, 70, 983, 983, 0, True, False), (10, 70, 983, 983, SEPARATE, False, False),
])
def test_launch_count(S, B, L, Z, flags, external, small):
    """predict's launches up to and including the product, then the three row passes (log-likelihood, weights,
    weighted mean).  Where predict runs the one-launch small kernel, the product is the CUDA-core path's: the Philox
    kernel (library noise) and the FMA product."""
    from mpvae_b200 import _lib
    from mpvae_b200.mpvae import predict, predict_conditional
    t, noise = _inputs(S, B, L, Z, external, seed=5)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        n0 = _lib.launch_count()
        predict(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
        n1 = _lib.launch_count()
        predict_conditional(t["fx_out"], t["r_sqrt_sigma"], _none(B, L), args, noise=noise)
        n2 = _lib.launch_count()
    torch.cuda.synchronize()
    n_pred, n_cond = n1 - n0, n2 - n1
    if small:
        assert n_pred == 1 and n_cond == (1 if external else 2) + 3, (n_pred, n_cond)
    else:
        assert n_cond == n_pred - 1 + 3, (n_pred, n_cond)


def test_conditional_scoring_of_a_trained_model():
    """The yeast-shaped setup of test_label_free_scoring_of_a_trained_model: infer.predict_conditional equals the hand
    loop bit for bit; with nothing observed its prob is predict_proba(labels=None)'s under the same torch seed; ess is
    in [1, S]."""
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_conditional, predict_proba
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    args = _yeast_args()
    x, y = _yeast_data(1500)
    n_train, n_valid = int(1500 * 0.7), int(1500 * 0.2)
    np.random.seed(4); torch.manual_seed(0)
    vae = VAE(args).to(DEV)
    opt = torch.optim.Adam(vae.parameters(), lr=1e-3, weight_decay=1e-5)
    sched = torch.optim.lr_scheduler.StepLR(opt, 9 * 5, 0.5)
    step = DataParallelStep(vae, opt, sched, args, clip_norm=100.0)
    for _ in range(12):
        train_one_epoch(step, x[:n_train], y[:n_train], 128, torch.randperm(n_train, device=DEV))
    xv, yv = x[n_train:n_train + n_valid], y[n_train:n_train + n_valid]
    mask = torch.rand(yv.shape, generator=torch.Generator().manual_seed(2)).to(DEV) < 0.5
    obs = torch.where(mask, yv.to(torch.int8), -1)
    torch.manual_seed(11)
    prob, le, ess = predict_conditional(vae, xv, obs, args, batch_size=128)
    assert prob.shape == (n_valid, 14) and le.shape == ess.shape == (n_valid,)
    vae.eval()
    a_t = copy.copy(args)
    a_t.mode = "test"
    hand = []
    torch.manual_seed(11)
    with torch.no_grad():
        for lo in range(0, n_valid, 128):
            hi = min(lo + 128, n_valid)
            a_t.dp_global_batch, a_t.dp_row0, a_t.noise_offset = n_valid, lo, 0
            hand.append(mpvae.predict_conditional(vae.feat_forward(xv[lo:hi])[0], vae.r_sqrt_sigma, obs[lo:hi], a_t))
    for i, got in enumerate((prob, le, ess)):
        assert torch.equal(torch.cat([h[i] for h in hand], 0), got)
    assert bool(((ess >= 1) & (ess <= args.n_test_sample)).all())
    vae.train()
    torch.manual_seed(11)
    none, _, _ = predict_conditional(vae, xv, torch.full_like(obs, -1), args, batch_size=128)
    torch.manual_seed(11)
    free, _ = predict_proba(vae, xv, None, args, batch_size=128)
    assert torch.equal(none, free)
