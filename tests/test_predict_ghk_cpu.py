"""CPU checks of the GHK conditional prediction (mpvae_probit_predict_conditional_ghk / probit.probit_predict_conditional_ghk /
mpvae.predict_conditional_ghk / infer.predict_conditional(predict_fn=...)): the fp64 oracle's clamped truncated sampler
against its CDF, the oracle against Gauss-Hermite quadrature, the closed form and the importance oracle, its exact cases;
the C-ABI surface and its argument checks; the host-side refusals; and the data-parallel scoring loop with the oracle
injected as predict_fn."""
import ctypes as C
import math
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import probit_elbo_oracle as orc
from tests import helpers as H
from tests import predict_conditional_oracle as CO
from tests import predict_exact_oracle as XO
from tests import predict_ghk_oracle as GO
from tests import predict_oracle as PO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


def _case(S, B, L, Z, seed, sigma=1.0, fx_scale=1.5):
    g = torch.Generator().manual_seed(seed)
    fx = torch.randn(B, L, generator=g) * fx_scale
    r = torch.randn(L, Z, generator=g, dtype=torch.float64) * sigma / np.sqrt(Z)
    xi = torch.randn(S, B, Z, generator=g)
    zeta = torch.randn(S, B, L, generator=g)
    U = torch.rand(S, B, L, generator=g, dtype=torch.float64).clamp(1e-12, 1 - 1e-12)
    return fx, r, xi, zeta, U


def _observe(B, L, frac, seed, y=None):
    g = torch.Generator().manual_seed(seed)
    vals = (torch.rand(B, L, generator=g) < 0.4).to(torch.int8) if y is None else y.to(torch.int8)
    keep = torch.rand(B, L, generator=g) < frac
    return torch.where(keep, vals, torch.full_like(vals, -1))


@pytest.mark.parametrize("y", [0, 1])
def test_sampler_inverts_its_cdf_on_the_correct_side(y):
    """eta = F_y^-1(U) for a in [-38, 38]: finite, F_y(eta) = U (relative to the smaller of U, 1 - U), and on y's side
    of a exactly when U falls in that side's share of the mass."""
    from scipy.special import ndtr
    a = torch.linspace(-38.0, 38.0, 153, dtype=torch.float64)[:, None]
    U = torch.cat([torch.tensor([1e-7, 1e-4, 0.01]), torch.linspace(0.05, 0.95, 19),
                   torch.tensor([0.99, 1 - 1e-4, 1 - 1e-7])]).double()[None, :]
    a, U = torch.broadcast_tensors(a, U)
    eta, Z = GO.draw(a, y, U)
    assert bool(torch.isfinite(eta).all())
    an, en, un = a.numpy(), eta.numpy(), U.numpy()
    F = GO.cdf(en, an, y)
    tail = np.minimum(un, 1 - un)
    err = np.abs(np.where(un <= 0.5, F - un, (1 - F) - (1 - un))) / tail
    # where the side's share of the mass is below fp64's resolution near 1 the draw is pinned to the boundary
    share = (GO.C_EPS + GO.K_EPS) * (ndtr(-an) if y else ndtr(an)) / (Z.numpy())
    resolvable = (share > 1e-12) & (share < 1 - 1e-12)
    assert np.all(err[resolvable | (np.abs(an) < 30)] < 1e-6), float(err.max())
    on_side = en >= an if y else en <= an
    want_side = (1 - un) < share if y else un < share
    clear = np.abs(np.where(y, 1 - un, un) - share) > 1e-9 * np.maximum(share, 1e-300)
    assert np.array_equal(on_side[clear & resolvable], want_side[clear & resolvable])
    Zw = GO.C_EPS + GO.K_EPS * (ndtr(-an) if y else ndtr(an))
    assert np.allclose(Z.numpy(), Zw, rtol=1e-12, atol=0)


@pytest.mark.parametrize("Z", [1, 2])
def test_oracle_matches_quadrature_with_most_labels_observed(Z):
    """Z = 1, 2 and L = 20 with ~80 % observed: evidence and conditional marginals within 6 SE of Gauss-Hermite."""
    S, B, L = 4000, 3, 20
    fx, r, xi, zeta, U = _case(S, B, L, Z, seed=10 + Z, sigma=1.5, fx_scale=1.0)
    obs = _observe(B, L, 0.8, seed=Z)
    prob, le, ess = GO.predict_conditional_ghk(fx, r, obs, xi, zeta, U)
    se_p, se_le = GO.stderr(fx, r, obs, xi, zeta, U)
    qp, qle = GO.quadrature(fx, r, obs)
    assert bool((ess > 0.05 * S).all()), ess
    assert bool(((le - qle).abs() <= 6 * se_le).all()), (le, qle, se_le)
    free = (obs != 0) & (obs != 1)
    assert bool(((prob - qp).abs()[free] <= 6 * se_p[free] + 1e-12).all())
    assert torch.equal(prob[~free], qp[~free])


def test_oracle_with_one_observed_label_is_the_closed_form():
    """|O| = 1: every sample has the weight c + k Phi(+-fx_o / sqrt(1 + |R_o|^2)) (ess = S, log_evidence its log); the
    unobserved cells converge to P(y_l = 1, y_o = 1) / P(y_o = 1) of the closed form."""
    S, B, L, Z = 20000, 2, 7, 3
    fx, r, xi, zeta, U = _case(S, B, L, Z, seed=5)
    obs = torch.full((B, L), -1, dtype=torch.int8)
    obs[0, 2], obs[1, 5] = 1, 0
    prob, le, ess = GO.predict_conditional_ghk(fx, r, obs, xi, zeta, U)
    se_p, _ = GO.stderr(fx, r, obs, xi, zeta, U)
    marg = XO.marginal(fx, r)
    assert torch.allclose(ess, torch.full((B,), float(S), dtype=torch.float64), rtol=1e-12)
    assert abs(float(le[0]) - math.log(float(marg[0, 2]))) < 1e-12
    assert abs(float(le[1]) - math.log(1 - float(marg[1, 5]))) < 1e-12
    for b, o, yo in ((0, 2, 1), (1, 5, 0)):
        pairs = torch.tensor([[l, o] for l in range(L) if l != o])
        joint = torch.from_numpy(np.asarray(XO.pair_prob(fx[b:b + 1], r, pairs))).double().reshape(-1)
        pl = marg[b, pairs[:, 0]]
        want = joint / marg[b, o] if yo else (pl - joint) / (1 - marg[b, o])
        got = prob[b, pairs[:, 0]]
        assert bool(((got - want).abs() <= 6 * se_p[b, pairs[:, 0]] + 1e-9).all()), (b, got, want)


def test_oracle_agrees_with_the_importance_oracle_at_large_s():
    """Few observed labels, S = 20000: the two estimators of the same conditional agree within their SEs."""
    S, B, L, Z = 20000, 3, 12, 4
    fx, r, xi, zeta, U = _case(S, B, L, Z, seed=8)
    obs = _observe(B, L, 0.25, seed=4)
    prob, le, _ = GO.predict_conditional_ghk(fx, r, obs, xi, zeta, U)
    se_p, se_le = GO.stderr(fx, r, obs, xi, zeta, U)
    xi2 = torch.randn(S, B, Z, generator=torch.Generator().manual_seed(99))
    iprob, ile, _ = CO.predict_conditional(fx, r, obs, xi2)
    ise = CO.stderr(fx, r, obs, xi2)
    tol = 6 * torch.sqrt(se_p ** 2 + ise ** 2) + 1e-6
    assert bool(((prob - iprob.double()).abs() <= tol).all())
    assert bool(((le - ile.double()).abs() <= 6 * se_le + 0.01).all())


def test_oracle_exact_cases():
    """O empty: lw = 0, x = n (prob = predict's mean of E, ess = S); R = 0: C = I and constant weights
    prod (c + k Phi(+-fx_o)), the unobserved cells are predict's mean of E."""
    S, B, L, Z = 40, 4, 9, 3
    fx, r, xi, zeta, U = _case(S, B, L, Z, seed=3)
    none = torch.full((B, L), -1, dtype=torch.int8)
    prob, le, ess = GO.predict_conditional_ghk(fx, r, none, xi, zeta, U)
    assert torch.allclose(prob, PO.predict(fx, r, xi).double(), atol=1e-6, rtol=0)
    assert torch.equal(le, torch.zeros(B, dtype=torch.float64))
    assert torch.equal(ess, torch.full((B,), float(S), dtype=torch.float64))
    r0 = torch.zeros_like(r)
    obs = _observe(B, L, 0.6, seed=9)
    prob, le, ess = GO.predict_conditional_ghk(fx, r0, obs, xi, zeta, U)
    free = (obs != 0) & (obs != 1)
    assert torch.allclose(ess, torch.full((B,), float(S), dtype=torch.float64), rtol=1e-12)
    P = GO.C_EPS + GO.K_EPS * torch.special.ndtr(fx.double())
    cell = torch.where(obs == 1, P, torch.where(obs == 0, 1 - P, torch.ones_like(P)))
    assert torch.allclose(le, torch.log(cell).sum(1), rtol=1e-12, atol=1e-12)
    assert torch.allclose(prob[free], P[free], rtol=1e-12, atol=0)


# ---- the C-ABI surface ----

def test_abi_surface(lib):
    from mpvae_b200 import _lib
    assert hasattr(lib, "mpvae_probit_predict_conditional_ghk") and hasattr(lib, "mpvae_ghk_workspace_bytes")
    assert "mpvae_probit_predict_conditional_ghk" in _lib.EXPORTS and "mpvae_ghk_workspace_bytes" in _lib.EXPORTS
    assert _lib.ABI_VERSION == 13 and lib.mpvae_abi_version() == 13
    ws = lib.mpvae_ghk_workspace_bytes
    assert ws(100, 8, 300, 64, 0, 0) < ws(100, 8, 300, 64, 30, 0) < ws(100, 8, 300, 64, 300, 0)
    assert ws(100, 8, 300, 64, 30, 0) < ws(100, 16, 300, 64, 30, 0)
    assert ws(100, 8, 300, 64, 301, 0) == 256 and ws(100, 8, 300, 64, -1, 0) == 256 and ws(0, 8, 300, 64, 3, 0) == 256
    # the existing workspace is unchanged
    assert lib.mpvae_workspace_bytes(100, 8, 300, 64, 0, 0) == lib.mpvae_workspace_bytes(100, 8, 300, 64, 0, 0)


def test_abi_refuses_bad_arguments(lib):
    from mpvae_b200 import _lib
    f = lib.mpvae_probit_predict_conditional_ghk
    p = _lib.ProbitParams()
    p.struct_bytes = C.sizeof(_lib.ProbitParams)
    p.S, p.B, p.L, p.Z = 4, 4, 9, 3
    p.fx_out, p.r, p.workspace, p.indiv_prob = 256, 256, 256, 256
    p.noise_b_global, p.noise_row0 = 4, 0
    p.workspace_bytes = 1 << 40
    need = lib.mpvae_ghk_workspace_bytes(4, 4, 9, 3, 5, 0)

    def call(observed=256, gws=256, gbytes=need, mo=5, le=256, ess=256):
        return f(C.byref(p), observed, None, None, None, gws, gbytes, mo, le, ess, None)

    for kw in ({"observed": None}, {"gws": None}, {"le": None}, {"ess": None}):
        assert call(**kw) == 1
        assert b"observed/log_evidence/ess/ghk_ws" in lib.mpvae_last_error()
    for mo in (-1, 10):
        assert call(mo=mo) == 1
        assert b"max_observed" in lib.mpvae_last_error()
    assert call(gbytes=need - 1) == 1
    assert b"ghk workspace too small for max_observed=5" in lib.mpvae_last_error()
    assert call(mo=6) == 1
    assert b"ghk workspace too small for max_observed=6" in lib.mpvae_last_error()
    assert call(gws=256 + 16) == 1
    assert b"256-byte aligned" in lib.mpvae_last_error()
    p.noise_b_global = 3
    assert call() == 1
    assert b"do not fit a global batch" in lib.mpvae_last_error()


def test_missing_symbol_asks_for_a_rebuild():
    from mpvae_b200 import _lib
    assert "mpvae_probit_predict_conditional_ghk" in _lib.EXPORTS
    src = open(os.path.join(ROOT, "mpvae-1_b200", "_lib.py")).read()
    assert "lacks symbols {missing}; rebuild" in src


class _FakeCuda:
    def __init__(self, t):
        self.shape, self.requires_grad, self.device = t.shape, False, torch.device("cuda:0")


def test_host_refusals():
    from mpvae_b200.mpvae import predict_conditional_ghk
    from mpvae_b200.probit import probit_predict_conditional_ghk
    case = H.load_golden("yeast_b16")
    t = H.to_torch(case["inputs"])
    args = orc.make_args(case["L"], case["Z"], n_test_sample=case["S"], mode="test")
    B, L = t["fx_out"].shape
    obs = torch.full((B, L), -1, dtype=torch.int8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"], obs, args)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        probit_predict_conditional_ghk(t["fx_out"], t["r_sqrt_sigma"].float(), obs, 4, 0, noise_spec=(4, 1, 0, None, 0))
    with pytest.raises(RuntimeError, match="inference only"):
        predict_conditional_ghk(t["fx_out"], torch.nn.Parameter(t["r_sqrt_sigma"]), obs, args)
    fake = _FakeCuda(t["fx_out"])
    with pytest.raises(TypeError, match="int8"):
        predict_conditional_ghk(fake, t["r_sqrt_sigma"], obs.float(), args)
    with pytest.raises(ValueError, match="shape"):
        predict_conditional_ghk(fake, t["r_sqrt_sigma"], obs[:, :-1], args)
    with pytest.raises(ValueError, match="is on"):
        predict_conditional_ghk(fake, t["r_sqrt_sigma"], obs, args)
    # the low-level wrapper: dtype and shape of the optional inputs, max_observed range (checked before any device work)
    r32 = t["r_sqrt_sigma"].float()
    with pytest.raises(ValueError, match="max_observed"):
        probit_predict_conditional_ghk(t["fx_out"], r32, obs, 4, L + 1, noise_spec=(4, 1, 0, None, 0))
    with pytest.raises(ValueError, match="gram has shape"):
        probit_predict_conditional_ghk(t["fx_out"], r32, obs, 4, 0, noise_spec=(4, 1, 0, None, 0),
                                       gram=torch.zeros(L, L + 1))
    with pytest.raises(ValueError, match="zeta has shape"):
        probit_predict_conditional_ghk(t["fx_out"], r32, obs, 4, 0, noise_spec=(4, 1, 0, None, 0),
                                       zeta=torch.zeros(4, B, L - 1))
    with pytest.raises(TypeError, match="int8"):
        probit_predict_conditional_ghk(t["fx_out"], r32, obs.to(torch.int16), 4, 0, noise_spec=(4, 1, 0, None, 0))


# ---- data-parallel GHK scoring (gloo, CPU; the oracle injected as predict_fn) ----

def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


def _score(n_rows, batch_size):
    sys.path.insert(0, ROOT)
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_conditional
    from mpvae_b200.mpvae import VAE
    torch.set_num_threads(1)
    args = _args()
    np.random.seed(4)
    torch.manual_seed(0)
    model = VAE(args)
    model._reparameterize = lambda mu, logvar: mu
    rng = np.random.RandomState(0)
    x = torch.from_numpy(rng.standard_normal((n_rows, args.feature_dim)).astype(np.float32))
    obs = torch.from_numpy(rng.randint(-1, 2, size=(n_rows, args.label_dim)).astype(np.int8))
    g = torch.Generator().manual_seed(77)
    S, L = args.n_test_sample, args.label_dim
    xi = torch.randn(S, n_rows, args.z_dim, generator=g)
    zeta = torch.randn(S, n_rows, L, generator=g)
    U = torch.rand(S, n_rows, L, generator=g, dtype=torch.float64).clamp(1e-12, 1 - 1e-12)
    seen = []

    def ghk(fx_out, r, observed, a, noise=None, gram=None):
        seen.append((a.mode, a.dp_global_batch, a.dp_row0, fx_out.shape[0]))
        lo, hi = a.dp_row0, a.dp_row0 + fx_out.shape[0]
        assert torch.equal(observed, obs[lo:hi])
        prob, le, ess = GO.predict_conditional_ghk(fx_out, r, observed, xi[:, lo:hi], zeta[:, lo:hi], U[:, lo:hi])
        return mpvae.ConditionalPrediction(prob.float(), le.float(), ess.float())

    prob, le, ess = predict_conditional(model, x, obs, args, batch_size=batch_size, predict_fn=ghk)
    assert seen and all(m == "test" and gb == n_rows for m, gb, _, _ in seen)
    return torch.cat([prob, le[:, None], ess[:, None]], 1)


def _worker(rank, world, port, n_rows, batch_size, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret[rank] = _score(n_rows, batch_size)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_ranks_ghk_equal_one_process():
    import socket
    n_rows, batch_size = 23, 12
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n_rows, batch_size, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(240)
        assert p.exitcode == 0
    want = _score(n_rows, batch_size)
    assert want.shape == (n_rows, _args().label_dim + 2)
    assert torch.equal(ret[0], want) and torch.equal(ret[1], want)
