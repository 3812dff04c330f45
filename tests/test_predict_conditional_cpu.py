"""CPU checks of conditional prediction (mpvae_probit_predict_conditional / probit.probit_predict_conditional /
mpvae.predict_conditional / infer.predict_conditional): the oracle restatement against predict's oracle, the loss's
nll_x, the closed form of one observed label and quadrature at Z = 1; the C-ABI surface and its argument checks; the
host-side refusals; and the data-parallel scoring loop with the oracle injected."""
import ctypes as C
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
from tests import predict_oracle as PO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


def _case(S, B, L, Z, seed, sigma=1.0):
    g = torch.Generator().manual_seed(seed)
    fx = torch.randn(B, L, generator=g) * 1.5
    r = torch.randn(L, Z, generator=g, dtype=torch.float64) * sigma / np.sqrt(Z)
    noise = torch.randn(S, B, Z, generator=g)
    return fx, r, noise


@pytest.mark.parametrize("stable", [False, True])
def test_oracle_with_nothing_observed_is_predict(stable):
    fx, r, noise = _case(37, 5, 11, 4, seed=1)
    obs = torch.full((5, 11), -1, dtype=torch.int8)
    obs[2, 3] = 5                                  # any value other than 0 / 1 is unobserved
    prob, le, ess = CO.predict_conditional(fx, r, obs, noise, stable=stable)
    assert torch.equal(prob, PO.predict(fx, r, noise, stable=stable))
    assert torch.equal(le, torch.zeros(5)) and torch.equal(ess, torch.full((5,), 37.0, dtype=torch.float64))


def test_oracle_with_everything_observed_is_the_row_nll_x():
    S, B, L, Z = 50, 6, 9, 3
    fx, r, noise = _case(S, B, L, Z, seed=2)
    y = (torch.rand(B, L, generator=torch.Generator().manual_seed(3)) < 0.4).float()
    prob, le, ess = CO.predict_conditional(fx, r, y.to(torch.int8), noise)
    assert torch.equal(prob, y)
    assert bool(((ess >= 1) & (ess <= S)).all())
    eps1 = torch.tensor([1e-6]).float()
    E = orc.clamped_probit(torch.tensordot(noise, r.T.float(), dims=1) + fx, eps1)
    for b in range(B):
        nll_x = orc.bernoulli_log_mean_exp(E[:, b:b + 1], y[b:b + 1], accum=torch.float64)
        assert abs(float(-le[b]) - float(nll_x)) <= 2e-6 * abs(float(nll_x)), (b, float(-le[b]), float(nll_x))


@pytest.mark.parametrize("y_o", [0, 1])
def test_oracle_converges_to_the_closed_form_of_one_observed_label(y_o):
    """P(y_u | y_o) = P_uo / P_o (y_o = 1) or (P_u - P_uo) / (1 - P_o) (y_o = 0), from predict_exact_oracle; every cell
    within 6 standard errors at S = 200 000."""
    S, B, L, Z = 200_000, 3, 6, 3
    fx, r, noise = _case(S, B, L, Z, seed=4 + y_o, sigma=1.5)
    fx = fx * 0.5
    o = 2
    obs = torch.full((B, L), -1, dtype=torch.int8)
    obs[:, o] = y_o
    prob, _, ess = CO.predict_conditional(fx, r, obs, noise)
    se = CO.stderr(fx, r, obs, noise)
    pairs = [(u, o) for u in range(L)]
    P_uo = XO.pair_prob(fx, r, pairs).numpy()
    P_u = XO.marginal(fx, r).numpy()
    P_o = P_u[:, [o]]
    want = P_uo / P_o if y_o == 1 else (P_u - P_uo) / (1 - P_o)
    free = [u for u in range(L) if u != o]
    z = np.abs(prob.double().numpy()[:, free] - want[:, free]) / se.numpy()[:, free]
    assert z.max() <= 6.0, z
    assert bool((prob[:, o] == float(y_o)).all())
    assert bool((ess > 1000).all())


def test_oracle_converges_to_quadrature_at_z1():
    """Z = 1: x_l = fx_l + R_l eps, so P(y_u = 1, y_O) and P(y_O) are one-dimensional integrals over eps; 120-node
    Gauss-Hermite quadrature of both, the oracle at S = 200 000 within 6 standard errors, log_evidence too."""
    from scipy.special import ndtr
    S, B, L = 200_000, 3, 7
    fx, r, noise = _case(S, B, L, 1, seed=9, sigma=1.8)
    obs = torch.full((B, L), -1, dtype=torch.int8)
    obs[0, [1, 4]] = torch.tensor([1, 0], dtype=torch.int8)
    obs[1, [0, 2, 5]] = torch.tensor([0, 0, 1], dtype=torch.int8)
    obs[2, 6] = 1
    prob, le, _ = CO.predict_conditional(fx, r, obs, noise)
    se = CO.stderr(fx, r, obs, noise)
    t, w = np.polynomial.hermite_e.hermegauss(120)
    w = w / np.sqrt(2 * np.pi)
    fx64, r64 = fx.double().numpy(), r.float().double().numpy()[:, 0]
    for b in range(B):
        E = XO.C_EPS + XO.K_EPS * ndtr(fx64[b][None, :] + r64[None, :] * t[:, None])     # (nodes, L)
        lik = np.ones_like(t)
        for l in range(L):
            if obs[b, l] in (0, 1):
                lik = lik * (E[:, l] if obs[b, l] == 1 else 1 - E[:, l])
        p_obs = float((w * lik).sum())
        want = (w[:, None] * lik[:, None] * E).sum(0) / p_obs
        for l in range(L):
            if obs[b, l] in (0, 1):
                continue
            assert abs(float(prob[b, l]) - want[l]) <= 6 * float(se[b, l]), (b, l, float(prob[b, l]), want[l])
        # log_evidence: the log of a mean of S weights, sd of the log ~ sd(lik) / (mean(lik) sqrt(S))
        sd = np.sqrt(float((w * lik * lik).sum()) - p_obs ** 2) / p_obs / np.sqrt(S)
        assert abs(float(le[b]) - np.log(p_obs)) <= 6 * sd + 1e-6, (b, float(le[b]), np.log(p_obs))


def test_header_declares_and_library_exports_predict_conditional(lib):
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    assert "mpvae_probit_predict_conditional" in declared_symbols()
    assert "mpvae_probit_predict_conditional" in _lib.EXPORTS
    assert hasattr(lib, "mpvae_probit_predict_conditional")
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION == 13


def test_stale_library_without_the_symbol_asks_for_a_rebuild(monkeypatch):
    from mpvae_b200 import _lib
    monkeypatch.setattr(_lib, "EXPORTS", _lib.EXPORTS + ("mpvae_no_such_symbol",))
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(_lib.LibraryMissing, match="rebuild"):
        _lib.lib()


def test_predict_conditional_entry_point_validates_arguments(lib):
    """Refused before anything touches the device."""
    from mpvae_b200 import _lib
    f = lib.mpvae_probit_predict_conditional
    p = _lib.ProbitParams()
    p.struct_bytes = 8
    assert f(C.byref(p), 256, 256, 256, None) == 1
    assert b"struct_bytes" in lib.mpvae_last_error()
    p.struct_bytes = C.sizeof(_lib.ProbitParams)
    p.S, p.B, p.L, p.Z = 10, 4, 14, 14
    p.B = 0
    assert f(C.byref(p), 256, 256, 256, None) == 1
    assert b"bad sizes" in lib.mpvae_last_error()
    p.B = 4
    assert f(C.byref(p), 256, 256, 256, None) == 1
    assert b"NULL input pointer" in lib.mpvae_last_error()
    p.fx_out, p.r, p.workspace = 256, 256, 256
    p.noise_b_global, p.noise_row0 = 4, 0
    assert f(C.byref(p), 256, 256, 256, None) == 1
    assert b"NULL forward output pointer" in lib.mpvae_last_error()
    p.indiv_prob = 256
    p.workspace_bytes = 16
    assert f(C.byref(p), 256, 256, 256, None) == 1
    assert b"workspace too small" in lib.mpvae_last_error()
    p.workspace_bytes = 1 << 40
    for args in ((None, 256, 256), (256, None, 256), (256, 256, None)):
        assert f(C.byref(p), *args, None) == 1
        assert b"observed/log_evidence/ess" in lib.mpvae_last_error()


def test_predict_conditional_refuses_cpu_tensors_grad_and_bad_observed():
    from mpvae_b200.mpvae import predict_conditional
    from mpvae_b200.probit import probit_predict_conditional
    case = H.load_golden("yeast_b16")
    t = H.to_torch(case["inputs"])
    args = orc.make_args(case["L"], case["Z"], n_test_sample=case["S"], mode="test")
    B, L = t["fx_out"].shape
    obs = torch.full((B, L), -1, dtype=torch.int8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        predict_conditional(t["fx_out"], t["r_sqrt_sigma"], obs, args)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        probit_predict_conditional(t["fx_out"], t["r_sqrt_sigma"].float(), obs, 4, noise_spec=(4, 1, 0, None, 0))
    with pytest.raises(RuntimeError, match="inference only"):
        predict_conditional(t["fx_out"], torch.nn.Parameter(t["r_sqrt_sigma"]), obs, args)
    with pytest.raises(RuntimeError, match="inference only"):
        predict_conditional(t["fx_out"].clone().requires_grad_(True), t["r_sqrt_sigma"], obs, args)
    # observed: dtype, shape, device -- checked on the host before the device is touched (an fx_out stand-in that
    # reports a CUDA device lets a CPU-only host reach these checks)
    fake = _FakeCuda(t["fx_out"])
    with pytest.raises(TypeError, match="int8"):
        predict_conditional(fake, t["r_sqrt_sigma"], obs.float(), args)
    with pytest.raises(TypeError, match="int8"):
        predict_conditional(fake, t["r_sqrt_sigma"], obs.numpy(), args)
    with pytest.raises(ValueError, match="shape"):
        predict_conditional(fake, t["r_sqrt_sigma"], obs[:, :-1], args)
    with pytest.raises(ValueError, match="is on"):
        predict_conditional(fake, t["r_sqrt_sigma"], obs, args)


class _FakeCuda:
    """An fx_out stand-in that reports a CUDA device, so the argument checks on `observed` run on a CPU-only host."""

    def __init__(self, t):
        self.shape, self.requires_grad, self.device = t.shape, False, torch.device("cuda:0")


# ---- data-parallel conditional scoring (gloo, CPU; the oracle injected as mpvae.predict_conditional) ----

def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


def _score(n_rows, batch_size):
    """infer.predict_conditional over n_rows rows in this process (one rank of the group, or the whole job)."""
    sys.path.insert(0, ROOT)
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_conditional
    from mpvae_b200.mpvae import VAE
    torch.set_num_threads(1)
    args = _args()
    np.random.seed(4)
    torch.manual_seed(0)
    model = VAE(args)
    model._reparameterize = lambda mu, logvar: mu       # the decoder on the posterior mean: no per-process randomness
    rng = np.random.RandomState(0)
    x = torch.from_numpy(rng.standard_normal((n_rows, args.feature_dim)).astype(np.float32))
    obs = torch.from_numpy(rng.randint(-1, 2, size=(n_rows, args.label_dim)).astype(np.int8))
    g = torch.Generator().manual_seed(77)
    full = torch.randn(args.n_test_sample, n_rows, args.z_dim, generator=g)
    seen = []

    def fake(fx_out, r, observed, a, noise=None):
        seen.append((a.mode, a.dp_global_batch, a.dp_row0, fx_out.shape[0]))
        lo = a.dp_row0
        assert torch.equal(observed, obs[lo:lo + fx_out.shape[0]])
        prob, le, ess = CO.predict_conditional(fx_out, r, observed, full[:, lo:lo + fx_out.shape[0]])
        return mpvae.ConditionalPrediction(prob, le, ess.float())

    mpvae.predict_conditional = fake
    prob, le, ess = predict_conditional(model, x, obs, args, batch_size=batch_size)
    assert all(m == "test" and gb == n_rows for m, gb, _, _ in seen)
    return torch.cat([prob, le[:, None], ess[:, None]], 1)


def _worker(rank, world, port, n_rows, batch_size, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret[rank] = _score(n_rows, batch_size)
    finally:
        dist.destroy_process_group()


def _two_ranks(n_rows, batch_size):
    import socket
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
    return ret[0], ret[1]


# 23 rows: shards [0, 12) and [12, 23), the one process in batches of 12 (same CPU matmul shapes); 1 row: rank 1 owns
# nothing and still joins the gather
@pytest.mark.timeout(300)
@pytest.mark.parametrize("n_rows,batch_size", [(23, 12), (1, 8)])
def test_two_ranks_conditional_equal_one_process(n_rows, batch_size):
    from mpvae_b200 import mpvae
    real = mpvae.predict_conditional
    try:
        got0, got1 = _two_ranks(n_rows, batch_size)
        want = _score(n_rows, batch_size)
    finally:
        mpvae.predict_conditional = real
    assert want.shape == (n_rows, _args().label_dim + 2)
    assert torch.equal(got0, want) and torch.equal(got1, want)
