"""CPU checks of the closed-form prediction (csrc/predictive.cu, csrc/bvn.cuh; probit.predict_exact / predict_pairs,
mpvae.predict_exact / PairPredictor, infer.predict_pairs): the fp64 oracle against scipy and a Monte Carlo, the bivariate
normal header compiled with g++ against the oracle, the C-ABI surface and its argument checks, the host-side refusals,
and the data-parallel pair scoring loop with the oracle injected."""
import os
import shutil
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy.stats import multivariate_normal

from tests import predict_exact_oracle as XO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host", "bvn_host.cpp")
NEW_SYMBOLS = ("mpvae_predictive_scale", "mpvae_predictive_rho", "mpvae_predict_exact", "mpvae_predict_pairs")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


@pytest.fixture(scope="module")
def bvn_binary(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = str(tmp_path_factory.mktemp("bvn") / "bvn_host")
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-o", out, SRC])
    return out


def run_bvn(binary, h, k, r):
    text = f"{len(h)}\n" + "\n".join(f"{float(a)!r} {float(b)!r} {float(c)!r}" for a, b, c in zip(h, k, r)) + "\n"
    res = subprocess.run([binary], input=text, capture_output=True, text=True, check=True)
    return np.array([float(v) for v in res.stdout.split()], dtype=np.float64)


def grid():
    vals = np.concatenate([np.linspace(-8.0, 8.0, 33), [37.0, -37.0, 0.0, 0.3, -1.7]])
    rhos = [0.0]
    for v in (0.3, 0.75, 0.925, 0.99, 1.0 - 1e-12, 1.0 - 1e-15):
        rhos += [v, -v]
    h, k, r = np.meshgrid(vals, vals, np.array(rhos), indexing="ij")
    return h.ravel(), k.ravel(), r.ravel()


# ---- the oracle ----

def test_oracle_bvn_matches_scipy_multivariate_normal():
    """Every branch of Owen's formula (h = 0, k = 0, both, hk < 0, hk > 0) against scipy's mvn CDF."""
    rng = np.random.RandomState(0)
    cases = [(0.0, 0.7, 0.4), (0.7, 0.0, -0.6), (0.0, 0.0, 0.5), (0.0, -1.2, 0.9), (-1.2, 0.0, -0.95),
             (1.1, -0.4, 0.3), (-2.0, 1.5, -0.8), (1.3, 2.2, 0.97), (-0.5, -1.5, 0.2), (-3.0, -3.0, -0.5)]
    cases += [(rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-0.99, 0.99)) for _ in range(60)]
    h, k, r = (np.array(c) for c in zip(*cases))
    got = XO.bvn(h, k, r)
    for i in range(len(h)):
        want = multivariate_normal.cdf([h[i], k[i]], mean=[0.0, 0.0], cov=[[1.0, r[i]], [r[i], 1.0]])
        assert abs(got[i] - want) <= 1e-6, (h[i], k[i], r[i], got[i], want)


def test_oracle_bvn_limits():
    from scipy.special import ndtr
    h, k = np.meshgrid(np.linspace(-4, 4, 17), np.linspace(-4, 4, 17))
    assert np.max(np.abs(XO.bvn(h, k, 0.0) - ndtr(h) * ndtr(k))) <= 1e-15
    # |rho| -> 1: Phi(min(h, k)) and max(0, Phi(h) + Phi(k) - 1); the gap closes like sqrt(1 - |rho|)
    for eps in (1e-8, 1e-12):
        assert np.max(np.abs(XO.bvn(h, k, 1.0 - eps) - ndtr(np.minimum(h, k)))) <= 2 * np.sqrt(eps)
        assert np.max(np.abs(XO.bvn(h, k, -1.0 + eps) - np.maximum(0.0, ndtr(h) + ndtr(k) - 1.0))) <= 2 * np.sqrt(eps)
    assert np.array_equal(XO.bvn(h, k, 1.0), ndtr(np.minimum(h, k)))


def test_oracle_agrees_with_monte_carlo():
    """1 M fp64 samples of the probit noise n = R eps: mean E(a + n_l) and mean E(a + n_i) E(a + n_j) against the closed
    forms of the marginal and the pair probability (L = 6, Z = 4)."""
    g = torch.Generator().manual_seed(5)
    L, Z, B, S = 6, 4, 3, 1_000_000
    r = torch.randn(L, Z, generator=g) * 0.7
    fx = torch.randn(B, L, generator=g) * 1.5
    pairs = torch.triu_indices(L, L, 1).T
    marg, pp = XO.marginal(fx, r), XO.pair_prob(fx, r, pairs)
    r64 = r.double()
    z_max = 0.0
    for b in range(B):
        eps = torch.randn(S, Z, generator=g, dtype=torch.float64)
        E = XO.C_EPS + XO.K_EPS * torch.special.ndtr(fx[b].double()[None, :] + eps @ r64.T)     # (S, L)
        m, sd = E.mean(0), E.std(0) / np.sqrt(S)
        z_max = max(z_max, float(((m - marg[b]) / sd).abs().max()))
        prod = E[:, pairs[:, 0]] * E[:, pairs[:, 1]]
        m2, sd2 = prod.mean(0), prod.std(0) / np.sqrt(S)
        z_max = max(z_max, float(((m2 - pp[b]) / sd2).abs().max()))
        var_mc = E.var(0)
        assert torch.allclose(var_mc, XO.marginal_var(fx[b:b + 1], r)[0], rtol=2e-2, atol=1e-6)
    assert z_max <= 6.0, z_max


# ---- csrc/bvn.cuh on the host ----

def test_host_bvn_header_matches_the_oracle(bvn_binary):
    h, k, r = grid()
    got = run_bvn(bvn_binary, h, k, r)
    want = XO.bvn(h, k, r)
    err = np.abs(got - want)
    assert err.max() <= 1e-12, (err.max(), h[err.argmax()], k[err.argmax()], r[err.argmax()])
    assert np.all(got >= 0.0) and np.all(got <= 1.0)


def test_host_gauss_legendre_tables(bvn_binary):
    res = subprocess.run([bvn_binary, "--tables"], capture_output=True, text=True, check=True)
    lines = res.stdout.strip().splitlines()
    assert [int(ln.split()[0]) for ln in lines] == [3, 6, 10]
    for ln in lines:
        v = np.array([float(t) for t in ln.split()[1:]])
        half = len(v) // 2
        x, w = np.polynomial.legendre.leggauss(2 * half)
        assert np.max(np.abs(v[:half] - x[half:][::-1])) <= 1e-15
        assert np.max(np.abs(v[half:] - w[half:][::-1])) <= 1e-15


# ---- C-ABI ----

def test_header_declares_and_library_exports_the_closed_form(lib):
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for s in NEW_SYMBOLS:
        assert s in declared_symbols() and s in _lib.EXPORTS and hasattr(lib, s)
    assert _lib.ABI_VERSION == 13 and lib.mpvae_abi_version() == 13


def test_entry_points_validate_arguments(lib):
    """Refused before anything touches the device (the non-NULL pointers below are never dereferenced)."""
    err = lambda: lib.mpvae_last_error().decode()
    d = 256
    assert lib.mpvae_predictive_scale(None, 4, 4, d, None) == 1 and "NULL" in err()
    assert lib.mpvae_predictive_scale(d, 4, 4, None, None) == 1 and "NULL" in err()
    assert lib.mpvae_predictive_scale(d, 0, 4, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predictive_scale(d, 4, -1, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predictive_rho(d, 4, 4, d, None, 3, d, None) == 1 and "NULL" in err()
    assert lib.mpvae_predictive_rho(d, 4, 4, d, d, -1, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predictive_rho(d, 0, 4, d, d, 3, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predictive_rho(d, 4, 0, d, d, 3, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predictive_rho(d, 4, 4, d, d + 4, 3, d, None) == 1 and "aligned" in err()
    assert lib.mpvae_predict_exact(None, 2, 4, d, 0, d, None) == 1 and "NULL" in err()
    assert lib.mpvae_predict_exact(d, 2, 4, None, 0, d, None) == 1 and "NULL" in err()
    assert lib.mpvae_predict_exact(d, -1, 4, d, 0, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predict_exact(d, 2, 0, d, 0, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predict_pairs(d, 2, 4, d, d, None, 3, 0, d, None) == 1 and "NULL" in err()
    assert lib.mpvae_predict_pairs(d, 2, 4, d, d, d, 3, 0, None, None) == 1 and "NULL" in err()
    assert lib.mpvae_predict_pairs(d, 2, 4, d, d, d, -1, 0, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predict_pairs(d, 2, 0, d, d, d, 3, 0, d, None) == 1 and "bad sizes" in err()
    assert lib.mpvae_predict_pairs(d, 2, 4, d, d + 4, d, 3, 0, d, None) == 1 and "aligned" in err()


# ---- host-side refusals ----

def test_refuses_cpu_tensors_bad_pairs_and_grad():
    from mpvae_b200 import mpvae, probit
    args = SimpleNamespace(mpvae_flags=0)
    fx, r = torch.randn(3, 5), torch.randn(5, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mpvae.predict_exact(fx, r, args)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mpvae.PairPredictor(r, [[0, 1]], args)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        probit.predictive_scale(r)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        probit.predict_exact(fx, torch.ones(5, dtype=torch.float64))
    for bad in ([[0, 5]], [[-1, 2]], [[0, 1], [4, 7]]):
        with pytest.raises(ValueError, match="outside"):
            mpvae.PairPredictor(r, bad, args)
        with pytest.raises(ValueError, match="outside"):
            probit.predict_pairs(fx, torch.ones(5, dtype=torch.float64), bad, torch.zeros(len(bad), dtype=torch.float64))
        with pytest.raises(ValueError, match="outside"):
            probit.predictive_rho(r, torch.ones(5, dtype=torch.float64), bad)
    with pytest.raises(ValueError):
        probit.label_pairs(torch.zeros(4, 3, dtype=torch.int64), 5)
    with pytest.raises(TypeError):
        probit.label_pairs(torch.zeros(4, 2), 5)
    with pytest.raises(RuntimeError, match="inference only"):
        mpvae.predict_exact(fx, torch.nn.Parameter(r), args)
    with pytest.raises(RuntimeError, match="inference only"):
        mpvae.predict_exact(fx.requires_grad_(True), r, args)
    with pytest.raises(RuntimeError, match="inference only"):
        mpvae.PairPredictor(torch.nn.Parameter(r), [[0, 1]], args)


def test_all_pairs_is_the_upper_triangle():
    from mpvae_b200.mpvae import all_pairs
    p = all_pairs(38)
    assert p.shape == (703, 2) and p.dtype == torch.int64
    assert bool((p[:, 0] < p[:, 1]).all())
    assert len({tuple(v) for v in p.tolist()}) == 703
    assert p[:3].tolist() == [[0, 1], [0, 2], [0, 3]] and p[-1].tolist() == [36, 37]
    assert all_pairs(1).shape == (0, 2)


# ---- data-parallel pair scoring (gloo, CPU; the oracle injected as PairPredictor) ----

def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


class _OraclePairs:
    """Stands in for mpvae.PairPredictor on the CPU: the fp64 oracle rounded to fp32."""

    def __init__(self, r_sqrt_sigma, pairs, args):
        self.r, self.pairs = r_sqrt_sigma.detach(), torch.as_tensor(pairs)

    def __call__(self, fx_out):
        return XO.pair_prob(fx_out, self.r, self.pairs).float()


def _score(n_rows, batch_size):
    sys.path.insert(0, ROOT)
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_pairs
    torch.set_num_threads(1)
    mpvae.PairPredictor = _OraclePairs
    args = _args()
    np.random.seed(4)
    torch.manual_seed(0)
    model = mpvae.VAE(args)
    model._reparameterize = lambda mu, logvar: mu       # the decoder on the posterior mean: no per-process randomness
    rng = np.random.RandomState(0)
    x = torch.from_numpy(rng.standard_normal((n_rows, args.feature_dim)).astype(np.float32))
    pairs = mpvae.all_pairs(args.label_dim)
    pairs = torch.cat([pairs, torch.tensor([[3, 3], [7, 2]])])
    return predict_pairs(model, x, pairs, args, batch_size=batch_size)


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


# 23 rows: shards [0, 12) and [12, 23), and a batch size of 12 gives the one process the same two batches (CPU BLAS
# results depend on the product shapes); 1 row: rank 1 owns nothing and still joins the gather
@pytest.mark.timeout(300)
@pytest.mark.parametrize("n_rows,batch_size", [(23, 12), (1, 8)])
def test_two_ranks_pairs_equal_one_process(n_rows, batch_size):
    from mpvae_b200 import mpvae
    real = mpvae.PairPredictor
    try:
        got0, got1 = _two_ranks(n_rows, batch_size)
        want = _score(n_rows, batch_size)
    finally:
        mpvae.PairPredictor = real
    assert want.shape == (n_rows, 36 + 2) and want.dtype == torch.float32
    assert torch.equal(got0, want) and torch.equal(got1, want)
