"""CPU checks of weighted training (compute_loss(..., row_weight=) / mpvae_probit_forward_weighted /
mpvae_probit_backward_weighted): the weighted oracle against the pinned oracle (all-ones weights, with and without a
mask) and against duplicated rows (integer weights); zero-weight rows; the C-ABI surface; the host-side refusals; and
DataParallelStep with weights on two gloo ranks against one process, the weighted oracle as loss_fn."""
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
from tests import masked_elbo_oracle as MO
from tests import weighted_elbo_oracle as WO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TERMS = ("total_loss", "nll_loss", "nll_loss_x", "c_loss", "c_loss_x", "kl_loss", "indiv_prob", "indiv_prob_label")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


def _golden(name):
    case = H.load_golden(name)
    t = H.to_torch(case["inputs"])
    return case, t, torch.from_numpy(case["noise"])


def _ranking(L):
    return "pairwise" if L <= 128 else "factorised"


def _same(a, b):
    """bit equality, NaN pattern included"""
    return a.shape == b.shape and torch.equal(torch.isnan(a), torch.isnan(b)) and \
        torch.equal(torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0))


@pytest.mark.parametrize("name", H.golden_names())
@pytest.mark.parametrize("masked", [False, True])
def test_all_ones_weights_are_the_pinned_oracle_bit_for_bit(name, masked):
    """Without a mask against the pinned oracle; with a random mask against the masked oracle (itself the pinned oracle
    bit for bit with an all-ones mask, test_masked_loss_cpu)."""
    case, t, noise = _golden(name)
    up = {k: torch.from_numpy(v) for k, v in case["upstream"].items()} or None
    kw = dict(ranking=_ranking(case["L"]))
    B, L = t["y"].shape
    if masked:
        mask = torch.rand(B, L, generator=torch.Generator().manual_seed(B + L)) < 0.6
        want, want_g = MO.masked_probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], mask, upstream=up, **kw)
    else:
        mask = None
        want, want_g = orc.probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], upstream=up, **kw)
    got, got_g = WO.weighted_probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], torch.ones(B), mask,
                                                    upstream=up, **kw)
    for k in TERMS:
        assert _same(getattr(got, k), getattr(want, k)), k
    for k in want_g:
        assert (got_g[k] is None) == (want_g[k] is None), k
        if want_g[k] is not None:
            assert _same(got_g[k], want_g[k]), k


def _random_case(S, B, L, Z, D=6, seed=0):
    g = torch.Generator().manual_seed(seed)
    t = {"y": (torch.rand(B, L, generator=g) < 0.35).float(),
         "fe_out": torch.randn(B, L, generator=g), "fx_out": torch.randn(B, L, generator=g),
         "fe_mu": torch.randn(B, D, generator=g), "fe_logvar": 0.3 * torch.randn(B, D, generator=g),
         "fx_mu": torch.randn(B, D, generator=g), "fx_logvar": 0.3 * torch.randn(B, D, generator=g),
         "r_sqrt_sigma": torch.randn(L, Z, generator=g, dtype=torch.float64) / np.sqrt(Z)}
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0                   # no degenerate row
    noise = torch.randn(S, B, Z, generator=g)
    return t, noise, g


def _duplicate(t, noise, counts):
    """every row b repeated counts[b] times (0: dropped), each copy with the row's noise column"""
    idx = torch.repeat_interleave(torch.arange(len(counts)), torch.as_tensor(counts))
    d = {k: (v if k == "r_sqrt_sigma" else v[idx]) for k, v in t.items()}
    return d, noise[:, idx], idx


@pytest.mark.parametrize("ranking", ["pairwise", "factorised"])
@pytest.mark.parametrize("masked", [False, True])
def test_integer_weights_equal_duplicated_rows(ranking, masked):
    """w_b = k_b (0 included) against the unweighted problem with row b repeated k_b times on the same noise column, in
    fp64: scalars x B agree, each row's gradient (total_loss x B) is the sum over its copies, g_R agrees, and a weighted
    row's predictions are each copy's."""
    S, B, L, Z = 5, 9, 13, 4
    t, noise, g = _random_case(S, B, L, Z, seed=7)
    counts = [1, 3, 0, 2, 1, 0, 4, 1, 2]
    mask = (torch.rand(B, L, generator=g) < 0.7) if masked else None
    if mask is not None:
        mask[:, :2] = True
    t64 = {k: v.double() for k, v in t.items()}
    w = torch.tensor(counts, dtype=torch.float64)
    Bd = int(sum(counts))
    got, got_g = WO.weighted_probit_elbo_with_grads(t64, noise.double(), 0.5, 10.0, w, mask, ranking=ranking,
                                                    dtype=torch.float64, upstream={"total_loss": torch.tensor(float(B))})
    d, dnoise, idx = _duplicate(t64, noise.double(), counts)
    dmask = mask[idx] if mask is not None else None
    want, want_g = WO.weighted_probit_elbo_with_grads(d, dnoise, 0.5, 10.0, torch.ones(Bd, dtype=torch.float64), dmask,
                                                      ranking=ranking, dtype=torch.float64,
                                                      upstream={"total_loss": torch.tensor(float(Bd))})
    for i in range(6):
        assert abs(float(got[i].detach()) * B - float(want[i].detach()) * Bd) <= 1e-12 * max(1.0, abs(float(want[i].detach()) * Bd)), TERMS[i]
    for i in (6, 7):
        assert torch.allclose(got[i][idx], want[i], rtol=0, atol=1e-12), TERMS[i]
    for k in ("fe_out", "fx_out", "fe_mu", "fe_logvar", "fx_mu", "fx_logvar"):
        summed = torch.zeros_like(got_g[k]).index_add_(0, idx, want_g[k])
        assert torch.allclose(got_g[k], summed, rtol=1e-10, atol=1e-13), k
        zero_rows = torch.tensor(counts) == 0
        assert torch.equal(got_g[k][zero_rows], torch.zeros_like(got_g[k][zero_rows])), k
    assert torch.allclose(got_g["r_sqrt_sigma"], want_g["r_sqrt_sigma"], rtol=1e-10, atol=1e-13)


def test_zero_weight_degenerate_row_gets_no_nan():
    """A degenerate row (no positive) with weight 0: every gradient finite without SANITIZE, the row's logit gradients
    exactly 0 with total_loss's cotangent alone, and the loss that of the batch without the row times (B - 1) / B."""
    S, B, L, Z = 4, 6, 11, 3
    t, noise, _ = _random_case(S, B, L, Z, seed=2)
    t["y"][2] = 0.0
    w = torch.ones(B)
    w[2] = 0.0
    got, got_g = WO.weighted_probit_elbo_with_grads(t, noise, 0.5, 10.0, w, ranking="pairwise")
    for k, v in got_g.items():
        assert bool(torch.isfinite(v).all()), k
    for k in ("fe_out", "fx_out", "fe_mu", "fe_logvar", "fx_mu", "fx_logvar"):
        assert torch.equal(got_g[k][2], torch.zeros_like(got_g[k][2])), k
    keep = [0, 1, 3, 4, 5]
    sub = {k: (v if k == "r_sqrt_sigma" else v[keep]) for k, v in t.items()}
    want = orc.probit_elbo(sub["y"], sub["fe_out"], sub["fe_mu"], sub["fe_logvar"], sub["fx_out"], sub["fx_mu"],
                           sub["fx_logvar"], sub["r_sqrt_sigma"], noise[:, keep], 0.5, 10.0)
    for i in range(6):
        assert abs(float(got[i]) - float(want[i]) * (B - 1) / B) <= 1e-6 * max(1.0, abs(float(want[i]))), TERMS[i]
    # unweighted, the same row gives NaN gradients (0/0 of its ranking normaliser)
    _, g1 = WO.weighted_probit_elbo_with_grads(t, noise, 0.5, 10.0, torch.ones(B), ranking="pairwise")
    assert bool(torch.isnan(g1["fe_out"][2]).all())


def test_header_declares_and_library_exports_the_weighted_entry_points(lib):
    """Additive entry points: the ABI version and mpvae_probit_params are unchanged."""
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for sym in ("mpvae_probit_forward_weighted", "mpvae_probit_backward_weighted"):
        assert sym in declared_symbols()
        assert sym in _lib.EXPORTS
        assert hasattr(lib, sym)
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION == 13


def test_weighted_entry_points_validate_arguments_like_the_masked_ones(lib):
    """Refused before anything touches the device, with the unweighted calls' messages."""
    from mpvae_b200 import _lib
    for f in (lib.mpvae_probit_forward_weighted, lib.mpvae_probit_backward_weighted):
        for mask, weight in ((None, 512), (256, 512), (None, None)):
            p = _lib.ProbitParams()
            p.struct_bytes = 8
            assert f(C.byref(p), mask, weight, None) == 1
            assert b"struct_bytes" in lib.mpvae_last_error()
            p.struct_bytes = C.sizeof(_lib.ProbitParams)
            p.S, p.B, p.L, p.Z = 10, 0, 14, 14
            assert f(C.byref(p), mask, weight, None) == 1
            assert b"bad sizes" in lib.mpvae_last_error()
            p.B = 4
            assert f(C.byref(p), mask, weight, None) == 1
            assert b"NULL input pointer" in lib.mpvae_last_error()


def test_row_weight_host_refusals():
    from mpvae_b200 import mpvae
    from mpvae_b200.probit import _check_row_weight
    case, t, noise = _golden("yeast_b16")
    args = orc.make_args(case["L"], case["Z"], n_train_sample=case["S"], mode="train")
    B = t["y"].shape[0]
    ok = torch.ones(B)
    call = lambda w: mpvae.compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"],  # noqa: E731
                                        t["fx_logvar"], t["r_sqrt_sigma"], args, row_weight=w)
    before = dict(mpvae._state)
    # refused before the device check and before noise_plan: no noise offset is consumed
    with pytest.raises(ValueError, match="requires grad"):
        call(ok.clone().requires_grad_(True))
    with pytest.raises(ValueError, match="shape"):
        call(ok[:-1])
    with pytest.raises(TypeError, match="floating"):
        call(ok.to(torch.int64))
    assert mpvae._state == before
    with pytest.raises(RuntimeError, match="no CPU fallback"):   # a valid weight reaches the device check
        call(ok)
    assert mpvae._state == before
    cuda = torch.device("cuda:0")          # the batch's device as the check sees it: CPU weights are then refused
    with pytest.raises(ValueError, match="is on"):
        _check_row_weight(ok, B, cuda)
    with pytest.raises(TypeError, match="floating"):
        _check_row_weight(ok.bool(), B, cuda)
    with pytest.raises(TypeError, match="floating"):
        _check_row_weight(ok.numpy(), B, cuda)
    with pytest.raises(ValueError, match="shape"):
        _check_row_weight(ok[None], B, cuda)
    w = _check_row_weight(torch.arange(2 * B, dtype=torch.float64)[::2], B, torch.device("cpu"))
    assert w.dtype == torch.float32 and w.is_contiguous() and torch.equal(w, torch.arange(0, 2 * B, 2, dtype=torch.float32))
    w = _check_row_weight(ok.half(), B, torch.device("cpu"))
    assert w.dtype == torch.float32


# ---- data-parallel training with weights (gloo, CPU; the weighted oracle as loss_fn) ----

def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


def _run_steps(n_steps=3, batch=11):
    sys.path.insert(0, ROOT)
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep
    torch.set_num_threads(1)
    args = _args()
    np.random.seed(4)
    torch.manual_seed(0)
    model = VAE(args)
    with torch.no_grad():                                   # the reparameterisation contributes < 1e-6 (test_dp_cpu)
        for head in (model.fe_logvar, model.fx_logvar):
            head.weight.zero_(); head.bias.fill_(-30.0)
    opt = torch.optim.SGD(model.parameters(), lr=0.05, weight_decay=1e-5)
    stepper = DataParallelStep(model, opt, None, args, clip_norm=100.0, loss_fn=WO.weighted_loss_fn)
    rng = np.random.RandomState(0)
    n = 23
    x = torch.from_numpy(rng.standard_normal((n, args.feature_dim)).astype(np.float32))
    y = torch.from_numpy((rng.uniform(size=(n, args.label_dim)) < 0.3).astype(np.float32))
    y[:, 0], y[:, 1] = 1.0, 0.0
    w = torch.from_numpy(rng.uniform(0.0, 3.0, size=n).astype(np.float32))
    w[[2, 9]] = 0.0
    w[5] = -0.5
    outs = []
    for i in range(n_steps):
        idx = torch.arange(i * 6, i * 6 + batch) % n
        noise = torch.randn(args.n_train_sample, batch, args.z_dim, generator=torch.Generator().manual_seed(1000 + i))
        outs.append(stepper.step(y[idx], x[idx], noise=noise, row_weight=w[idx]))
    return model, outs


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        model, outs = _run_steps()
        ret[rank] = ({k: v.clone() for k, v in model.state_dict().items()}, [tuple(float(t) for t in o[:6]) for o in outs])
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_ranks_with_weights_equal_one_process():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(240)
        assert p.exitcode == 0
    model, outs = _run_steps()
    ref = model.state_dict()
    for rank in range(2):
        sd, scal = ret[rank]
        for k in ref:
            assert torch.allclose(sd[k].double(), ref[k].double(), rtol=2e-4, atol=2e-6), (rank, k)
            assert bool(torch.isfinite(sd[k]).all()), (rank, k)
        for got, want in zip(scal, outs):
            for a, b in zip(got, want[:6]):
                assert abs(a - float(b)) <= 2e-5 * max(1.0, abs(float(b))), (rank, a, float(b))
    for k in ref:
        assert torch.equal(ret[0][0][k], ret[1][0][k]), k
