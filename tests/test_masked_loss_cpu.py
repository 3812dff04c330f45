"""CPU checks of partially labelled training (compute_loss(..., label_mask=) / mpvae_probit_forward_masked /
mpvae_probit_backward_masked): the masked oracle against the pinned oracle (all-ones mask, deleted label columns), its
two ranking forms against each other, its insensitivity to unobserved label values; the C-ABI surface; the host-side
refusals; and DataParallelStep with masks on two gloo ranks against one process, the masked oracle as loss_fn."""
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
    return "pairwise" if L <= 128 else "factorised"     # the pairwise form materialises (S, B, L, L)


def _same(a, b):
    """bit equality, NaN pattern included"""
    return a.shape == b.shape and torch.equal(torch.isnan(a), torch.isnan(b)) and \
        torch.equal(torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0))


@pytest.mark.parametrize("name", H.golden_names())
def test_all_ones_mask_is_the_pinned_oracle_bit_for_bit(name):
    case, t, noise = _golden(name)
    up = {k: torch.from_numpy(v) for k, v in case["upstream"].items()} or None
    kw = dict(ranking=_ranking(case["L"]))
    want, want_g = orc.probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], upstream=up, **kw)
    ones = torch.ones(t["y"].shape, dtype=torch.bool)
    got, got_g = MO.masked_probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], ones, upstream=up, **kw)
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
    noise = torch.randn(S, B, Z, generator=g)
    return t, noise, g


@pytest.mark.parametrize("frac", [0.1, 0.5, 0.9])
def test_pairwise_and_factorised_ranking_agree_under_random_masks(frac):
    t, noise, g = _random_case(6, 9, 23, 7, seed=int(frac * 10))
    mask = torch.rand(t["y"].shape, generator=g) < frac
    mask[0] = False                                     # a row with nothing observed
    t64 = {k: v.double() for k, v in t.items()}
    a, ga = MO.masked_probit_elbo_with_grads(t64, noise.double(), 0.5, 10.0, mask, ranking="pairwise", dtype=torch.float64)
    b, gb = MO.masked_probit_elbo_with_grads(t64, noise.double(), 0.5, 10.0, mask, ranking="factorised", dtype=torch.float64)
    for k in TERMS:
        assert torch.allclose(getattr(a, k), getattr(b, k), rtol=1e-12, atol=1e-14), k
    for k in ga:
        assert torch.allclose(ga[k], gb[k], rtol=1e-10, atol=1e-14, equal_nan=True), k   # NaN: degenerate rows


@pytest.mark.parametrize("ranking", ["pairwise", "factorised"])
def test_hidden_columns_equal_the_problem_without_them(ranking):
    """A mask that hides whole label columns in every row = the unmasked oracle with those columns (and R's rows)
    deleted: same log-likelihoods, ranking losses, KL and gradients of the kept cells; hidden cells get no gradient."""
    t, noise, g = _random_case(8, 12, 19, 5, seed=3)
    keep = torch.ones(19, dtype=torch.bool)
    keep[[0, 4, 5, 11, 18]] = False
    mask = keep[None, :].expand(12, 19)
    t64 = {k: v.double() for k, v in t.items()}
    got, got_g = MO.masked_probit_elbo_with_grads(t64, noise.double(), 0.5, 10.0, mask, ranking=ranking, dtype=torch.float64)
    sub = dict(t64)
    for k in ("y", "fe_out", "fx_out"):
        sub[k] = t64[k][:, keep]
    sub["r_sqrt_sigma"] = t64["r_sqrt_sigma"][keep]
    want, want_g = orc.probit_elbo_with_grads(sub, noise.double(), 0.5, 10.0, ranking=ranking, dtype=torch.float64)
    for k in TERMS[:6]:
        assert abs(float(getattr(got, k)) - float(getattr(want, k))) <= 1e-6 * max(1.0, abs(float(getattr(want, k)))), k
    for k in ("indiv_prob", "indiv_prob_label"):
        assert torch.allclose(getattr(got, k)[:, keep], getattr(want, k), rtol=1e-6, atol=1e-7), k
    for k in ("fe_out", "fx_out"):
        assert torch.allclose(got_g[k][:, keep], want_g[k], rtol=1e-6, atol=1e-9), k
        assert torch.equal(got_g[k][:, ~keep], torch.zeros_like(got_g[k][:, ~keep])), k
    for k in ("fe_mu", "fe_logvar", "fx_mu", "fx_logvar"):
        assert torch.allclose(got_g[k], want_g[k], rtol=1e-6, atol=1e-9), k
    assert torch.allclose(got_g["r_sqrt_sigma"][keep], want_g["r_sqrt_sigma"], rtol=1e-6, atol=1e-9)
    assert torch.equal(got_g["r_sqrt_sigma"][~keep], torch.zeros_like(got_g["r_sqrt_sigma"][~keep]))


@pytest.mark.parametrize("fill", ["random", 0.5, 7.0, float("nan")])
def test_unobserved_label_values_change_nothing(fill):
    t, noise, g = _random_case(6, 10, 17, 5, seed=5)
    mask = torch.rand(t["y"].shape, generator=g) < 0.5
    base, base_g = MO.masked_probit_elbo_with_grads(t, noise, 0.5, 10.0, mask, ranking="pairwise")
    t2 = dict(t)
    other = torch.rand(t["y"].shape, generator=g).round() if fill == "random" else torch.full(t["y"].shape, fill)
    t2["y"] = torch.where(mask, t["y"], other)
    got, got_g = MO.masked_probit_elbo_with_grads(t2, noise, 0.5, 10.0, mask, ranking="pairwise")
    for k in TERMS:
        assert _same(getattr(got, k), getattr(base, k)), k
    for k in base_g:
        assert _same(got_g[k], base_g[k]), k


def test_header_declares_and_library_exports_the_masked_entry_points(lib):
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for sym in ("mpvae_probit_forward_masked", "mpvae_probit_backward_masked"):
        assert sym in declared_symbols()
        assert sym in _lib.EXPORTS
        assert hasattr(lib, sym)
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION == 13


def test_masked_entry_points_validate_arguments_like_the_unmasked_ones(lib):
    """Refused before anything touches the device, with the unmasked calls' messages."""
    import ctypes as C
    from mpvae_b200 import _lib
    for f in (lib.mpvae_probit_forward_masked, lib.mpvae_probit_backward_masked):
        p = _lib.ProbitParams()
        p.struct_bytes = 8
        assert f(C.byref(p), 256, None) == 1
        assert b"struct_bytes" in lib.mpvae_last_error()
        p.struct_bytes = C.sizeof(_lib.ProbitParams)
        p.S, p.B, p.L, p.Z = 10, 0, 14, 14
        assert f(C.byref(p), 256, None) == 1
        assert b"bad sizes" in lib.mpvae_last_error()
        p.B = 4
        assert f(C.byref(p), 256, None) == 1
        assert b"NULL input pointer" in lib.mpvae_last_error()


def test_label_mask_host_refusals():
    from mpvae_b200.mpvae import compute_loss
    from mpvae_b200.probit import _check_label_mask
    case, t, noise = _golden("yeast_b16")
    args = orc.make_args(case["L"], case["Z"], n_train_sample=case["S"], mode="train")
    B, L = t["y"].shape
    ok = torch.ones(B, L, dtype=torch.bool)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                     t["r_sqrt_sigma"], args, noise=noise, label_mask=ok)
    cuda = torch.device("cuda:0")          # the batch's device as the check sees it: CPU masks are then refused
    with pytest.raises(TypeError, match="bool or uint8"):
        _check_label_mask(ok.float(), B, L, cuda)
    with pytest.raises(TypeError, match="bool or uint8"):
        _check_label_mask(ok.to(torch.int8), B, L, cuda)
    with pytest.raises(TypeError, match="bool or uint8"):
        _check_label_mask(ok.numpy(), B, L, cuda)
    with pytest.raises(ValueError, match="shape"):
        _check_label_mask(ok[:, :-1], B, L, cuda)
    with pytest.raises(ValueError, match="shape"):
        _check_label_mask(ok.T.contiguous(), B, L, cuda)
    with pytest.raises(ValueError, match="is on"):
        _check_label_mask(ok, B, L, cuda)
    m = _check_label_mask(ok[:, ::1], B, L, torch.device("cpu"))
    assert m.dtype == torch.uint8 and m.is_contiguous() and bool((m == 1).all())


# ---- data-parallel training with masks (gloo, CPU; the masked oracle as loss_fn) ----

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
    stepper = DataParallelStep(model, opt, None, args, clip_norm=100.0, loss_fn=MO.masked_loss_fn)
    rng = np.random.RandomState(0)
    n = 23
    x = torch.from_numpy(rng.standard_normal((n, args.feature_dim)).astype(np.float32))
    y = torch.from_numpy((rng.uniform(size=(n, args.label_dim)) < 0.3).astype(np.float32))
    mask = torch.from_numpy(rng.uniform(size=(n, args.label_dim)) < 0.6)
    y[:, 0], y[:, 1] = 1.0, 0.0                             # every row has an observed positive and negative ...
    mask[:, :2] = True
    mask[3] = False                                         # ... but this one, which has nothing observed
    y = torch.where(mask, y, 0.0)                           # unknown labels written as 0 for the label encoder
    outs = []
    for i in range(n_steps):
        idx = torch.arange(i * 6, i * 6 + batch) % n
        noise = torch.randn(args.n_train_sample, batch, args.z_dim, generator=torch.Generator().manual_seed(1000 + i))
        outs.append(stepper.step(y[idx], x[idx], noise=noise, label_mask=mask[idx]))
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
def test_two_ranks_with_masks_equal_one_process():
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
