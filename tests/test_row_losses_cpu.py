"""CPU checks of per-row losses (compute_loss(..., reduction='none') / mpvae_probit_forward_rows /
mpvae_probit_backward_rows): the per-row oracle against the batch oracles on every golden fixture (mask, row weights,
label weights), the zero-cotangent rule for degenerate rows, the C-ABI surface, the host-side refusals, and
DataParallelStep(row_objective=) on two gloo ranks against one process, the per-row oracle as loss_fn."""
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
from tests import label_weighted_elbo_oracle as LWO
from tests import row_elbo_oracle as RO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


@pytest.mark.parametrize("name", H.golden_names())
@pytest.mark.parametrize("options", ["plain", "mask_weights"])
def test_per_row_terms_average_to_the_batch_oracle(name, options):
    """fp64: the mean over the rows of each per-row output is the (label-)weighted oracle's batch output, and the
    per-row predictions are the same tensors."""
    case, t, noise = _golden(name)
    B, L = t["y"].shape
    g = torch.Generator().manual_seed(B * 31 + L)
    mask = rw = lw = None
    if options == "mask_weights":
        mask = torch.rand(B, L, generator=g) < 0.7
        rw = torch.rand(B, generator=g, dtype=torch.float64) * 2.0
        rw[0] = 0.0
        lw = 0.25 + torch.rand(2, L, generator=g, dtype=torch.float64) * 2.0
    kw = dict(ranking="pairwise" if L <= 128 else "factorised", dtype=torch.float64)
    t64 = [t[k].double() for k in ("y", "fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar")]
    coeffs = (case["nll_coeff"], case["c_coeff"])
    rows = RO.row_probit_elbo(*t64, t["r_sqrt_sigma"], noise, *coeffs, rw, mask, lw, **kw)
    want = LWO.label_weighted_probit_elbo(*t64, t["r_sqrt_sigma"], noise, *coeffs,
                                          torch.ones(2, L, dtype=torch.float64) if lw is None else lw, rw, mask, **kw)
    for i in range(6):
        assert rows[i].shape == (B,), RO.ROW_TERMS[i]
        got, ref = float(rows[i].mean()), float(want[i])
        assert abs(got - ref) <= 1e-12 * max(1.0, abs(ref)), (RO.ROW_TERMS[i], got, ref)
    if rw is not None:
        for i in range(6):
            assert float(rows[i][0]) == 0.0, RO.ROW_TERMS[i]
    assert torch.equal(rows[6], want[6]) and torch.equal(rows[7], want[7])


def test_zero_cotangent_rows_leave_degenerate_rows_out():
    """A degenerate row (all-0 labels) and one with all-1 labels, both left out of the objective (zero cotangents):
    every gradient finite, their logit gradients exactly 0; selected, they give NaN as the batch oracle does."""
    g = torch.Generator().manual_seed(3)
    S, B, L, Z, D = 4, 6, 9, 3, 5
    t = {"y": (torch.rand(B, L, generator=g) < 0.4).float(), "fe_out": torch.randn(B, L, generator=g),
         "fx_out": torch.randn(B, L, generator=g), "fe_mu": torch.randn(B, D, generator=g),
         "fe_logvar": 0.3 * torch.randn(B, D, generator=g), "fx_mu": torch.randn(B, D, generator=g),
         "fx_logvar": 0.3 * torch.randn(B, D, generator=g),
         "r_sqrt_sigma": torch.randn(L, Z, generator=g, dtype=torch.float64) / np.sqrt(Z)}
    t["y"][:, 0], t["y"][:, 1] = 1.0, 0.0
    t["y"][1], t["y"][4] = 0.0, 1.0
    noise = torch.randn(S, B, Z, generator=g)
    keep = torch.ones(B)
    keep[[1, 4]] = 0.0
    _, grads = RO.row_probit_elbo_with_grads(t, noise, 0.5, 10.0, {"total_loss": keep}, ranking="pairwise")
    for k, v in grads.items():
        assert bool(torch.isfinite(v).all()), k
    for k in ("fe_out", "fx_out", "fe_mu", "fe_logvar", "fx_mu", "fx_logvar"):
        assert torch.equal(grads[k][[1, 4]], torch.zeros_like(grads[k][[1, 4]])), k
    _, grads = RO.row_probit_elbo_with_grads(t, noise, 0.5, 10.0, {"total_loss": torch.ones(B)}, ranking="pairwise")
    assert bool(torch.isnan(grads["fe_out"][1]).all()) and bool(torch.isnan(grads["fe_out"][4]).all())


def test_header_declares_and_library_exports_the_row_entry_points(lib):
    """Additive entry points: the ABI version is unchanged, and so is mpvae_probit_params (test_lib_cpu pins its size
    and INTEGRATION.md's prefix of it)."""
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for sym in ("mpvae_probit_forward_rows", "mpvae_probit_backward_rows"):
        assert sym in declared_symbols()
        assert sym in _lib.EXPORTS
        assert hasattr(lib, sym)
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION == 13


def test_row_entry_points_validate_arguments_like_the_batch_ones(lib):
    from mpvae_b200 import _lib
    for f in (lib.mpvae_probit_forward_rows, lib.mpvae_probit_backward_rows):
        for mask, rw, lw in ((None, None, None), (256, 512, 1024)):
            p = _lib.ProbitParams()
            p.struct_bytes = 8
            assert f(C.byref(p), mask, rw, lw, None) == 1
            assert b"struct_bytes" in lib.mpvae_last_error()
            p.struct_bytes = C.sizeof(_lib.ProbitParams)
            p.S, p.B, p.L, p.Z = 10, 0, 14, 14
            assert f(C.byref(p), mask, rw, lw, None) == 1
            assert b"bad sizes" in lib.mpvae_last_error()
            p.B = 4
            assert f(C.byref(p), mask, rw, lw, None) == 1
            assert b"NULL input pointer" in lib.mpvae_last_error()


def test_bad_reduction_is_refused_before_any_noise_offset():
    from mpvae_b200 import mpvae
    case, t, _ = _golden("yeast_b16")
    args = orc.make_args(case["L"], case["Z"], n_train_sample=case["S"], mode="train")
    before = dict(mpvae._state)
    for bad in ("sum", "None", None, "MEAN"):
        with pytest.raises(ValueError, match="reduction"):
            mpvae.compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                               t["r_sqrt_sigma"], args, reduction=bad)
    assert mpvae._state == before
    with pytest.raises(RuntimeError, match="no CPU fallback"):   # a valid reduction reaches the device check
        mpvae.compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                           t["r_sqrt_sigma"], args, reduction="none")
    assert mpvae._state == before


def test_predict_proba_refuses_per_rows_without_labels():
    from mpvae_b200 import infer
    with pytest.raises(ValueError, match="labels"):
        infer.predict_proba(None, torch.zeros(3, 4), None, _args(), reduction="none")
    with pytest.raises(ValueError, match="reduction"):
        infer.predict_proba(None, torch.zeros(3, 4), torch.zeros(3, 2), _args(), reduction="sum")


# ---- data-parallel training with a row objective (gloo, CPU; the per-row oracle as loss_fn) ----

def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


def _small_loss(out, rows):
    """keep the rows whose detached total is at most the shard-independent threshold 40 (a fixed cut, so that shards
    select exactly what one process selects), plus half of nll_x on every row"""
    keep = (out[0].detach() <= 40.0).float()
    return keep * out[0] + 0.5 * out[2]


def test_row_objective_and_regulariser_are_refused_together():
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep
    args = _args()
    model = VAE(args)
    with pytest.raises(ValueError, match="row_objective or regulariser"):
        DataParallelStep(model, torch.optim.SGD(model.parameters(), lr=0.1), None, args, row_objective=_small_loss,
                         regulariser=lambda out, rows: None)


def _run_steps(n_steps=3, batch=11, loss_fn=RO.row_loss_fn, row_objective=_small_loss):
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
    stepper = DataParallelStep(model, opt, None, args, clip_norm=100.0, loss_fn=loss_fn, row_objective=row_objective)
    rng = np.random.RandomState(0)
    n = 23
    x = torch.from_numpy(rng.standard_normal((n, args.feature_dim)).astype(np.float32))
    y = torch.from_numpy((rng.uniform(size=(n, args.label_dim)) < 0.3).astype(np.float32))
    y[:, 0], y[:, 1] = 1.0, 0.0
    w = torch.from_numpy(rng.uniform(0.0, 3.0, size=n).astype(np.float32))
    w[[2, 9]] = 0.0
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


def test_row_objective_of_the_totals_is_the_weighted_mean_step():
    """One process, phi_b = total_b: the objective sum_b phi_b / B is the batch total_loss, so the steps and the returned
    scalars (the per-row means) agree with an ordinary weighted step up to rounding."""
    from tests import weighted_elbo_oracle as WO
    model, outs = _run_steps(row_objective=lambda out, rows: out[0])
    ref_model, ref_outs = _run_steps(loss_fn=WO.weighted_loss_fn, row_objective=None)
    ref = ref_model.state_dict()
    for k, v in model.state_dict().items():
        assert torch.allclose(v.double(), ref[k].double(), rtol=1e-5, atol=1e-6), k
    for got, want in zip(outs, ref_outs):
        for a, b in zip(got[:6], want[:6]):
            assert a.shape == () and abs(float(a) - float(b)) <= 1e-5 * max(1.0, abs(float(b)))


@pytest.mark.timeout(300)
def test_two_ranks_with_a_row_objective_equal_one_process():
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
