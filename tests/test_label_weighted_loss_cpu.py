"""CPU checks of label-weighted training (compute_loss(..., pos_weight=, neg_weight=) /
mpvae_probit_forward_label_weighted / mpvae_probit_backward_label_weighted): the label-weighted oracle against the
weighted oracle (all-ones weights), against duplicated labels (integer weights), soft labels, zero and negative
weights; the C-ABI surface; the host-side refusals; and DataParallelStep with label weights on two gloo ranks against
one process, the label-weighted oracle as loss_fn."""
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
from tests import label_weighted_elbo_oracle as LO
from tests import weighted_elbo_oracle as WO
from tests.test_weighted_loss_cpu import TERMS, _golden, _random_case, _ranking, _same

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOGIT_LEAVES = ("fe_out", "fx_out")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


@pytest.mark.parametrize("name", H.golden_names())
@pytest.mark.parametrize("masked", [False, True])
def test_all_ones_label_weights_are_the_weighted_oracle_bit_for_bit(name, masked):
    """Random row weights (a zero among them) and, optionally, a random mask on both sides."""
    case, t, noise = _golden(name)
    up = {k: torch.from_numpy(v) for k, v in case["upstream"].items()} or None
    kw = dict(ranking=_ranking(case["L"]))
    B, L = t["y"].shape
    g = torch.Generator().manual_seed(B + 3 * L)
    mask = (torch.rand(B, L, generator=g) < 0.6) if masked else None
    w = torch.rand(B, generator=g) * 2.0
    w[B // 2] = 0.0
    want, want_g = WO.weighted_probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], w, mask, upstream=up, **kw)
    got, got_g = LO.label_weighted_probit_elbo_with_grads(t, noise, case["nll_coeff"], case["c_coeff"], torch.ones(2, L), w,
                                                          mask, upstream=up, **kw)
    for k in TERMS:
        assert _same(getattr(got, k), getattr(want, k)), k
    for k in want_g:
        assert (got_g[k] is None) == (want_g[k] is None), k
        if want_g[k] is not None:
            assert _same(got_g[k], want_g[k]), k


def _duplicate_labels(t, counts):
    """label l's column of y / fe_out / fx_out and row of R repeated counts[l] times (0: dropped)"""
    idx = torch.repeat_interleave(torch.arange(len(counts)), torch.as_tensor(counts))
    d = {k: (v[idx] if k == "r_sqrt_sigma" else v[:, idx] if k in ("y", "fe_out", "fx_out") else v) for k, v in t.items()}
    return d, idx


@pytest.mark.parametrize("ranking", ["pairwise", "factorised"])
@pytest.mark.parametrize("masked", [False, True])
def test_integer_weights_equal_duplicated_labels(ranking, masked):
    """The same integer k_l (0 included) on both rows of label l against the unweighted problem with label l's column
    and R row repeated k_l times, in fp64: nll_loss and nll_loss_x agree, and so do their gradients with respect to the
    logits (summed over a label's copies) and R (summed over a row's copies)."""
    S, B, L, Z = 5, 7, 9, 4
    t, noise, g = _random_case(S, B, L, Z, seed=11)
    counts = [1, 3, 0, 2, 1, 1, 4, 0, 2]
    mask = None
    if masked:
        mask = torch.rand(B, L, generator=g) < 0.7
    t64 = {k: v.double() for k, v in t.items()}
    lw = torch.tensor(counts, dtype=torch.float64).expand(2, L)
    up = {"nll_loss": torch.tensor(0.7, dtype=torch.float64), "nll_loss_x": torch.tensor(1.3, dtype=torch.float64)}
    got, got_g = LO.label_weighted_probit_elbo_with_grads(t64, noise.double(), 0.5, 10.0, lw, None, mask, ranking=ranking,
                                                          dtype=torch.float64, upstream=up)
    d, idx = _duplicate_labels(t64, counts)
    dmask = mask[:, idx] if mask is not None else None
    want, want_g = WO.weighted_probit_elbo_with_grads(d, noise.double(), 0.5, 10.0, torch.ones(B, dtype=torch.float64),
                                                      dmask, ranking=ranking, dtype=torch.float64, upstream=up)
    for i in (1, 2):
        assert abs(float(got[i].detach()) - float(want[i].detach())) <= 1e-12 * max(1.0, abs(float(want[i].detach()))), TERMS[i]
    for k in LOGIT_LEAVES:
        summed = torch.zeros_like(got_g[k]).index_add_(1, idx, want_g[k])
        assert torch.allclose(got_g[k], summed, rtol=1e-10, atol=1e-13), k
        assert torch.equal(got_g[k][:, [2, 7]], torch.zeros_like(got_g[k][:, [2, 7]])), k
    summed = torch.zeros_like(got_g["r_sqrt_sigma"]).index_add_(0, idx, want_g["r_sqrt_sigma"])
    assert torch.allclose(got_g["r_sqrt_sigma"], summed, rtol=1e-10, atol=1e-13)


def _direct_nll(t, noise, lw, mask=None):
    """nll_loss, nll_loss_x of the weighted cell formula written out in fp64 with logsumexp (no where, no ranking)"""
    y, R = t["y"].double(), t["r_sqrt_sigma"].double()
    m = torch.ones_like(y) if mask is None else mask.double()
    nr = torch.einsum("sbz,lz->sbl", noise.double(), R)
    out = []
    for f in ("fe_out", "fx_out"):
        x = nr + t[f].double()
        E = (0.5 * (1 + torch.erf(x / np.sqrt(2)))) * (1 - 1e-6) + 0.5e-6
        ll = lw[1] * y * torch.log(E) + lw[0] * (1 - y) * torch.log(1 - E)
        lp = torch.sum(ll * m, dim=2)
        out.append(float(torch.mean(-(torch.logsumexp(lp, dim=0) - np.log(lp.shape[0])))))
    return out


@pytest.mark.parametrize("kind", ["soft", "zero", "negative"])
def test_soft_zero_and_negative_weights(kind):
    """Soft labels with random weights, zero weights (also: both zero on a label = that label's likelihood left out),
    and negative weights, in fp64 against the formula written out; a zero-weight cell's log-likelihood gradient is 0."""
    S, B, L, Z = 6, 5, 8, 3
    t, noise, g = _random_case(S, B, L, Z, seed=5)
    t64 = {k: v.double() for k, v in t.items()}
    lw = torch.rand(2, L, generator=g, dtype=torch.float64) * 3.0
    if kind == "soft":
        t64["y"][:, 4:] = torch.rand(B, L - 4, generator=g, dtype=torch.float64)
    elif kind == "zero":
        lw[:, 3] = 0.0
        lw[0, 5] = 0.0
        lw[1, 6] = 0.0
    else:
        lw[:, 2:5] *= -1.0
    up = {"nll_loss": torch.tensor(1.0, dtype=torch.float64), "nll_loss_x": torch.tensor(1.0, dtype=torch.float64)}
    got, got_g = LO.label_weighted_probit_elbo_with_grads(t64, noise.double(), 0.5, 10.0, lw, ranking="pairwise",
                                                          dtype=torch.float64, upstream=up)
    want = _direct_nll(t64, noise, lw)
    for i, w in zip((1, 2), want):
        assert abs(float(got[i].detach()) - w) <= 1e-12 * max(1.0, abs(w)), (i, float(got[i].detach()), w)
    if kind == "zero":
        for k in LOGIT_LEAVES:
            assert torch.equal(got_g[k][:, 3], torch.zeros(B, dtype=torch.float64)), k
            zero_cells = torch.cat([(t64["y"][:, 5] == 0), (t64["y"][:, 6] == 1)])
            assert torch.equal(got_g[k][:, [5, 6]].T.flatten()[zero_cells], torch.zeros(int(zero_cells.sum()), dtype=torch.float64))
        hidden = torch.ones(B, L, dtype=torch.bool)
        hidden[:, 3] = False
        ref = _direct_nll(t64, noise, lw, hidden)
        for i, w in zip((1, 2), ref):
            assert abs(float(got[i].detach()) - w) <= 1e-12 * max(1.0, abs(w))


def test_header_declares_and_library_exports_the_label_weighted_entry_points(lib):
    """Additive entry points: the ABI version and mpvae_probit_params are unchanged."""
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for sym in ("mpvae_probit_forward_label_weighted", "mpvae_probit_backward_label_weighted"):
        assert sym in declared_symbols()
        assert sym in _lib.EXPORTS
        assert hasattr(lib, sym)
        assert len(getattr(lib, sym).argtypes) == 5
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION == 13


def test_label_weighted_entry_points_validate_arguments(lib):
    """Refused before anything touches the device, with the unweighted calls' messages."""
    from mpvae_b200 import _lib
    for f in (lib.mpvae_probit_forward_label_weighted, lib.mpvae_probit_backward_label_weighted):
        for mask, weight, lw in ((None, None, 1024), (256, 512, 1024), (None, None, None)):
            p = _lib.ProbitParams()
            p.struct_bytes = 8
            assert f(C.byref(p), mask, weight, lw, None) == 1
            assert b"struct_bytes" in lib.mpvae_last_error()
            p.struct_bytes = C.sizeof(_lib.ProbitParams)
            p.S, p.B, p.L, p.Z = 10, 0, 14, 14
            assert f(C.byref(p), mask, weight, lw, None) == 1
            assert b"bad sizes" in lib.mpvae_last_error()
            p.B = 4
            assert f(C.byref(p), mask, weight, lw, None) == 1
            assert b"NULL input pointer" in lib.mpvae_last_error()


def test_label_weight_host_refusals():
    from mpvae_b200 import mpvae
    from mpvae_b200.probit import _check_label_weight
    case, t, noise = _golden("yeast_b16")
    args = orc.make_args(case["L"], case["Z"], n_train_sample=case["S"], mode="train")
    L = t["y"].shape[1]
    ok = torch.ones(L)
    call = lambda **kw: mpvae.compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"],  # noqa: E731
                                           t["fx_logvar"], t["r_sqrt_sigma"], args, **kw)
    before = dict(mpvae._state)
    # refused before the device check and before noise_plan: no noise offset is consumed
    for name in ("pos_weight", "neg_weight"):
        with pytest.raises(ValueError, match="requires grad"):
            call(**{name: ok.clone().requires_grad_(True)})
        with pytest.raises(ValueError, match="shape"):
            call(**{name: ok[:-1]})
        with pytest.raises(TypeError, match="floating"):
            call(**{name: ok.to(torch.int64)})
    assert mpvae._state == before
    with pytest.raises(RuntimeError, match="no CPU fallback"):   # valid weights reach the device check
        call(pos_weight=ok, neg_weight=ok)
    assert mpvae._state == before
    cuda = torch.device("cuda:0")
    with pytest.raises(ValueError, match="is on"):
        _check_label_weight(ok, None, L, cuda)
    with pytest.raises(TypeError, match="floating"):
        _check_label_weight(None, ok.numpy(), L, cpu := torch.device("cpu"))
    with pytest.raises(ValueError, match="shape"):
        _check_label_weight(ok[None], None, L, cpu)
    assert _check_label_weight(None, None, L, cpu) is None
    pos = torch.arange(2 * L, dtype=torch.float64)[::2]
    lw = _check_label_weight(pos, None, L, cpu)
    assert lw.dtype == torch.float32 and lw.is_contiguous() and lw.shape == (2, L)
    assert torch.equal(lw[0], torch.ones(L)) and torch.equal(lw[1], pos.float())
    lw = _check_label_weight(None, ok.half() * 3, L, cpu)
    assert torch.equal(lw, torch.stack([torch.full((L,), 3.0), torch.ones(L)]))


# ---- data-parallel training with label weights (gloo, CPU; the label-weighted oracle as loss_fn) ----

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
    with torch.no_grad():
        for head in (model.fe_logvar, model.fx_logvar):
            head.weight.zero_(); head.bias.fill_(-30.0)
    opt = torch.optim.SGD(model.parameters(), lr=0.05, weight_decay=1e-5)
    stepper = DataParallelStep(model, opt, None, args, clip_norm=100.0, loss_fn=LO.label_weighted_loss_fn)
    rng = np.random.RandomState(0)
    n = 23
    x = torch.from_numpy(rng.standard_normal((n, args.feature_dim)).astype(np.float32))
    y = torch.from_numpy((rng.uniform(size=(n, args.label_dim)) < 0.3).astype(np.float32))
    y[:, 0], y[:, 1] = 1.0, 0.0
    pos = torch.from_numpy(rng.uniform(0.5, 4.0, size=args.label_dim).astype(np.float32))
    neg = torch.from_numpy(rng.uniform(0.0, 1.5, size=args.label_dim).astype(np.float32))
    pos[3], neg[5] = 0.0, -0.5
    w = torch.from_numpy(rng.uniform(0.0, 2.0, size=n).astype(np.float32))
    outs = []
    for i in range(n_steps):
        idx = torch.arange(i * 6, i * 6 + batch) % n
        noise = torch.randn(args.n_train_sample, batch, args.z_dim, generator=torch.Generator().manual_seed(1000 + i))
        outs.append(stepper.step(y[idx], x[idx], noise=noise, row_weight=w[idx], pos_weight=pos, neg_weight=neg))
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
def test_two_ranks_with_label_weights_equal_one_process():
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
