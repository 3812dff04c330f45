"""CPU checks of the label-free prediction path (mpvae_probit_predict / probit.probit_predict / mpvae.predict /
infer.predict_proba(labels=None)): the oracle restatement against the reference's recorded predictions, the C-ABI
surface and its argument checks, the host-side refusals, and the data-parallel scoring loop with the oracle injected."""
import ctypes as C
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import helpers as H
from tests import predict_oracle as PO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


@pytest.mark.parametrize("name", H.golden_names())
def test_oracle_predict_reproduces_reference_indiv_prob(name):
    """Bit for bit the indiv_prob of the full oracle (which test_oracle_golden pins to the reference's record) on the
    same host; and the record itself to within an ulp or two.  The record reproduces bit for bit only where the host's
    CPU BLAS splits the products as the recording host's did (test_oracle_golden.py::GOLDEN_THREADS)."""
    from oracle import probit_elbo_oracle as orc
    from tests.test_oracle_golden import GOLDEN_THREADS
    case = H.load_golden(name)
    if "indiv_prob" not in case["out"]:
        pytest.skip("fixture records no indiv_prob")
    t = H.to_torch(case["inputs"])
    noise = torch.from_numpy(case["noise"])
    before = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        got = PO.predict(t["fx_out"], t["r_sqrt_sigma"], noise)
        full = orc.probit_elbo(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                               t["r_sqrt_sigma"], noise, case["nll_coeff"], case["c_coeff"], ranking="factorised")
    finally:
        torch.set_num_threads(before)
    assert torch.equal(got, full.indiv_prob)
    assert float(np.max(np.abs(got.numpy().astype(np.float64) - case["out"]["indiv_prob"]))) <= 2.5e-7


def test_header_declares_and_library_exports_predict(lib):
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    assert "mpvae_probit_predict" in declared_symbols()
    assert "mpvae_probit_predict" in _lib.EXPORTS
    assert hasattr(lib, "mpvae_probit_predict")
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION


def test_predict_entry_point_validates_arguments(lib):
    """Refused before anything touches the device; the fields predict ignores may stay NULL."""
    from mpvae_b200 import _lib
    p = _lib.ProbitParams()
    p.struct_bytes = 8
    assert lib.mpvae_probit_predict(C.byref(p), None) == 1
    assert b"struct_bytes" in lib.mpvae_last_error()
    p.struct_bytes = C.sizeof(_lib.ProbitParams)
    p.S, p.B, p.L, p.Z = 10, 4, 14, 14
    assert lib.mpvae_probit_predict(C.byref(p), None) == 1
    assert b"NULL input pointer" in lib.mpvae_last_error()
    p.B = 0
    assert lib.mpvae_probit_predict(C.byref(p), None) == 1
    assert b"bad sizes" in lib.mpvae_last_error()
    # fx_out / r / workspace set (never dereferenced: validation fails first), no y, fe_out, mu/logvar or scalars
    p.B = 4
    p.fx_out, p.r, p.workspace = 256, 256, 256
    p.noise_b_global, p.noise_row0 = 4, 0
    assert lib.mpvae_probit_predict(C.byref(p), None) == 1
    assert b"NULL forward output pointer" in lib.mpvae_last_error()
    p.indiv_prob = 256
    p.workspace_bytes = 16
    assert lib.mpvae_probit_predict(C.byref(p), None) == 1
    assert b"workspace too small" in lib.mpvae_last_error()
    p.noise_b_global = 3
    assert lib.mpvae_probit_predict(C.byref(p), None) == 1
    assert b"library-side noise" in lib.mpvae_last_error()


def test_predict_refuses_cpu_tensors_and_bad_shapes():
    from mpvae_b200.mpvae import predict
    from mpvae_b200.probit import probit_predict
    from oracle import probit_elbo_oracle as orc
    case = H.load_golden("yeast_b16")
    t = H.to_torch(case["inputs"])
    args = orc.make_args(case["L"], case["Z"], n_test_sample=case["S"], mode="test")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        predict(t["fx_out"], t["r_sqrt_sigma"], args)
    r32 = t["r_sqrt_sigma"].float()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        probit_predict(t["fx_out"], r32, 4, noise_spec=(4, 1, 0, None, 0))
    B, L = t["fx_out"].shape
    Z = r32.shape[1]
    with pytest.raises(ValueError):
        probit_predict(t["fx_out"], r32[:-1], 4, noise_spec=(4, 1, 0, None, 0))      # R rows != label_dim
    with pytest.raises(ValueError):
        probit_predict(t["fx_out"], r32, 4, noise=torch.zeros(4, B + 1, Z))         # noise rows != batch
    with pytest.raises(ValueError):
        probit_predict(t["fx_out"], r32, 4, noise=torch.zeros(3, B, Z))             # noise samples != S
    with pytest.raises(ValueError):
        probit_predict(t["fx_out"][0], r32, 4, noise_spec=(4, 1, 0, None, 0))       # not (batch, label_dim)
    with pytest.raises(ValueError):
        probit_predict(t["fx_out"], r32, 4)                                          # neither noise nor spec


def test_predict_refuses_to_drop_a_graph():
    """Inference only: with grad mode on and an input that requires grad, predict says so instead of returning a tensor
    without a graph."""
    from mpvae_b200.mpvae import predict
    from oracle import probit_elbo_oracle as orc
    case = H.load_golden("yeast_b16")
    t = H.to_torch(case["inputs"])
    args = orc.make_args(case["L"], case["Z"], mode="test")
    r = torch.nn.Parameter(t["r_sqrt_sigma"])
    with pytest.raises(RuntimeError, match="inference only"):
        predict(t["fx_out"], r, args)
    with pytest.raises(RuntimeError, match="inference only"):
        predict(t["fx_out"].requires_grad_(True), t["r_sqrt_sigma"], args)


# ---- data-parallel label-free scoring (gloo, CPU; the oracle injected as predict_fn) ----

def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


def _score(n_rows, batch_size):
    """predict_proba(labels=None) over n_rows rows in this process (one rank of the group, or the whole job)."""
    sys.path.insert(0, ROOT)
    from mpvae_b200.infer import predict_proba
    from mpvae_b200.mpvae import VAE
    torch.set_num_threads(1)
    args = _args()
    np.random.seed(4)
    torch.manual_seed(0)
    model = VAE(args)
    model._reparameterize = lambda mu, logvar: mu       # the decoder on the posterior mean: no per-process randomness
    rng = np.random.RandomState(0)
    x = torch.from_numpy(rng.standard_normal((n_rows, args.feature_dim)).astype(np.float32))
    g = torch.Generator().manual_seed(77)
    full = torch.randn(args.n_test_sample, n_rows, args.z_dim, generator=g)
    seen = []

    def predict_fn(fx_out, r, a):
        seen.append((a.mode, a.dp_global_batch, a.dp_row0, fx_out.shape[0]))
        return PO.predict(fx_out, r, full[:, a.dp_row0:a.dp_row0 + fx_out.shape[0]])

    probs, sums = predict_proba(model, x, None, args, batch_size=batch_size, predict_fn=predict_fn)
    assert sums is None
    assert all(m == "test" and gb == n_rows for m, gb, _, _ in seen)
    return probs


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


# 23 rows: shards [0, 12) and [12, 23); a batch size of 12 gives the one process the same two batches, so every row sees
# the same CPU matmul shapes (CPU BLAS results depend on them) -- what is compared is the sharding, the global-row noise
# keys and the padded gather.  1 row: rank 1 owns nothing and still joins the gather.
@pytest.mark.timeout(300)
@pytest.mark.parametrize("n_rows,batch_size", [(23, 12), (1, 8)])
def test_two_ranks_label_free_equal_one_process(n_rows, batch_size):
    from mpvae_b200.train import shard_rows
    assert n_rows == 1 or shard_rows(n_rows, 0, 2) == (0, batch_size)
    got0, got1 = _two_ranks(n_rows, batch_size)
    want = _score(n_rows, batch_size)
    assert want.shape == (n_rows, _args().label_dim)
    assert torch.equal(got0, want) and torch.equal(got1, want)
