"""CPU checks of the sampled predictors' row gather (infer._score_rows): infer.predict_sets and infer.predict_mode over
two gloo ranks return what one process returns, bit for bit, field by field (bool, int32 and fp64 fields, fp64 values
that fp32 cannot hold), also when one rank owns no rows.  The predictors are replaced by deterministic stand-ins keyed
by the global row, so the test needs no GPU."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _args():
    return SimpleNamespace(feature_dim=12, label_dim=9, latent_dim=6, z_dim=5, keep_prob=0.0, scale_coeff=1.0,
                           residue_sigma="", n_train_sample=4, n_test_sample=6, mode="train", nll_coeff=0.5,
                           c_coeff=10.0, batch_size=8)


def _fields(fx_out, a):
    """Per-row fields of a predictor result from fx_out and the global rows of the batch: a (B, L) bool set, fp64
    values with bits below fp32's precision, and int32 values above 2^24."""
    rows = torch.arange(a.dp_row0, a.dp_row0 + fx_out.shape[0], dtype=torch.int64)
    f64 = fx_out.double().sum(1) * (1.0 + 2.0 ** -40) + rows.double() * 1e-13
    return fx_out > 0, f64, (rows + (1 << 28) + 3).to(torch.int32)


def _score(kind, n_rows, batch_size):
    """infer.predict_sets or infer.predict_mode over n_rows rows in this process (one rank of the group, or the job)."""
    sys.path.insert(0, ROOT)
    from mpvae_b200 import infer, mpvae
    from mpvae_b200.mpvae import VAE
    torch.set_num_threads(1)
    args = _args()
    np.random.seed(4)
    torch.manual_seed(0)
    model = VAE(args)
    model._reparameterize = lambda mu, logvar: mu       # the decoder on the posterior mean: no per-process randomness
    rng = np.random.RandomState(0)
    x = torch.from_numpy(rng.standard_normal((n_rows, args.feature_dim)).astype(np.float32))
    seen = []

    def sets(fx_out, r, a, beta=1.0, max_size=None, noise=None):
        seen.append((a.mode, a.dp_global_batch, fx_out.shape[0]))
        return mpvae.SetPrediction(*_fields(fx_out, a))

    def mode(fx_out, r, a, max_flips=None, noise=None):
        seen.append((a.mode, a.dp_global_batch, fx_out.shape[0]))
        s, f64, big = _fields(fx_out, a)
        return mpvae.ModePrediction(s, f64, -f64 / 3.0, s.sum(1, dtype=torch.int32), big)

    real = mpvae.predict_sets, mpvae.predict_mode
    mpvae.predict_sets, mpvae.predict_mode = sets, mode
    try:
        if kind == "sets":
            res = infer.predict_sets(model, x, args, batch_size=batch_size)
        else:
            res = infer.predict_mode(model, x, args, batch_size=batch_size)
    finally:
        mpvae.predict_sets, mpvae.predict_mode = real
    assert seen and all(m == "test" and gb == n_rows for m, gb, _ in seen)
    assert type(res) is (mpvae.SetPrediction if kind == "sets" else mpvae.ModePrediction)
    return res


def _worker(rank, world, port, kind, n_rows, batch_size, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret[rank] = tuple(_score(kind, n_rows, batch_size))
    finally:
        dist.destroy_process_group()


def _two_ranks(kind, n_rows, batch_size):
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, n_rows, batch_size, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(240)
        assert p.exitcode == 0
    return ret[0], ret[1]


# 23 rows: shards [0, 12) and [12, 23), the one process in batches of 12; 1 row: rank 1 owns nothing and still joins
# the gather
@pytest.mark.timeout(300)
@pytest.mark.parametrize("kind", ["sets", "mode"])
@pytest.mark.parametrize("n_rows,batch_size", [(23, 12), (1, 8)])
def test_two_ranks_equal_one_process(kind, n_rows, batch_size):
    want = _score(kind, n_rows, batch_size)
    L = _args().label_dim
    dtypes = [torch.bool, torch.float64, torch.int32] if kind == "sets" else \
        [torch.bool, torch.float64, torch.float64, torch.int32, torch.int32]
    assert [f.dtype for f in want] == dtypes
    assert [tuple(f.shape) for f in want] == [(n_rows, L)] + [(n_rows,)] * (len(dtypes) - 1)
    f64 = want[1]
    assert not torch.equal(f64.float().double(), f64)       # an fp32 round trip would show
    got0, got1 = _two_ranks(kind, n_rows, batch_size)
    for got in (got0, got1):
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert g.dtype == w.dtype and g.shape == w.shape
            assert torch.equal(g.view(torch.uint8) if g.dtype == torch.bool else g,
                               w.view(torch.uint8) if w.dtype == torch.bool else w)
