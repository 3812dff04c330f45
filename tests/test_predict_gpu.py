"""GPU: the label-free prediction path (mpvae_probit_predict: probit_predict_rows_kernel after the nt product, or the
one-launch probit_small_predict_kernel) against the loss path's indiv_prob, the oracle, itself over row windows, and at
the model level through infer.predict_proba(labels=None)."""
import copy
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import helpers as H
from tests import predict_oracle as PO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

STABLE, FMA, TENSOR, SEPARATE, FUSED = 0x8, 0x4, 0x2, 0x20, 0x10


def _inputs(S, B, L, Z, external, seed):
    from mpvae_b200 import synth
    inp = synth.loss_inputs(L, Z, B, S, seed=seed, sigma=1.0, label_rate=max(0.05, 20.0 / L), with_noise=external)
    t = {k: torch.from_numpy(v).to(DEV) for k, v in inp.items()}
    return t, t.pop("noise", None)


def _args(S, L, Z, flags=0, **kw):
    return orc.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=4242, noise_offset=6, mpvae_flags=flags, **kw)


def _loss_and_predict(t, noise, args):
    from mpvae_b200.mpvae import compute_loss, predict
    with torch.no_grad():
        loss = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                            t["r_sqrt_sigma"], args, noise=noise)[6]
        pred = predict(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
    torch.cuda.synchronize()
    return loss, pred


# (S, B, L, Z, flags, external noise): small regime (mirflickr, yeast, NUS-WIDE shapes), the CUDA-core regime (eurlex L with
# Z = 10, and whatever CONTRACT_FMA / STABLE_CDF send there), the dense regime (delicious, eurlex at S = 100, B = 1024);
# S in {1, 3, 10, 100}, ragged B, L not a multiple of 4 or of 128
EQUALITY_CASES = [
    (10, 16, 38, 38, 0, False), (10, 16, 38, 38, 0, True), (1, 5, 14, 14, 0, False), (3, 33, 14, 14, 0, True),
    (100, 128, 81, 81, 0, False), (100, 37, 81, 81, 0, True),
    (10, 33, 3993, 10, 0, False), (3, 17, 3993, 10, 0, True), (100, 12, 983, 10, 0, False), (1, 9, 983, 10, 0, False),
    (10, 16, 38, 38, STABLE, False), (100, 7, 81, 81, STABLE, True), (10, 70, 983, 983, FMA, False), (3, 9, 130, 64, FMA, True),
    (10, 70, 983, 983, 0, False), (10, 70, 983, 983, 0, True), (3, 77, 130, 256, 0, True), (100, 12, 300, 128, SEPARATE, False),
    (1, 300, 256, 256, 0, False), (7, 5, 130, 64, TENSOR, False), (10, 40, 257, 300, STABLE, False),
    (10, 33, 513, 130, FUSED, False), (3, 19, 983, 983, SEPARATE, True), (100, 1024, 3993, 3993, 0, False),
]


@pytest.mark.parametrize("S,B,L,Z,flags,external", EQUALITY_CASES)
def test_predict_equals_the_loss_path(S, B, L, Z, flags, external):
    """predict(fx_out, R, args) is compute_loss(..., mode='test')[6] bit for bit: same regime, same E, same sample order."""
    t, noise = _inputs(S, B, L, Z, external, seed=S + B + L)
    loss, pred = _loss_and_predict(t, noise, _args(S, L, Z, flags))
    assert pred.shape == (B, L) and torch.isfinite(pred).all()
    assert torch.equal(loss, pred)


@pytest.mark.parametrize("S,B,L,Z,flags", [(100, 128, 81, 81, 0), (10, 33, 983, 10, 0), (10, 70, 983, 983, 0),
                                           (3, 77, 130, 256, 0), (10, 16, 38, 38, STABLE), (10, 70, 300, 256, STABLE)])
def test_predict_against_the_oracle(S, B, L, Z, flags):
    """The library's Philox noise, handed to the oracle through philox_normal: within 1e-5, and the thresholded decisions
    identical away from ties (the bar of the loss path's inference test)."""
    from mpvae_b200.mpvae import predict
    from mpvae_b200.probit import philox_normal
    t, _ = _inputs(S, B, L, Z, False, seed=3 * S + B)
    with torch.no_grad():
        pred = predict(t["fx_out"], t["r_sqrt_sigma"], _args(S, L, Z, flags))
        noise = philox_normal(S, B, Z, seed=4242, offset=6, device=DEV)
        ref = PO.predict(t["fx_out"], t["r_sqrt_sigma"], noise, stable=bool(flags & STABLE))
    got, want = pred.cpu().numpy(), ref.cpu().numpy()
    dp = float(np.max(np.abs(got.astype(np.float64) - want)))
    assert dp <= 1e-5, dp
    assert H.threshold_mismatches(got, want, tie=2 * dp + 1e-7) == 0


@pytest.mark.parametrize("S,L,Z,flags,windows", [
    (100, 81, 81, 0, [(0, 1), (1, 64), (64, 100)]),                 # small regime
    (10, 983, 10, 0, [(0, 37), (37, 38), (38, 100)]),               # CUDA-core regime
    (10, 983, 983, TENSOR, [(0, 5), (5, 61), (61, 100)]),           # dense regime (kept there for the 5-row window)
    (3, 300, 256, STABLE | TENSOR, [(0, 50), (50, 100)]),
])
def test_predictions_do_not_depend_on_batching(S, L, Z, flags, windows):
    """A row's prediction depends on its global row key, not on the rows it is scored with: one call over N rows equals
    the concatenation of calls over row windows (library noise keyed by the global row), bit for bit."""
    from mpvae_b200.mpvae import predict
    N = windows[-1][1]
    t, _ = _inputs(S, N, L, Z, False, seed=N + L)
    with torch.no_grad():
        full = predict(t["fx_out"], t["r_sqrt_sigma"], _args(S, L, Z, flags, dp_global_batch=N, dp_row0=0))
        parts = [predict(t["fx_out"][lo:hi], t["r_sqrt_sigma"], _args(S, L, Z, flags, dp_global_batch=N, dp_row0=lo))
                 for lo, hi in windows]
    assert torch.equal(torch.cat(parts, 0), full)


@pytest.mark.parametrize("S,B,L,Z,flags,external,small", [
    (100, 128, 81, 81, 0, False, True), (10, 16, 38, 38, 0, True, True),
    (10, 33, 3993, 10, 0, False, False), (10, 33, 3993, 10, 0, True, False),
    (10, 70, 983, 983, 0, False, False), (10, 70, 983, 983, 0, True, False), (10, 70, 983, 983, SEPARATE, False, False),
])
def test_launch_count(S, B, L, Z, flags, external, small):
    """Small regime: one launch.  Otherwise the test-mode forward's launches up to and including the product, then ONE
    row kernel -- where the forward runs two (the tiled cell kernel and the per-row finalize)."""
    from mpvae_b200 import _lib
    from mpvae_b200.mpvae import compute_loss, predict
    t, noise = _inputs(S, B, L, Z, external, seed=5)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        n0 = _lib.launch_count()
        compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                     t["r_sqrt_sigma"], args, noise=noise)
        n1 = _lib.launch_count()
        predict(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
        n2 = _lib.launch_count()
    torch.cuda.synchronize()
    n_loss, n_pred = n1 - n0, n2 - n1
    if small:
        assert n_loss == 1 and n_pred == 1, (n_loss, n_pred)
    else:
        assert n_pred == n_loss - 1, (n_loss, n_pred)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (100, 33, 81, 81, 0), (10, 33, 983, 10, 0),
                                           (7, 33, 513, 130, 0), (10, 128, 983, 983, 0), (3, 77, 130, 256, SEPARATE),
                                           (10, 40, 257, 300, STABLE)])
def test_poisoned_workspace_gives_the_same_bits(S, B, L, Z, flags, monkeypatch):
    """With MPVAE_POISON_WORKSPACE=1 the scratch and the output start as 0xFF bytes: nothing is read before it is written."""
    from mpvae_b200.mpvae import predict
    t, _ = _inputs(S, B, L, Z, False, seed=S + L)
    with torch.no_grad():
        clean = predict(t["fx_out"], t["r_sqrt_sigma"], _args(S, L, Z, flags))
        monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
        poisoned = predict(t["fx_out"], t["r_sqrt_sigma"], _args(S, L, Z, flags))
    assert torch.isfinite(poisoned).all()
    assert torch.equal(clean, poisoned)


def test_empty_batch_and_offset_consumption():
    """B == 0 returns an empty (0, L) tensor; without args.noise_offset a call consumes one offset, as compute_loss does."""
    from mpvae_b200 import mpvae
    L, Z = 14, 14
    args = orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9)
    with torch.no_grad():
        out = mpvae.predict(torch.empty(0, L, device=DEV), torch.zeros(L, Z, dtype=torch.float64, device=DEV), args)
    assert out.shape == (0, L)
    t, _ = _inputs(10, 8, L, Z, False, seed=1)
    mpvae.set_noise_seed(77, offset=3)
    with torch.no_grad():
        a = mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], args)
        b = mpvae.compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                               t["r_sqrt_sigma"], args)[6]
        c = mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9,
                                                                         noise_offset=3))
        d = mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], orc.make_args(L, Z, n_test_sample=10, mode="test", noise_seed=9,
                                                                         noise_offset=4))
    assert torch.equal(a, c) and torch.equal(b, d) and not torch.equal(a, b)


def _yeast_args(**kw):
    a = SimpleNamespace(feature_dim=103, label_dim=14, latent_dim=50, z_dim=14, keep_prob=0.5, scale_coeff=1.0,
                        residue_sigma="", n_train_sample=10, n_test_sample=100, mode="train", nll_coeff=0.5,
                        c_coeff=10.0, batch_size=128, noise_seed=2024)
    a.__dict__.update(kw)
    return a


def _yeast_data(n=1500, seed=0):
    from mpvae_b200 import synth
    rng = np.random.RandomState(seed)
    x = synth.features(n, 103, rng)
    w = rng.standard_normal((103, 14)).astype(np.float32) * 0.3
    y = ((x @ w + rng.standard_normal((n, 14)).astype(np.float32)) > 1.0).astype(np.float32)   # learnable labels
    y[:, 0], y[:, 1] = 1.0, 0.0
    return torch.from_numpy(x).to(DEV), torch.from_numpy(y).to(DEV)


def _f1(probs, y):
    pred = (probs >= 0.5).float()
    tp = (pred * y)[:, 2:].sum()
    return float(2 * tp / (pred[:, 2:].sum() + y[:, 2:].sum() + 1e-6))


def test_label_free_scoring_of_a_trained_model():
    """The setup of test_train_gpu.py::test_training_reduces_the_loss_and_learns.  (1) predict_proba(labels=None) is the
    hand loop feat_forward + mpvae.predict under the same torch seed, bit for bit; (2) its thresholded F1 on held-out
    rows clears the bar the label path clears there."""
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_proba
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
    torch.manual_seed(11)
    probs, sums = predict_proba(vae, xv, None, args, batch_size=128)
    assert sums is None and probs.shape == (n_valid, 14)
    # the hand loop
    vae.eval()
    a_t = copy.copy(args)
    a_t.mode = "test"
    hand = []
    torch.manual_seed(11)
    with torch.no_grad():
        for lo in range(0, n_valid, 128):
            hi = min(lo + 128, n_valid)
            a_t.dp_global_batch, a_t.dp_row0, a_t.noise_offset = n_valid, lo, 0
            hand.append(mpvae.predict(vae.feat_forward(xv[lo:hi])[0], vae.r_sqrt_sigma, a_t))
    assert torch.equal(torch.cat(hand, 0), probs)
    f1_free = _f1(probs, yv)
    f1_label, _ = predict_proba(vae, xv, yv, args, batch_size=128)
    f1_label = _f1(f1_label, yv)
    assert f1_free > 0.3 and f1_label > 0.3, (f1_free, f1_label)
