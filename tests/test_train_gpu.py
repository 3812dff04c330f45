"""GPU: the callers either side of the hot path -- the training step wrapper (train.py:103-129) and the
test-time inference loop (test.py:45-77) -- running on the real CUDA loss."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def yeast_args(**kw):
    a = SimpleNamespace(feature_dim=103, label_dim=14, latent_dim=50, z_dim=14, keep_prob=0.5, scale_coeff=1.0,
                        residue_sigma="", n_train_sample=10, n_test_sample=100, mode="train", nll_coeff=0.5,
                        c_coeff=10.0, batch_size=128, noise_seed=2024)
    a.__dict__.update(kw)
    return a


def yeast_data(n=1500, seed=0):
    from mpvae_b200 import synth
    rng = np.random.RandomState(seed)
    x = synth.features(n, 103, rng)
    w = rng.standard_normal((103, 14)).astype(np.float32) * 0.3
    y = ((x @ w + rng.standard_normal((n, 14)).astype(np.float32)) > 1.0).astype(np.float32)   # learnable labels
    y[:, 0], y[:, 1] = 1.0, 0.0
    return torch.from_numpy(x).to(DEV), torch.from_numpy(y).to(DEV)


def test_first_step_gradients_match_reference_loop():
    """One step of DataParallelStep (world 1) == the literal loop body with the oracle loss on the same device."""
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep
    args = yeast_args(keep_prob=0.0)
    x, y = yeast_data(256)
    np.random.seed(4); torch.manual_seed(0)
    ours = VAE(args).to(DEV)
    twin = VAE(args).to(DEV)
    twin.load_state_dict(ours.state_dict())
    opt = torch.optim.SGD(ours.parameters(), lr=0.0)
    step = DataParallelStep(ours, opt, None, args, clip_norm=1e9)
    noise = torch.randn(10, 128, 14, device=DEV)
    torch.manual_seed(7)
    out = step.step(y[:128], x[:128], noise=noise)
    torch.manual_seed(7)
    o = twin(y[:128], x[:128])
    terms = orc.compute_loss(y[:128], *o, twin.r_sqrt_sigma, args, noise=noise)
    terms[0].backward()
    assert H.rel_err(out.total_loss.item(), terms[0].item()) <= 1e-5
    for (n, p), (_, q) in zip(ours.named_parameters(), twin.named_parameters()):
        assert p.grad.dtype == q.grad.dtype, n
        assert H.rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) <= 2e-5, (n, H.rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()))


def test_training_reduces_the_loss_and_learns():
    """BASELINE.json configs[1]: yeast-shaped full train loop on 1 GPU (70/20/10 split, a few epochs)."""
    from mpvae_b200.infer import predict_proba
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep, train_one_epoch
    args = yeast_args()
    x, y = yeast_data(1500)
    n_train, n_valid = int(1500 * 0.7), int(1500 * 0.2)
    np.random.seed(4); torch.manual_seed(0)
    vae = VAE(args).to(DEV)
    opt = torch.optim.Adam(vae.parameters(), lr=1e-3, weight_decay=1e-5)
    sched = torch.optim.lr_scheduler.StepLR(opt, 9 * 5, 0.5)
    step = DataParallelStep(vae, opt, sched, args, clip_norm=100.0)
    first = last = None
    for epoch in range(12):
        order = torch.randperm(n_train, device=DEV)
        outs = train_one_epoch(step, x[:n_train], y[:n_train], 128, order)
        assert len(outs) == 9                       # int(1050/128)+1 steps, ragged last batch of 26 rows
        mean_total = float(torch.stack([o.total_loss for o in outs]).mean())
        first = mean_total if first is None else first
        last = mean_total
        assert all(torch.isfinite(o.grad_norm) for o in outs)
    assert last < 0.8 * first, (first, last)
    args_t = yeast_args(n_test_sample=100)
    probs, sums = predict_proba(vae, x[n_train:n_train + n_valid], y[n_train:n_train + n_valid], args_t, batch_size=128)
    assert probs.shape == (n_valid, 14)
    pred = (probs >= 0.5).float()
    yy = y[n_train:n_train + n_valid]
    tp = (pred * yy)[:, 2:].sum()
    f1 = 2 * tp / (pred[:, 2:].sum() + yy[:, 2:].sum() + 1e-6)
    assert f1 > 0.3, float(f1)                      # far above chance: the model has learned the synthetic rule


def test_inference_path_matches_oracle():
    """test.py:64-65: no_grad, eval, mode='test' => S = n_test_sample; predictions vs the oracle on the same noise."""
    from mpvae_b200.infer import predict_proba
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.probit import philox_normal
    args = yeast_args(n_test_sample=100, noise_seed=31, feature_dim=128, label_dim=81, z_dim=81)
    rng = np.random.RandomState(2)
    from mpvae_b200 import synth
    x = torch.from_numpy(synth.features(200, 128, rng)).to(DEV)
    y = torch.from_numpy(synth.labels(200, 81, 0.1, rng)).to(DEV)
    np.random.seed(4); torch.manual_seed(0)
    vae = VAE(args).to(DEV)
    probs, _ = predict_proba(vae, x, y, args, batch_size=128)
    # replay: same model outputs (eval mode is deterministic up to randn_like -> reseed), same Philox noise
    vae.eval()
    got = []
    with torch.no_grad():
        for i, (a, b) in enumerate(((0, 128), (128, 200))):
            noise = philox_normal(100, b - a, 81, seed=31, offset=i, device=DEV, global_batch=200, row0=a)
            torch.manual_seed(100 + i)
            o = vae(y[a:b], x[a:b])
            t_args = yeast_args(n_test_sample=100, mode="test", label_dim=81, z_dim=81)
            ref = orc.compute_loss(y[a:b], *o, vae.r_sqrt_sigma, t_args, noise=noise)
            torch.manual_seed(100 + i)
            args_i = yeast_args(n_test_sample=100, mode="test", noise_seed=31, noise_offset=i, dp_global_batch=200,
                                dp_row0=a, label_dim=81, z_dim=81)
            from mpvae_b200.mpvae import compute_loss
            mine = compute_loss(y[a:b], *vae(y[a:b], x[a:b]), vae.r_sqrt_sigma, args_i)
            assert H.threshold_mismatches(mine[6].cpu().numpy(), ref.indiv_prob.cpu().numpy()) == 0
            assert H.rel_err(mine[0].item(), ref.total_loss.item()) <= 1e-5
            got.append(mine[6])
    assert probs.shape == (200, 81)
    assert float(probs.min()) > 0 and float(probs.max()) < 1


def test_graphed_step_equals_eager_step():
    """GraphedTrainStep (CUDA-graph replay, device-side Philox counter) walks the same trajectory as the eager
    DataParallelStep when the host-visible randomness is removed (no dropout, collapsed posteriors)."""
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.train import DataParallelStep, GraphedTrainStep
    x, y = yeast_data(640)

    def build():
        args = yeast_args(keep_prob=0.0, noise_seed=77)
        np.random.seed(4); torch.manual_seed(0)
        vae = VAE(args).to(DEV)
        with torch.no_grad():
            for head in (vae.fe_logvar, vae.fx_logvar):
                head.weight.zero_(); head.bias.fill_(-30.0)
        opt = torch.optim.Adam(vae.parameters(), lr=torch.tensor(1e-3, device=DEV), weight_decay=1e-5, capturable=True)
        sched = torch.optim.lr_scheduler.StepLR(opt, 4, 0.5)
        return vae, DataParallelStep(vae, opt, sched, args, clip_norm=100.0)

    batches = [(y[i * 128:(i + 1) * 128], x[i * 128:(i + 1) * 128]) for i in range(5)]
    vae_g, st_g = build()
    graphed = GraphedTrainStep(st_g, warmup=3)
    losses_g = [float(graphed.step(*b).total_loss) for b in batches]
    vae_e, st_e = build()
    # the warm-up and the capture run on a snapshot that is restored: the first graphed step is exactly ONE update
    losses_e = [float(st_e.step(*b).total_loss) for b in batches]
    for a, b in zip(losses_g, losses_e):
        assert abs(a - b) <= 2e-4 * abs(b), (losses_g, losses_e)
    for (n, p), (_, q) in zip(vae_g.named_parameters(), vae_e.named_parameters()):
        assert torch.allclose(p.double(), q.double(), rtol=1e-3, atol=2e-5), n
    assert float(st_g.optimizer.param_groups[0]["lr"]) == pytest.approx(float(st_e.optimizer.param_groups[0]["lr"]))


# ----------------------------------------------------------------------------- fused clip + Adam (optim.py)
def test_fused_adam_matches_torch_adam():
    """mpvae_grad_norm + mpvae_adam_step against clip_grad_norm_ + torch.optim.Adam (train.py:93,126-128) on a mixed
    fp32 / fp64 parameter set, several steps, with and without the clip biting."""
    from mpvae_b200.optim import FusedAdam
    g = torch.Generator(device="cpu").manual_seed(5)
    shapes = [(37, 11), (11,), (300, 129), (129,)]

    def make():
        ps = [torch.nn.Parameter(torch.randn(s, generator=g).to(DEV)) for s in shapes]
        ps.append(torch.nn.Parameter((torch.randn(83, 83, generator=g).double() * 0.05).to(DEV)))   # r_sqrt_sigma-like
        return ps

    g.manual_seed(5); ref_p = make()
    g.manual_seed(5); my_p = make()
    ref = torch.optim.Adam(ref_p, lr=2e-3, weight_decay=1e-5)
    mine = FusedAdam(my_p, lr=2e-3, weight_decay=1e-5)
    for it, max_norm in enumerate((100.0, 0.5, 100.0, 0.05, 100.0)):
        grads = [torch.randn(p.shape, generator=g).to(DEV) * (0.1 + it) for p in ref_p]
        for p, q, gr in zip(ref_p, my_p, grads):
            p.grad = gr.to(p.dtype).clone()
            q.grad = gr.clone() if q.dtype == torch.float32 else None
        norm_ref = torch.nn.utils.clip_grad_norm_(ref_p, max_norm)
        ref.step()
        mine.step(max_norm=max_norm, f32_grads={my_p[-1]: grads[-1]})
        assert H.rel_err(mine.grad_norm.item(), norm_ref.item()) <= 1e-6
        for p, q in zip(ref_p, my_p):
            # fp64: torch carries the total norm in fp64 when an fp64 gradient takes part, the kernel reports it (and the
            # clip coefficient) in fp32 -- a 6e-8 relative difference of the coefficient, 1e-10 of the parameter
            tol = 2e-6 if p.dtype == torch.float32 else 1e-9
            assert H.rel_err(q.detach().cpu().numpy(), p.detach().cpu().numpy()) <= tol, (it, p.shape)
    sd = mine.state_dict()
    assert set(sd["state"][0].keys()) == {"step", "exp_avg", "exp_avg_sq"} and float(sd["state"][0]["step"]) == 5.0
    for a, b in zip(ref.state_dict()["state"].values(), sd["state"].values()):
        assert H.rel_err(b["exp_avg_sq"].cpu().numpy(), a["exp_avg_sq"].cpu().numpy()) <= 2e-6


def test_fused_step_equals_torch_step():
    """DataParallelStep with FusedAdam walks the same trajectory as with clip_grad_norm_ + torch.optim.Adam."""
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.optim import FusedAdam
    from mpvae_b200.train import DataParallelStep
    x, y = yeast_data(512)

    def build(fused):
        args = yeast_args(keep_prob=0.0, noise_seed=77)
        np.random.seed(4); torch.manual_seed(0)
        vae = VAE(args).to(DEV)
        with torch.no_grad():
            for head in (vae.fe_logvar, vae.fx_logvar):
                head.weight.zero_(); head.bias.fill_(-30.0)
        cls = FusedAdam if fused else torch.optim.Adam
        opt = cls(vae.parameters(), lr=1e-3, weight_decay=1e-5)
        sched = torch.optim.lr_scheduler.StepLR(opt, 2, 0.5)
        return vae, DataParallelStep(vae, opt, sched, args, clip_norm=1.0)     # a clip that bites

    batches = [(y[i * 128:(i + 1) * 128], x[i * 128:(i + 1) * 128]) for i in range(4)]
    vae_f, st_f = build(True)
    vae_t, st_t = build(False)
    for b in batches:
        of, ot = st_f.step(*b), st_t.step(*b)
        assert H.rel_err(float(of.total_loss), float(ot.total_loss)) <= 1e-5
        assert H.rel_err(float(of.grad_norm), float(ot.grad_norm)) <= 1e-5
    for (n, p), (_, q) in zip(vae_f.named_parameters(), vae_t.named_parameters()):
        assert p.dtype == q.dtype
        assert torch.allclose(p.double(), q.double(), rtol=1e-4, atol=2e-6), n
    assert float(st_f.optimizer.param_groups[0]["lr"]) == pytest.approx(float(st_t.optimizer.param_groups[0]["lr"]))
    # checkpoints keep the reference's layout: state_dict keys and dtypes unchanged by the flattening
    assert {k: v.dtype for k, v in vae_f.state_dict().items()} == {k: v.dtype for k, v in vae_t.state_dict().items()}


# ----------------------------------------------------------------------------- MLP layers on the tensor engine (dense.py)
@pytest.mark.parametrize("B,n_in,n_out,x_grad", [(1024, 5050, 256, True), (1024, 8993, 512, False), (1024, 512, 3993, True),
                                                 (128, 1483, 983, True)])
def test_tensor_linear_matches_fp64_linear(B, n_in, n_out, x_grad):
    """The large nn.Linear layers of VAE.forward run on the split-precision tcgen05 product: forward, input gradient and
    weight gradient must be as close to the exact (fp64) result as torch's fp32 SGEMM path is."""
    from mpvae_b200.dense import linear, uses_tensor_engine
    g = torch.Generator(device="cpu").manual_seed(B + n_in + n_out)
    layer = torch.nn.Linear(n_in, n_out).to(DEV)
    x = torch.randn(B, n_in, generator=g).to(DEV).requires_grad_(x_grad)
    gy = (torch.randn(B, n_out, generator=g) * 1e-3).to(DEV)
    assert uses_tensor_engine(layer, x)
    y = linear(layer, x)
    y.backward(gy)
    got = {"y": y.detach(), "gw": layer.weight.grad.clone(), "gb": layer.bias.grad.clone(), "gx": x.grad.clone() if x_grad else None}
    layer.zero_grad(); x.grad = None
    y_t = layer(x)
    y_t.backward(gy)
    ref32 = {"y": y_t.detach(), "gw": layer.weight.grad.clone(), "gb": layer.bias.grad.clone(), "gx": x.grad.clone() if x_grad else None}
    xd, wd, bd = x.detach().double(), layer.weight.detach().double(), layer.bias.detach().double()
    truth = {"y": xd @ wd.T + bd, "gw": gy.double().T @ xd, "gb": gy.double().sum(0), "gx": gy.double() @ wd}
    for k in ("y", "gw", "gb", "gx"):
        if got[k] is None:
            continue
        err = H.rel_err(got[k].cpu().numpy(), truth[k].cpu().numpy())
        err32 = H.rel_err(ref32[k].cpu().numpy(), truth[k].cpu().numpy())
        assert err <= max(3e-6, 2 * err32), (k, err, err32)
    # element by element, the split-precision product's error bound (tests/test_contract_bound_gpu.py): y less its bias
    # (plus the bias add's own rounding), gx = gy . W and gW = gy^T . x, K-sliced partial waves allowed
    xd32, wd32 = x.detach(), layer.weight.detach()
    H.assert_within_contract_bound(got["y"].double() - bd, xd32, wd32, ksplit=True, what="y",
                                   extra=2.0 ** -24 * ((xd.abs() @ wd.abs().T) + bd.abs()))
    H.assert_within_contract_bound(got["gw"], gy.T, xd32.T, ksplit=True, what="gW")
    if x_grad:
        H.assert_within_contract_bound(got["gx"], gy, wd32.T, ksplit=True, what="gx")


def test_fused_adam_state_dict_round_trip():
    """Checkpoint / resume: a FusedAdam restored from state_dict continues exactly where the original would have."""
    from mpvae_b200.optim import FusedAdam
    g = torch.Generator(device="cpu").manual_seed(9)

    def make():
        g.manual_seed(9)
        return [torch.nn.Parameter(torch.randn(50, 7, generator=g).to(DEV)),
                torch.nn.Parameter((torch.randn(31, 31, generator=g).double() * 0.1).to(DEV))]

    def feed(ps, k):
        gg = torch.Generator(device="cpu").manual_seed(100 + k)
        for p in ps:
            p.grad = torch.randn(p.shape, generator=gg).to(DEV).to(p.dtype)

    a = make()
    opt_a = FusedAdam(a, lr=3e-3, weight_decay=1e-5)
    for k in range(3):
        feed(a, k)
        opt_a.step(max_norm=1.0)
    b = make()
    with torch.no_grad():
        for p, q in zip(a, b):
            q.copy_(p)
    opt_b = FusedAdam(b, lr=3e-3, weight_decay=1e-5)
    opt_b.load_state_dict(opt_a.state_dict())
    assert float(opt_b.state_dict()["state"][0]["step"]) == 3.0
    for k in range(3, 6):
        feed(a, k); feed(b, k)
        opt_a.step(max_norm=1.0)
        opt_b.step(max_norm=1.0)
    for p, q in zip(a, b):
        assert torch.equal(p, q)


def test_reference_training_script_flow_on_the_device():
    """The whole of the reference's train.py flow with every replacement in place and no host round trip inside the
    loop: FusedAdam (train.py:93), the step (train.py:103-129) as a CUDA graph, the per-step metrics
    (train.py:131-136) as device scalars, and the final threshold sweep of the validation pass
    (train.py:277-289 / test.py:90-101) -- checked against the numpy restatement of evals.compute_metrics."""
    from oracle import evals_oracle as ev
    from mpvae_b200.infer import predict_proba
    from mpvae_b200.metrics import batch_metrics, sweep_metrics
    from mpvae_b200.mpvae import VAE
    from mpvae_b200.optim import FusedAdam
    from mpvae_b200.train import DataParallelStep, GraphedTrainStep
    args = yeast_args()
    x, y = yeast_data(1408)
    n_train = 1152                                           # nine full batches of 128: one captured graph
    np.random.seed(4); torch.manual_seed(0)
    vae = VAE(args).to(DEV)
    opt = FusedAdam(vae.parameters(), lr=torch.tensor(1e-3, device=DEV), weight_decay=1e-5)
    sched = torch.optim.lr_scheduler.StepLR(opt, 9 * 5, 0.5)
    graphed = GraphedTrainStep(DataParallelStep(vae, opt, sched, args, clip_norm=100.0))
    history = []
    for epoch in range(10):
        order = torch.randperm(n_train, device=DEV)
        for i in range(9):
            idx = order[i * 128:(i + 1) * 128]
            out = graphed.step(y[idx], x[idx])
            m = batch_metrics(out.indiv_prob, y[idx], 0.5)           # device scalars: nothing synchronises here
            history.append(torch.stack([out.total_loss.double(), m["miF1"], m["HA"]]))
    hist = torch.stack(history).cpu().numpy()                        # ONE transfer for the whole run
    assert np.isfinite(hist).all()
    assert hist[-9:, 0].mean() < 0.8 * hist[:9, 0].mean()            # the loss went down
    assert hist[-9:, 1].mean() > hist[:9, 1].mean()                  # micro-F1 went up
    assert float(opt.param_groups[0]["lr"]) == pytest.approx(0.25e-3)   # StepLR(45, 0.5) stepped 90 times
    # validation pass + threshold sweep on the device, against the numpy restatement on the same predictions
    args_t = yeast_args(n_test_sample=100)
    probs, _ = predict_proba(vae, x[n_train:], y[n_train:], args_t, batch_size=128)
    thresholds = [0.05, 0.25, 0.5, 0.75]
    got = sweep_metrics(probs, y[n_train:], thresholds)
    p_np, y_np = probs.cpu().numpy(), y[n_train:].cpu().numpy()
    for t, m in zip(thresholds, got):
        want = ev.full_metrics(p_np, y_np, t)
        for k in ("ACC", "HA", "ebF1", "miF1", "maF1", "p_at_1", "meanAUC", "medianAUPR", "varFDR"):
            a, b = m[k].item(), float(want[k])
            assert (np.isnan(a) and np.isnan(b)) or abs(a - b) <= 3e-6 * max(abs(b), 1.0), (t, k, a, b)
