"""GPU: mode prediction (mpvae_probit_score_sets and mpvae_probit_predict_mode: predict's nt product, then
probit_mode_rows_kernel, mode_score_kernel and mode_ascent_kernel) against the fp64 oracle on the library's own E,
against the library's scorer in every regime, an exhaustive search, the R = 0 identities, the links to
predict_conditional and the loss, a planted model where the mode beats thresholding on exact match, the invariants
under batching, repetition and a poisoned workspace, launch counts, and infer.predict_mode."""
import copy
import math

import numpy as np
import pytest
import torch

from tests import predict_mode_oracle as MO
from tests import predict_sets_oracle as SO
from tests.test_predict_gpu import _args, _inputs, _yeast_args, _yeast_data

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

STABLE, FMA, TENSOR, SEPARATE = 0x8, 0x4, 0x2, 0x20


def _dense(S, B, L, Z, flags):
    """Whether the library takes the tcgen05 product for this call (capi.cu use_tensor)."""
    if flags & FMA or Z < 8 or L < 8:
        return False
    return bool(flags & TENSOR) or (Z >= 128 and L >= 128 and S * B >= 128)


def _weak(B, L, Z, seed, spread=0.3, load=0.5):
    """fx_out and R of a model with weak loadings on many directions, whose mixtures often have a mode that is neither
    a sample's mode nor the thresholded marginals."""
    g = torch.Generator().manual_seed(seed)
    fx = (torch.randn(B, L, generator=g) * spread).to(DEV)
    r = (torch.randn(L, Z, generator=g, dtype=torch.float64) * load).to(DEV)
    return fx, r


def _slice_E(fx, r, noise, args):
    """(S, B, L) E of each sample: predict(S = 1) on each noise slice, checked bit-equal to the E of the S-sample call
    (sample_labels compares U < E: U = E_slice gives 0 and U = the next fp32 below E_slice gives 1 only where the
    in-batch E equals E_slice)."""
    from mpvae_b200.mpvae import predict, sample_labels, unpack_label_samples
    S, L = noise.shape[0], fx.shape[1]
    a1 = copy.copy(args)
    a1.n_test_sample = 1
    E = torch.stack([predict(fx, r, a1, noise=noise[s:s + 1]) for s in range(S)])
    below = torch.nextafter(E, torch.zeros_like(E))
    at = unpack_label_samples(sample_labels(fx, r, args, noise=noise, uniform=E), L).transpose(0, 1)
    under = unpack_label_samples(sample_labels(fx, r, args, noise=noise, uniform=below), L).transpose(0, 1)
    assert not bool(at.any()) and bool(under.all()), "a slice's E differs from the in-batch E"
    return E


def _all_neighbours(sets):
    """(B, L, W) bits of every single-flip neighbour of each row's set."""
    L = sets.shape[1]
    return SO.pack(sets[:, None, :] ^ torch.eye(L, dtype=torch.bool, device=sets.device)[None])


def _close(a, b, rel=1e-12):
    return bool(((a - b).abs() <= rel * b.abs() + 1e-300).all())


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (100, 37, 81, 81, 0), (10, 33, 983, 10, 0),
                                           (3, 9, 130, 64, FMA), (64, 40, 12, 12, 0), (16, 60, 10, 30, 0)])
def test_same_E_as_the_oracle(S, B, L, Z, flags):
    """CUDA-core path, external noise, E = predict(S = 1) per slice: sets, size and flips equal the oracle's; log_prob
    and ess within 1e-12 relative."""
    from mpvae_b200.mpvae import predict_mode
    if L <= 12:
        fx, r = _weak(B, L, Z, seed=S + L)
    else:
        t, _ = _inputs(S, B, L, Z, False, seed=S + B + L)
        fx, r = t["fx_out"], t["r_sqrt_sigma"]
    noise = torch.randn(S, B, Z, generator=torch.Generator().manual_seed(L)).to(DEV)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        E = _slice_E(fx, r, noise, args)
        got = predict_mode(fx, r, args, noise=noise)
    sets, log_prob, ess, size, flips = (t.cpu() for t in MO.mode(E))
    print(f"\n[oracle] S={S} B={B} L={L}: flips on {int((flips > 0).sum())} rows, median ess {float(ess.median()):.2f}")
    assert torch.equal(got.sets.cpu(), sets)
    assert torch.equal(got.size.cpu().long(), size) and torch.equal(got.flips.cpu().long(), flips)
    assert _close(got.log_prob.cpu(), log_prob) and _close(got.ess.cpu(), ess)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 70, 983, 983, 0), (7, 5, 130, 64, TENSOR)])
def test_dense_regime_against_the_oracle(S, B, L, Z, flags):
    """tcgen05 product: the oracle's fp32 E is not the library's.  DESIGN §5's rule on lp_s: the library is at most twice
    as far from the fp64 contraction's lp_s as the oracle's fp32 path, d32 (the per-cell log differences summed over
    the labels), so within 3 d32 of the oracle's.  The sets agree on at least 90 % of the rows, and there log_prob is
    within 3 d32 of the oracle's."""
    from mpvae_b200.mpvae import predict_mode
    assert _dense(S, B, L, Z, flags)
    t, _ = _inputs(S, B, L, Z, False, seed=S + B + L)
    fx, r = t["fx_out"], t["r_sqrt_sigma"]
    noise = torch.randn(S, B, Z, generator=torch.Generator().manual_seed(L)).to(DEV)
    with torch.no_grad():
        got = predict_mode(fx, r, _args(S, L, Z, flags), noise=noise)
    E = SO.sample_E(fx, r, noise).cpu()
    x64 = torch.tensordot(noise.double(), r.double().T, dims=1) + fx.double()
    E64 = SO.probit64(x64).cpu()
    (p32, n32), (p64, n64) = MO.cell_logs(E), (torch.log(E64), torch.log1p(-E64))
    d32 = float(torch.maximum((p32 - p64).abs(), (n32 - n64).abs()).sum(2).max())
    want = MO.mode(E)
    same = (got.sets.cpu() == want[0]).all(1)
    print(f"\n[dense] sets equal on {int(same.sum())}/{B} rows, d32 {d32:.3g}")
    assert float(same.double().mean()) >= 0.9
    assert float((got.log_prob.cpu() - want[1])[same].abs().max()) <= 3 * d32


REGIMES = [(10, 16, 38, 38, 0), (10, 33, 983, 10, 0), (10, 70, 983, 983, 0), (10, 16, 38, 38, STABLE),
           (3, 9, 130, 64, FMA), (7, 5, 130, 64, TENSOR), (100, 12, 300, 128, SEPARATE), (40, 30, 12, 40, 0)]


@pytest.mark.parametrize("S,B,L,Z,flags", REGIMES)
def test_against_the_library_scorer(S, B, L, Z, flags):
    """(log_prob, ess) = score_sets(the set) bit for bit; no single-flip neighbour scores higher beyond rounding; and
    log_prob >= the score of 1[predict >= 0.5], of the empty set and of every sample's mode (sample_labels with U = 1/2,
    which is the sample's mode except in cells where E is exactly 1/2)."""
    from mpvae_b200.mpvae import predict, predict_mode, sample_labels, score_sets
    if L <= 12:
        fx, r = _weak(B, L, Z, seed=S)
    else:
        t, _ = _inputs(S, B, L, Z, False, seed=S + B + L)
        fx, r = t["fx_out"], t["r_sqrt_sigma"]
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        got = predict_mode(fx, r, args)
        sc = score_sets(fx, r, SO.pack(got.sets[:, None]), args)
        nb = score_sets(fx, r, _all_neighbours(got.sets), args)
        c0 = SO.pack((predict(fx, r, args) >= 0.5)[:, None])
        modes = sample_labels(fx, r, args, uniform=torch.full((S, B, L), 0.5, device=DEV))
        cand = score_sets(fx, r, torch.cat([c0, torch.zeros_like(c0), modes], 1), args)
    assert torch.equal(sc.log_prob[:, 0], got.log_prob) and torch.equal(sc.ess[:, 0], got.ess)
    lim = got.log_prob[:, None] + 1e-12 * got.log_prob.abs()[:, None]
    assert bool((nb.log_prob <= lim).all())
    assert bool((cand.log_prob <= lim).all())
    assert torch.equal(got.size, got.sets.sum(1).int())
    assert bool(((got.ess >= 1 - 1e-12) & (got.ess <= S * (1 + 1e-12))).all())


def test_exhaustive_search_at_ten_labels():
    """L = 10, S = 100: all 1024 sets scored with score_sets; the mode is their argmax on at least 95 % of the rows."""
    from mpvae_b200.mpvae import predict_mode, score_sets
    S, B, L, Z = 100, 256, 10, 10
    fx, r = _weak(B, L, Z, seed=10, spread=0.3, load=0.5)
    args = _args(S, L, Z)
    hs = MO.all_sets(L).to(DEV)
    with torch.no_grad():
        got = predict_mode(fx, r, args)
        allsc = score_sets(fx, r, SO.pack(hs)[None].expand(B, -1, -1).contiguous(), args)
    best = allsc.log_prob.max(1).values
    assert bool((got.log_prob <= best).all())
    share = float((got.log_prob == best).double().mean())
    print(f"\n[exhaustive] mode = argmax on {100 * share:.1f} % of {B} rows; flips on {int((got.flips > 0).sum())} rows")
    assert share >= 0.95


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (3, 33, 983, 10, 0), (5, 12, 130, 64, TENSOR),
                                           (10, 16, 38, 38, STABLE)])
def test_zero_r_is_the_product_mode(S, B, L, Z, flags):
    """R = 0: every sample is one product distribution: the set is 1[E > 1/2], log_prob = sum_l log max(E, 1 - E),
    ess = S, flips = 0."""
    from mpvae_b200.mpvae import predict, predict_mode
    g = torch.Generator().manual_seed(S + L)
    fx = (torch.randn(B, L, generator=g) * 2).to(DEV)
    r = torch.zeros(L, Z, dtype=torch.float64, device=DEV)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        got = predict_mode(fx, r, args)
        a1 = copy.copy(args)
        a1.n_test_sample = 1
        e = predict(fx, r, a1)
    assert torch.equal(got.sets, e > 0.5)
    assert bool((got.flips == 0).all()) and bool((got.ess == S).all())
    llp, lln = MO.cell_logs(e[None])
    want = torch.maximum(llp, lln)[0].sum(1).cpu()
    if not flags & STABLE:      # the oracle's 1 - E is the reference's
        assert _close(got.log_prob.cpu(), want)


def test_links_to_predict_conditional_and_the_loss():
    """score_sets of the true labels against predict_conditional with every label observed, and against -nll_loss_x of a
    one-row test-mode compute_loss.  Those round lp_s to fp32 before the log-mean-exp (an exponent error of 2^-24 |lp_s|
    on the samples that carry weight, whose lp_s lie within log S of the maximum), exponentiate and sum in fp32 terms and
    round the result to fp32: |log_evidence - log_prob| <= 2^-22 (|log_prob| + log S + 1)."""
    from mpvae_b200.mpvae import compute_loss, predict_conditional, score_sets
    S, B, L, Z = 100, 24, 81, 81
    t, noise = _inputs(S, B, L, Z, True, seed=3)
    args = _args(S, L, Z)
    y = t["y"] > 0.5
    with torch.no_grad():
        sc = score_sets(t["fx_out"], t["r_sqrt_sigma"], SO.pack(y[:, None]), args, noise=noise)
        cond = predict_conditional(t["fx_out"], t["r_sqrt_sigma"], y.to(torch.int8), args, noise=noise)
    lp = sc.log_prob[:, 0]
    tol = 2.0 ** -22 * (lp.abs() + math.log(S) + 1)
    assert bool(((cond.log_evidence.double() - lp).abs() <= tol).all())
    for b in (0, 7):
        a = copy.copy(args)
        with torch.no_grad():
            out = compute_loss(t["y"][b:b + 1], t["fe_out"][b:b + 1], t["fe_mu"][b:b + 1], t["fe_logvar"][b:b + 1],
                               t["fx_out"][b:b + 1], t["fx_mu"][b:b + 1], t["fx_logvar"][b:b + 1], t["r_sqrt_sigma"], a,
                               noise=noise[:, b:b + 1])
            one = score_sets(t["fx_out"][b:b + 1], t["r_sqrt_sigma"], SO.pack(y[b:b + 1, None]), a,
                             noise=noise[:, b:b + 1])
        assert _close(one.log_prob[0], sc.log_prob[b])
        assert abs(-float(out[2]) - float(lp[b])) <= float(tol[b])


def _planted_pairs(n, L, Z, seed):
    """Pairs of labels loading with opposite signs on one latent direction each: a row usually carries exactly one label
    of each pair, and every marginal is below 1/2.  Labels are drawn from the model itself."""
    g = torch.Generator().manual_seed(seed)
    r = torch.zeros(L, Z, dtype=torch.float64)
    for j in range(L // 2):
        r[2 * j, j % Z] = 3.0
        r[2 * j + 1, j % Z] = -3.0
    fx = -0.5 + 0.05 * torch.randn(n, L, generator=g, dtype=torch.float64)
    z = torch.randn(n, Z, generator=g, dtype=torch.float64)
    xlat = fx + z @ r.T + torch.randn(n, L, generator=g, dtype=torch.float64)
    return fx.float().to(DEV), r.to(DEV), (xlat > 0).to(DEV)


def test_planted_model_mode_beats_thresholding_on_exact_match():
    """~2 000 rows, L = 6 in three exclusive pairs: predict_mode's exact-match accuracy beats predict_exact >= 0.5 by more
    than 5 paired standard errors; predict_sets' accuracy is printed beside them."""
    from mpvae_b200.mpvae import predict_exact, predict_mode, predict_sets
    n, L, Z = 2000, 6, 3
    fx, r, y = _planted_pairs(n, L, Z, seed=5)
    args = _args(1000, L, Z)
    with torch.no_grad():
        res = predict_mode(fx, r, args)
        p = predict_exact(fx, r, args)
        fs = predict_sets(fx, r, args)
    assert bool((p < 0.5).all())
    acc_mode = (res.sets == y).all(1).double()
    acc_thr = ((p >= 0.5) == y).all(1).double()
    acc_sets = (fs.sets == y).all(1).double()
    dlt = acc_mode - acc_thr
    se = float(dlt.std() / np.sqrt(n))
    print(f"\n[planted] exact match: mode {float(acc_mode.mean()):.4f}  thr0.5 {float(acc_thr.mean()):.4f}  "
          f"F1 sets {float(acc_sets.mean()):.4f}  diff/SE {float(dlt.mean()) / se:.1f}  "
          f"model's expected {float(res.log_prob.exp().mean()):.4f}  median ess {float(res.ess.median()):.1f}")
    assert float(dlt.mean()) > 5 * se


def test_rows_alone_repeat_poison_empty_offsets_caps(monkeypatch):
    """A row alone gives its batch result; repeated and poisoned runs give the same bits; B = 0; one offset per call and
    predict's noise at a fixed offset; max_flips = 0 returns the best candidate and max_flips caps the flips; garbage in
    the padding bits changes no score."""
    from mpvae_b200 import mpvae
    S, B, L, Z = 64, 400, 12, 12
    fx, r = _weak(B, L, Z, seed=77, spread=0.2, load=0.4)
    args = _args(S, L, Z)
    with torch.no_grad():
        full = mpvae.predict_mode(fx, r, args)
        assert int(full.flips.max()) >= 1, "the inputs should need some flips"
        for lo, hi in ((0, 1), (17, 18), (5, 29)):
            a = copy.copy(args)
            a.dp_global_batch, a.dp_row0 = B, lo
            part = mpvae.predict_mode(fx[lo:hi], r, a)
            for u, v in zip(part, full):
                assert torch.equal(u, v[lo:hi])
        monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
        again = mpvae.predict_mode(fx, r, args)
        sc = mpvae.score_sets(fx, r, SO.pack(full.sets[:, None]), args)
        monkeypatch.delenv("MPVAE_POISON_WORKSPACE")
        for u, v in zip(again, full):
            assert torch.equal(u, v)
        assert torch.equal(sc.log_prob[:, 0], full.log_prob) and torch.equal(sc.ess[:, 0], full.ess)
        # B = 0
        e = mpvae.predict_mode(fx[:0], r, args)
        assert e.sets.shape == (0, L) and e.log_prob.dtype == torch.float64 and e.flips.dtype == torch.int32
        es = mpvae.score_sets(fx[:0], r, torch.zeros(0, 3, 1, dtype=torch.int32, device=DEV), args)
        assert es.log_prob.shape == (0, 3) and es.ess.dtype == torch.float64
        # max_flips = 0: the best candidate; max_flips = 1: at most one flip, taken where the unbounded search took one
        zero = mpvae.predict_mode(fx, r, args, max_flips=0)
        c0 = SO.pack((mpvae.predict(fx, r, args) >= 0.5)[:, None])
        modes = mpvae.sample_labels(fx, r, args, uniform=torch.full((S, B, L), 0.5, device=DEV))
        cand = mpvae.score_sets(fx, r, torch.cat([c0, torch.zeros_like(c0), modes], 1), args)
        assert bool((zero.flips == 0).all()) and torch.equal(zero.log_prob, cand.log_prob.max(1).values)
        one = mpvae.predict_mode(fx, r, args, max_flips=1)
        assert torch.equal(one.flips, torch.clamp(full.flips, max=1))
        assert bool((one.log_prob >= zero.log_prob).all())
        # padding bits
        bits = SO.pack(full.sets[:, None])
        dirty = bits | torch.tensor(-(1 << L), dtype=torch.int32, device=DEV)
        sd = mpvae.score_sets(fx, r, dirty, args)
        assert torch.equal(sd.log_prob, sc.log_prob) and torch.equal(sd.ess, sc.ess)
        # one offset per call, and with the offset fixed at 6, predict's noise
        a = copy.copy(args)
        del a.noise_offset
        mpvae.set_noise_seed(4242, 6)
        first = mpvae.predict_mode(fx, r, a)
        assert mpvae._state["offset"] == 7
        for u, v in zip(first, full):
            assert torch.equal(u, v)
        mpvae.score_sets(fx, r, bits, a)
        assert mpvae._state["offset"] == 8


@pytest.mark.parametrize("S,B,L,Z,flags,external", [
    (10, 16, 38, 38, 0, False), (10, 16, 38, 38, 0, True), (10, 33, 983, 10, 0, False), (10, 70, 983, 983, 0, False),
    (10, 70, 983, 983, SEPARATE, False)])
def test_launch_count(S, B, L, Z, flags, external):
    """score_sets: predict's product (the CUDA-core one where predict runs its one-launch small kernel) plus two;
    predict_mode: plus four."""
    from mpvae_b200 import _lib
    from mpvae_b200.mpvae import predict_conditional, predict_mode, score_sets
    t, noise = _inputs(S, B, L, Z, external, seed=5)
    args = _args(S, L, Z, flags)
    none = torch.full((B, L), -1, dtype=torch.int8, device=DEV)
    bits = torch.zeros(B, 2, (L + 31) // 32, dtype=torch.int32, device=DEV)
    with torch.no_grad():
        n0 = _lib.launch_count()
        predict_conditional(t["fx_out"], t["r_sqrt_sigma"], none, args, noise=noise)   # the product, then three passes
        n1 = _lib.launch_count()
        score_sets(t["fx_out"], t["r_sqrt_sigma"], bits, args, noise=noise)
        n2 = _lib.launch_count()
        predict_mode(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
        n3 = _lib.launch_count()
    torch.cuda.synchronize()
    product = n1 - n0 - 3
    assert n2 - n1 == product + 2 and n3 - n2 == product + 4, (n1 - n0, n2 - n1, n3 - n2)


def test_mode_of_a_trained_model():
    """The yeast-shaped setup of test_set_scoring_of_a_trained_model: infer.predict_mode equals the hand loop bit for
    bit; the exact-match accuracy of the mode and of thresholding are printed."""
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_mode, predict_proba
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
    got = predict_mode(vae, xv, args, batch_size=128)
    assert got.sets.shape == (n_valid, 14) and got.sets.dtype == torch.bool
    assert got.log_prob.dtype == torch.float64 and got.flips.dtype == torch.int32
    vae.eval()
    a_t = copy.copy(args)
    a_t.mode = "test"
    hand = []
    torch.manual_seed(11)
    with torch.no_grad():
        for lo in range(0, n_valid, 128):
            hi = min(lo + 128, n_valid)
            a_t.dp_global_batch, a_t.dp_row0, a_t.noise_offset = n_valid, lo, 0
            hand.append(mpvae.predict_mode(vae.feat_forward(xv[lo:hi])[0], vae.r_sqrt_sigma, a_t))
    for i, g in enumerate(got):
        assert torch.equal(torch.cat([h[i] for h in hand], 0), g)
    torch.manual_seed(11)
    prob, _ = predict_proba(vae, xv, None, args, batch_size=128)
    yb = yv > 0.5
    acc_mode = float((got.sets == yb).all(1).double().mean())
    acc_thr = float(((prob >= 0.5) == yb).all(1).double().mean())
    print(f"\n[yeast] exact match: mode {acc_mode:.4f}, thresholding {acc_thr:.4f}; "
          f"model's expected {float(got.log_prob.exp().mean()):.4f}; flips on {int((got.flips > 0).sum())} rows")
    vae.train()
