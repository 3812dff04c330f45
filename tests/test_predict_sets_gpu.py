"""GPU: set prediction (mpvae_probit_sample_labels: predict's nt product, then probit_sample_labels_kernel;
mpvae_f1_sets: f1_sets_kernel) against the fp64 oracle and a brute-force search, the R = 0 identities, the statistics of
the library's stream against the closed form, a planted model where the F1-optimal sets beat thresholding, the
invariants under batching, repetition and a poisoned workspace, launch counts, and infer.predict_sets."""
import copy

import numpy as np
import pytest
import torch

from tests import predict_sets_oracle as SO
from tests.test_predict_gpu import EQUALITY_CASES, _args, _inputs, _yeast_args, _yeast_data

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

STABLE, FMA, TENSOR, SEPARATE = 0x8, 0x4, 0x2, 0x20


def _decode(y, beta=1.0, max_size=None):
    """The library decoder on (B, S, L) bool samples."""
    from mpvae_b200.mpvae import f1_optimal_sets
    out = f1_optimal_sets(SO.pack(y.to(DEV)), y.shape[2], beta, max_size)
    torch.cuda.synchronize()
    return out


def _random_rows(B, S, L, seed):
    """(B, S, L) bool: random densities, row 0 empty, row 1 full, row 2 with every label in some sample, row 3 one
    sample of groups."""
    g = torch.Generator().manual_seed(seed)
    dens = torch.rand(B, 1, 1, generator=g) * 0.6
    y = torch.rand(B, S, L, generator=g) < dens
    if B > 3:
        y[0] = False
        y[1] = True
        y[2] = torch.rand(S, L, generator=g) < 0.5
        y[2, 0] = True
        y[3] = False
        y[3, :, : min(L, 3)] = torch.rand(S, 1, generator=g) < 0.7
    return y


@pytest.mark.parametrize("B,S,L", [(40, 1, 1), (40, 7, 5), (60, 64, 12), (33, 100, 70), (20, 13, 257), (8, 300, 33)])
@pytest.mark.parametrize("beta", [0.5, 1.0, 2.0])
def test_decoder_against_the_oracle(B, S, L, beta):
    """Identical sets and sizes, expected_f within 1e-12 relative, for max_size None, 0, 1 and 3; brute force at L <= 12."""
    y = _random_rows(B, S, L, seed=B + S + L)
    for ms in (None, 0, 1, 3):
        got = _decode(y, beta, ms)
        sets, ef, size = SO.gfm(y.to(DEV), beta, ms)
        assert torch.equal(got.size.long(), size), ms
        assert torch.equal(got.sets, sets), ms
        assert float(((got.expected_f - ef).abs() / ef.abs().clamp_min(1e-300)).max()) <= 1e-12, ms
        assert bool((got.expected_f[0] == 1.0) & (got.size[0] == 0))      # the empty row
        if L <= 12:
            for b in range(min(B, 12)):
                all_ef, _ = SO.brute_force(y[b].double(), beta, ms)
                assert abs(float(got.expected_f[b]) - float(all_ef.max())) <= 1e-12


def test_decoder_reaches_past_256_words():
    """L = 8300: ceil(L / 32) = 260 words, so U_b is compacted over two rounds of 256 words; sparse rows keep the
    oracle's k loop short."""
    B, S, L = 6, 20, 8300
    g = torch.Generator().manual_seed(8300)
    y = torch.rand(B, S, L, generator=g) < 0.002
    y[1, :, 8290:] = True                        # labels in the second round, the last word included
    for ms in (3, 25):
        got = _decode(y, 1.0, ms)
        sets, ef, size = SO.gfm(y.to(DEV), 1.0, ms)
        assert torch.equal(got.size.long(), size) and torch.equal(got.sets, sets), ms
        assert float(((got.expected_f - ef).abs() / ef).max()) <= 1e-12, ms


@pytest.mark.parametrize("L", [1, 5, 40, 70, 257])
def test_decoder_ignores_the_padding_bits(L):
    """Whatever the bits at and above L hold -- random garbage, or every bit set as torch.full(..., -1) leaves them --
    the result is the masked bits' result."""
    from mpvae_b200.mpvae import f1_optimal_sets
    B, S = 24, 9
    y = _random_rows(B, S, L, seed=L)
    clean = SO.pack(y.to(DEV))
    pad = L % 32
    if pad == 0:
        pytest.skip("no padding bits")
    g = torch.Generator().manual_seed(L + 1)
    junk = torch.randint(0, 2 ** 32, clean.shape[:2], generator=g, dtype=torch.int64).to(DEV)
    v = (clean[:, :, -1].long() & 0xFFFFFFFF) | (junk & (0xFFFFFFFF ^ ((1 << pad) - 1)))   # garbage above L only
    dirty = clean.clone()
    dirty[:, :, -1] = torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)
    assert not torch.equal(dirty, clean)
    want = f1_optimal_sets(clean, L)
    for bits in (dirty, torch.full_like(clean, -1)):
        got = f1_optimal_sets(bits, L)
        if bits is dirty:
            for u, v in zip(got, want):
                assert torch.equal(u, v)
        else:
            full = f1_optimal_sets(SO.pack(torch.ones(B, S, L, dtype=torch.bool, device=DEV)), L)
            for u, v in zip(got, full):
                assert torch.equal(u, v)
            assert bool(got.sets.all()) and bool((got.size == L).all())


def _zero_r_case(S, B, L, Z, flags, seed):
    g = torch.Generator().manual_seed(seed)
    fx = (torch.randn(B, L, generator=g) * 2).to(DEV)
    r = torch.zeros(L, Z, dtype=torch.float64, device=DEV)
    U = torch.rand(S, B, L, generator=g).clamp(1e-7, 1 - 1e-7).to(DEV)
    return fx, r, U, _args(S, L, Z, flags)


@pytest.mark.parametrize("S,B,L,Z,flags", [(10, 16, 38, 38, 0), (3, 33, 983, 10, 0), (4, 70, 256, 256, 0),
                                           (5, 12, 130, 64, TENSOR), (10, 16, 38, 38, STABLE), (3, 40, 300, 256, STABLE)])
def test_zero_r_bits_are_u_below_predict(S, B, L, Z, flags):
    """R = 0 makes nr exactly 0, so with the caller's U every sample s is U[s] < predict(S = 1), bit for bit, in the
    small, CUDA-core and dense regimes and under STABLE_CDF."""
    from mpvae_b200.mpvae import predict, sample_labels, unpack_label_samples
    fx, r, U, args = _zero_r_case(S, B, L, Z, flags, seed=S + L)
    with torch.no_grad():
        bits = sample_labels(fx, r, args, uniform=U)
        a1 = copy.copy(args)
        a1.n_test_sample = 1
        e = predict(fx, r, a1)
    y = unpack_label_samples(bits, L)
    assert bits.shape == (B, S, (L + 31) // 32)
    assert torch.equal(y, (U < e[None]).transpose(0, 1))
    if L % 32:
        assert int((bits[:, :, -1] >> (L % 32)).abs().sum()) == 0


def _dense(S, B, L, Z, flags):
    """Whether the library takes the tcgen05 product for this call (capi.cu use_tensor)."""
    if flags & FMA or Z < 8 or L < 8:
        return False
    return bool(flags & TENSOR) or (Z >= 128 and L >= 128 and S * B >= 128)


# the EQUALITY_CASES shapes and flags; the sampler is always fed external noise and U here, so the cases that differ
# only in `external` are one case
ORACLE_CASES = sorted({c[:5] for c in EQUALITY_CASES})


@pytest.mark.parametrize("S,B,L,Z,flags", ORACLE_CASES)
def test_sampler_against_the_oracle(S, B, L, Z, flags):
    """External noise and U: a bit differs from the oracle's only in a cell with |U - E_oracle| below the regime's E
    tolerance.  CUDA-core path: 1e-5.  Dense regime, DESIGN §5's rule: at least as close to the exact contraction as
    the reference's own fp32 path, with 2x slack -- twice the largest |E_fp32 - E_fp64| over the tensor, where E_fp64 is
    E of the fp64 contraction (the truth) and E_fp32 the oracle's fp32 path."""
    from mpvae_b200.mpvae import sample_labels, unpack_label_samples
    t, _ = _inputs(S, B, L, Z, False, seed=S + B + L)
    g = torch.Generator().manual_seed(L)
    noise = torch.randn(S, B, Z, generator=g).to(DEV)
    U = torch.rand(S, B, L, generator=g).clamp(1e-7, 1 - 1e-7).to(DEV)
    stable = bool(flags & STABLE)
    with torch.no_grad():
        y = unpack_label_samples(sample_labels(t["fx_out"], t["r_sqrt_sigma"], _args(S, L, Z, flags), noise=noise,
                                               uniform=U), L).transpose(0, 1)
        E = SO.sample_E(t["fx_out"], t["r_sqrt_sigma"], noise, stable).double()
        if _dense(S, B, L, Z, flags):
            x64 = torch.tensordot(noise.double(), t["r_sqrt_sigma"].double().T, dims=1) + t["fx_out"].double()
            E64 = SO.probit64(x64)
            tol = 2.0 * float((E - E64).abs().max())
            E = E64
        else:
            tol = 1e-5
    want = U.double() < E
    near = (U.double() - E).abs() < tol
    assert not bool((y != want)[~near].any()), (int((y != want).sum()), tol)


def test_library_stream_is_the_oracle_uniforms():
    """Library U, R = 0: every bit is the oracle's U < E for the Philox uniforms of tests/predict_sets_oracle.py."""
    from mpvae_b200.mpvae import sample_labels, unpack_label_samples
    S, B, L, Z = 6, 9, 70, 8
    fx, r, _, args = _zero_r_case(S, B, L, Z, 0, seed=1)
    with torch.no_grad():
        y = unpack_label_samples(sample_labels(fx, r, args), L).transpose(0, 1)
    U = SO.library_uniform(S, B, L, seed=4242, offset=6).to(DEV)
    E = SO.sample_E(fx, r, torch.zeros(S, B, Z, device=DEV))
    assert torch.equal(y, U < E.double())


def _se_check(freq, p, n, k=6.0):
    se = torch.sqrt(p * (1 - p) / n).clamp_min(1.0 / n)
    z = ((freq - p).abs() / se).max()
    assert float(z) < k, float(z)


@pytest.mark.parametrize("L,Z,flags", [(14, 14, 0), (38, 38, 0), (81, 81, STABLE)])
def test_library_stream_statistics(L, Z, flags):
    """S = 10 000: the per-cell frequency within 6 binomial standard errors of predict_exact, and pair co-occurrence of
    PairPredictor's."""
    from mpvae_b200.mpvae import PairPredictor, all_pairs, predict_exact, sample_labels, unpack_label_samples
    S, B = 10000, 6
    t, _ = _inputs(S, B, L, Z, False, seed=L)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        y = unpack_label_samples(sample_labels(t["fx_out"], t["r_sqrt_sigma"], args), L).double()
        p = predict_exact(t["fx_out"], t["r_sqrt_sigma"], args).double()
        pairs = all_pairs(L)[:200]
        pp = PairPredictor(t["r_sqrt_sigma"], pairs, args)(t["fx_out"]).double()
    _se_check(y.mean(1), p, S)
    co = (y[:, :, pairs[:, 0]] * y[:, :, pairs[:, 1]]).mean(1)
    _se_check(co, pp, S)


def test_uniforms_where_the_comparison_reads_them():
    """R = 0 and fx_out set so that E runs over a grid spanning (c, 1 - c): the share of set bits matches E at every
    grid point within 6 standard errors."""
    from mpvae_b200.mpvae import predict, sample_labels, unpack_label_samples
    from scipy.stats import norm
    S, B, L, Z = 10000, 4, 64, 8
    q = torch.tensor(np.concatenate([[1e-6, 1e-5, 1e-4, 1e-3], np.linspace(0.01, 0.99, 56), [0.999, 0.9999, 0.99999,
                                                                                              0.999999]]))
    fx = torch.tensor(norm.ppf(q.numpy()), dtype=torch.float32).repeat(B, 1).to(DEV)
    r = torch.zeros(L, Z, dtype=torch.float64, device=DEV)
    args = _args(S, L, Z)
    with torch.no_grad():
        y = unpack_label_samples(sample_labels(fx, r, args), L).double()
        a1 = copy.copy(args)
        a1.n_test_sample = 1
        e = predict(fx, r, a1).double()
    _se_check(y.mean(1), e, S)


def _planted(n, L, Z, seed):
    """Rows that usually carry one whole group of labels: R loads each group on its own latent direction, fx_out pulls
    every marginal below 0.5; the labels are drawn from the model itself."""
    g = torch.Generator().manual_seed(seed)
    groups = L // 5
    r = torch.zeros(L, Z, dtype=torch.float64)
    for j in range(groups):
        r[5 * j:5 * j + 5, j % Z] = 2.5
    z = torch.randn(n, Z, generator=g, dtype=torch.float64)
    fx = (-1.2 + 0.4 * torch.randn(n, L, generator=g, dtype=torch.float64))
    xlat = fx + z @ r.T + torch.randn(n, L, generator=g, dtype=torch.float64)
    return fx.float().to(DEV), r.to(DEV), (xlat > 0).to(DEV)


def test_planted_model_sets_beat_thresholding():
    """~2 000 rows, L = 30 in six correlated groups: the per-row F1 of predict_sets beats predict_exact thresholded at
    0.5 by more than 5 paired standard errors and is within 2 of the best of 27 global thresholds."""
    from mpvae_b200.mpvae import predict_exact, predict_sets
    n, L, Z = 2000, 30, 6
    fx, r, y = _planted(n, L, Z, seed=3)
    args = _args(1000, L, Z)
    with torch.no_grad():
        res = predict_sets(fx, r, args)
        p = predict_exact(fx, r, args)
    f_sets = SO.f_measure(res.sets, y)
    thr = [0.05 * i for i in range(1, 20)] + [0.01, 0.02, 0.03, 0.04, 0.96, 0.97, 0.98, 0.99]
    f_thr = {t: SO.f_measure(p >= t, y) for t in thr}
    d = f_sets - f_thr[0.5]
    se = float(d.std() / np.sqrt(n))
    t_best = max(thr, key=lambda t: float(f_thr[t].mean()))
    d_best = f_sets - f_thr[t_best]
    se_best = float(d_best.std() / np.sqrt(n))

    def eb_f1(h):   # the reference's ebF1: rows with an empty denominator dropped
        den = h.double().sum(1) + y.double().sum(1)
        keep = den > 0
        return float((2 * (h.double() * y.double()).sum(1)[keep] / den[keep]).mean())
    print(f"\n[planted] F1 sets {float(f_sets.mean()):.4f}  thr0.5 {float(f_thr[0.5].mean()):.4f}  "
          f"best thr {t_best:.2f} {float(f_thr[t_best].mean()):.4f}  diff/SE {float(d.mean()) / se:.1f}  "
          f"vs best {float(d_best.mean()) / se_best:.1f}  ebF1 sets {eb_f1(res.sets):.4f} thr0.5 {eb_f1(p >= 0.5):.4f}  "
          f"mean size {float(res.size.double().mean()):.2f}")
    assert float(d.mean()) > 5 * se
    assert float(d_best.mean()) > -2 * se_best


@pytest.mark.parametrize("L,Z,flags", [(300, 256, TENSOR), (983, 10, 0)])
def test_rows_alone_repeat_poison_empty_offsets(L, Z, flags, monkeypatch):
    """A row alone gives its bits in the batch; repeated and poisoned runs give the same bits; B = 0; one offset."""
    from mpvae_b200 import mpvae
    S, B = 10, 40
    t, _ = _inputs(S, B, L, Z, False, seed=9)
    args = _args(S, L, Z, flags)
    with torch.no_grad():
        full = mpvae.sample_labels(t["fx_out"], t["r_sqrt_sigma"], args)
        for lo, hi in ((0, 1), (17, 18), (5, 29)):
            a = copy.copy(args)
            a.dp_global_batch, a.dp_row0 = B, lo
            part = mpvae.sample_labels(t["fx_out"][lo:hi], t["r_sqrt_sigma"], a)
            assert torch.equal(part, full[lo:hi])
        sets = mpvae.predict_sets(t["fx_out"], t["r_sqrt_sigma"], args, max_size=20)
        monkeypatch.setenv("MPVAE_POISON_WORKSPACE", "1")
        assert torch.equal(mpvae.sample_labels(t["fx_out"], t["r_sqrt_sigma"], args), full)
        again = mpvae.predict_sets(t["fx_out"], t["r_sqrt_sigma"], args, max_size=20)
        monkeypatch.delenv("MPVAE_POISON_WORKSPACE")
        for u, v in zip(sets, again):
            assert torch.equal(u, v)
        assert mpvae.sample_labels(t["fx_out"][:0], t["r_sqrt_sigma"], args).shape == (0, S, (L + 31) // 32)
        empty = mpvae.predict_sets(t["fx_out"][:0], t["r_sqrt_sigma"], args)
        assert empty.sets.shape == (0, L) and empty.expected_f.shape == (0,) and empty.size.shape == (0,)
        e = mpvae.f1_optimal_sets(full[:0], L)
        assert e.sets.shape == (0, L)
        # a call without args.noise_offset consumes one offset, as predict does, and with the same offset uses its noise
        a = copy.copy(args)
        del a.noise_offset
        mpvae.set_noise_seed(4242, 6)
        first = mpvae.sample_labels(t["fx_out"], t["r_sqrt_sigma"], a)
        assert mpvae._state["offset"] == 7 and torch.equal(first, full)
        mpvae.predict(t["fx_out"], t["r_sqrt_sigma"], a)
        assert mpvae._state["offset"] == 8


@pytest.mark.parametrize("S,B,L,Z,flags,external", [
    (10, 16, 38, 38, 0, False), (10, 16, 38, 38, 0, True), (10, 33, 983, 10, 0, False), (10, 70, 983, 983, 0, False),
    (10, 70, 983, 983, 0, True), (10, 70, 983, 983, SEPARATE, False)])
def test_launch_count(S, B, L, Z, flags, external):
    """sample_labels: predict's product (the CUDA-core one where predict runs its one-launch small kernel) plus one;
    predict_sets: one more."""
    from mpvae_b200 import _lib
    from mpvae_b200.mpvae import predict_conditional, predict_sets, sample_labels
    t, noise = _inputs(S, B, L, Z, external, seed=5)
    args = _args(S, L, Z, flags)
    none = torch.full((B, L), -1, dtype=torch.int8, device=DEV)
    with torch.no_grad():
        n0 = _lib.launch_count()
        predict_conditional(t["fx_out"], t["r_sqrt_sigma"], none, args, noise=noise)   # the product, then three passes
        n1 = _lib.launch_count()
        sample_labels(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
        n2 = _lib.launch_count()
        predict_sets(t["fx_out"], t["r_sqrt_sigma"], args, noise=noise)
        n3 = _lib.launch_count()
    torch.cuda.synchronize()
    product = n1 - n0 - 3
    assert n2 - n1 == product + 1 and n3 - n2 == product + 2, (n1 - n0, n2 - n1, n3 - n2)


def test_set_scoring_of_a_trained_model():
    """The yeast-shaped setup of test_label_free_scoring_of_a_trained_model: infer.predict_sets equals the hand loop bit
    for bit."""
    from mpvae_b200 import mpvae
    from mpvae_b200.infer import predict_sets
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
    got = predict_sets(vae, xv, args, batch_size=128)
    assert got.sets.shape == (n_valid, 14) and got.sets.dtype == torch.bool
    vae.eval()
    a_t = copy.copy(args)
    a_t.mode = "test"
    hand = []
    torch.manual_seed(11)
    with torch.no_grad():
        for lo in range(0, n_valid, 128):
            hi = min(lo + 128, n_valid)
            a_t.dp_global_batch, a_t.dp_row0, a_t.noise_offset = n_valid, lo, 0
            hand.append(mpvae.predict_sets(vae.feat_forward(xv[lo:hi])[0], vae.r_sqrt_sigma, a_t))
    for i, g in enumerate(got):
        assert torch.equal(torch.cat([h[i] for h in hand], 0), g)
    f = SO.f_measure(got.sets, yv)
    print(f"\n[yeast] F1 of the sets {float(f.mean()):.4f}, mean size {float(got.size.double().mean()):.2f}")
    vae.train()
