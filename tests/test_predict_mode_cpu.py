"""CPU: the mode-prediction oracle (tests/predict_mode_oracle.py) against a direct fp64 mixture, its candidates and an
exhaustive search over every label set, and the refusals of the C-ABI and of the Python wrappers, which all happen
before anything touches a device."""
import ctypes as C
import types

import pytest
import torch

from tests import predict_mode_oracle as MO


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


def _random_E(S, B, L, seed, spread=2.0, load=1.5, Z=2):
    """(S, B, L) fp32 per-sample probabilities of a correlated model: a shared logit per (row, label) plus per-sample
    noise along Z latent directions."""
    g = torch.Generator().manual_seed(seed)
    fx = torch.randn(B, L, generator=g) * spread
    r = torch.randn(L, Z, generator=g) * load
    x = fx[None] + torch.einsum("sbz,lz->sbl", torch.randn(S, B, Z, generator=g), r)
    return (0.5e-6 + (1 - 1e-6) * 0.5 * torch.special.erfc(-x.double() / 2 ** 0.5)).float()


def test_log_prob_is_the_direct_mixture():
    E = _random_E(13, 6, 9, seed=1)
    y = torch.rand(6, 5, 9, generator=torch.Generator().manual_seed(2)) < 0.4
    llp, lln = MO.cell_logs(E)
    got, ess = MO.score(llp, lln, y)
    want = MO.direct_log_prob(E, y)
    assert float(((got - want).abs() / want.abs()).max()) <= 1e-12
    assert bool(((ess >= 1 - 1e-12) & (ess <= 13 + 1e-9)).all())


# weak loadings on many directions make mixtures whose mode is neither a component's mode nor the thresholded marginals
@pytest.mark.parametrize("S,L,seed,spread,load,Z", [(1, 4, 0, 2.0, 1.5, 2), (7, 6, 1, 2.0, 1.5, 2), (100, 10, 3, 0.3, 1.5, 2),
                                                   (8, 10, 1, 0.3, 0.5, 10), (16, 10, 1, 0.0, 0.4, 10),
                                                   (32, 10, 1, 0.2, 0.3, 20)])
def test_mode_beats_every_candidate_and_is_a_local_maximum(S, L, seed, spread, load, Z):
    B = 400
    E = _random_E(S, B, L, seed, spread, load, Z)
    sets, log_prob, ess, size, flips = MO.mode(E)
    llp, lln = MO.cell_logs(E)
    cl, _ = MO.score(llp, lln, MO.candidates(E))
    assert bool((log_prob[:, None] >= cl - 1e-12 * cl.abs()).all())
    # every single-flip neighbour scores no higher, beyond rounding
    nb = sets[:, None, :] ^ torch.eye(L, dtype=torch.bool)[None]
    nl, _ = MO.score(llp, lln, nb)
    assert bool((nl <= log_prob[:, None] + 1e-12 * log_prob.abs()[:, None]).all())
    assert torch.equal(size, sets.sum(1))
    # a local search: the global optimum on most rows, not on every row
    lpb, hs = MO.exhaustive(E)
    exact = (lpb.max(1).values - log_prob).abs() <= 1e-12 * log_prob.abs()
    print(f"\n[oracle] S={S} L={L}: global optimum on {int(exact.sum())}/{B} rows, flips on {int((flips > 0).sum())}")
    assert int(exact.sum()) >= 0.95 * B


@pytest.mark.parametrize("L", [1, 5, 10])
def test_product_inputs_give_the_exhaustive_argmax(L):
    """All components equal: the mixture is one product distribution, whose mode the candidates already hold."""
    S, B = 8, 30
    E = _random_E(1, B, L, seed=L).expand(S, B, L).contiguous()
    sets, log_prob, ess, size, flips = MO.mode(E)
    lpb, hs = MO.exhaustive(E)
    best = lpb.argmax(1)
    assert torch.equal(sets, hs[best])
    assert bool((flips == 0).all())
    assert torch.allclose(ess, torch.full_like(ess, float(S)), rtol=0, atol=1e-9)
    assert torch.equal(sets, E[0] > 0.5)


def test_two_exclusive_labels_the_issue_example():
    """Two labels that exclude each other, each on in about 45 % of the components: thresholding predicts neither,
    whose probability is near 0.1, and the mode predicts one of them, near 0.45."""
    S = 20
    E = torch.full((S, 1, 2), 1e-4)
    E[: S * 9 // 20, 0, 0] = 1 - 1e-4
    E[S * 9 // 20: S * 18 // 20, 0, 1] = 1 - 1e-4
    sets, log_prob, *_ = MO.mode(E)
    assert not bool(MO.candidates(E)[0, 0].any())       # c0: every marginal is below 0.5
    assert int(sets.sum()) == 1 and abs(float(log_prob.exp()) - 0.45) < 1e-3


def test_header_declares_and_library_exports_mode_prediction(lib):
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for s in ("mpvae_mode_workspace_bytes", "mpvae_probit_score_sets", "mpvae_probit_predict_mode"):
        assert s in declared_symbols() and s in _lib.EXPORTS and hasattr(lib, s)


def test_entry_points_validate_arguments(lib):
    """Refused before anything touches the device (the non-NULL pointers below are never dereferenced)."""
    from mpvae_b200 import _lib
    err = lambda: lib.mpvae_last_error().decode()
    d = C.c_void_p(256)
    S, B, L, Z = 4, 3, 40, 5
    ws = int(lib.mpvae_mode_workspace_bytes(S, B, L))
    assert ws >= B * S * L * 8 and lib.mpvae_mode_workspace_bytes(0, B, L) == 256
    p = _lib.ProbitParams()
    p.struct_bytes = C.sizeof(_lib.ProbitParams)
    p.S, p.B, p.L, p.Z = S, B, L, Z
    p.fx_out = p.r = p.workspace = p.noise = d
    p.workspace_bytes = 1 << 30
    p.noise_b_global, p.noise_row0 = B, 0
    score = lambda bits=d, C_=2, out=d, ptr=d, n=ws: lib.mpvae_probit_score_sets(C.byref(p), bits, C_, out, d, ptr, n, None)
    mode = lambda mf=3, sets=d, ptr=d, n=ws: lib.mpvae_probit_predict_mode(C.byref(p), mf, sets, d, d, d, d, ptr, n, None)
    assert score(bits=None) == 1 and "NULL" in err()
    assert score(out=None) == 1 and "NULL" in err()
    assert score(C_=0) == 1 and "set count" in err()
    assert score(ptr=None) == 1 and "mode_ws" in err()
    assert score(n=ws - 1) == 1 and "too small" in err()
    assert score(ptr=C.c_void_p(256 + 8)) == 1 and "aligned" in err()
    assert mode(sets=None) == 1 and "NULL" in err()
    assert mode(mf=-1) == 1 and "max_flips" in err()
    assert mode(ptr=None) == 1 and "mode_ws" in err()
    assert mode(n=ws - 1) == 1 and "too small" in err()
    assert mode(ptr=C.c_void_p(256 + 8)) == 1 and "aligned" in err()
    p.B = 0
    assert score() == 1 and "bad sizes" in err()
    assert mode() == 1 and "bad sizes" in err()
    p.B, p.fx_out = B, None
    assert mode() == 1 and "NULL input" in err()


def test_python_refusals():
    from mpvae_b200 import mpvae
    from mpvae_b200.mpvae import _state
    args = types.SimpleNamespace(n_test_sample=4, z_dim=3, noise_seed=1, noise_offset=0, mpvae_flags=0)
    fx, r = torch.zeros(2, 40), torch.zeros(40, 3, dtype=torch.float64)
    bits = torch.zeros(2, 3, 2, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="needs CUDA tensors"):
        mpvae.predict_mode(fx, r, args)
    with pytest.raises(RuntimeError, match="needs CUDA tensors"):
        mpvae.score_sets(fx, r, bits, args)
    with pytest.raises(TypeError, match="int32"):
        mpvae.score_sets(fx, r, bits.long(), args)
    for bad in (torch.zeros(2, 3, 3, dtype=torch.int32), torch.zeros(2, 0, 2, dtype=torch.int32),
                torch.zeros(3, 3, 2, dtype=torch.int32), torch.zeros(2, 2, dtype=torch.int32)):
        with pytest.raises(ValueError, match="expected"):
            mpvae.score_sets(fx, r, bad, args)
    fr = torch.zeros(2, 40, requires_grad=True)
    with pytest.raises(RuntimeError, match="inference only"):
        mpvae.predict_mode(fr, r, args)
    with pytest.raises(RuntimeError, match="inference only"):
        mpvae.score_sets(fr, r, bits, args)
    # refused before the noise plan: no offset is consumed
    args.noise_offset = None
    before = _state["offset"]
    for mf in (-1, -100):
        with pytest.raises(ValueError, match="max_flips"):
            mpvae.predict_mode(fx, r, args, max_flips=mf)
    with pytest.raises(ValueError, match="expected"):
        mpvae.score_sets(fx, r, bits[:, :, :1], args)
    assert _state["offset"] == before
    from mpvae_b200.infer import predict_mode
    with pytest.raises(ValueError, match="max_flips"):
        predict_mode(None, fx, args, max_flips=-1)
