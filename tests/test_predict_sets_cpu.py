"""CPU: the set-prediction oracle (tests/predict_sets_oracle.py) against a brute-force search over every label set, the
sampler oracle against predict's oracle, the library stream's uniforms, the bit packing, and the refusals of the C-ABI
and of the Python wrappers, which all happen before anything touches a device."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from tests import predict_oracle as PO
from tests import predict_sets_oracle as SO


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


def _bits(S, L, density, seed):
    g = torch.Generator().manual_seed(seed)
    if density == "empty":
        return torch.zeros(S, L)
    if density == "full":
        return torch.ones(S, L)
    if density == "mixed":     # whole groups of labels, as a correlated model draws them, and some empty samples
        y = torch.zeros(S, L)
        for i in range(S):
            u = float(torch.rand(1, generator=g))
            if u < 0.25:
                continue
            lo = int(torch.randint(0, L, (1,), generator=g))
            y[i, lo:lo + 3] = 1
        return y
    return (torch.rand(S, L, generator=g) < density).double()


@pytest.mark.parametrize("beta", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("S", [1, 7, 64])
@pytest.mark.parametrize("density", ["empty", 0.1, 0.4, 0.8, "full", "mixed"])
def test_gfm_is_the_brute_force_optimum(beta, S, density):
    """For L <= 12 and every max_size in {0, 1, 3, L}: the oracle's expected F is the best over all 2^L sets to 1e-12,
    its set scores that value, and where the optimum is unique by a margin the sets are equal."""
    for L in (1, 5, 12):
        y = _bits(S, L, density, seed=S * 31 + L + int(10 * beta))
        for max_size in (0, 1, 3, L):
            sets, ef, size = SO.gfm(y[None], beta, max_size)
            all_ef, hs = SO.brute_force(y, beta, max_size)
            best = float(all_ef.max())
            assert abs(float(ef[0]) - best) <= 1e-12, (L, max_size, float(ef[0]), best)
            assert int(size[0]) == int(sets[0].sum()) <= max_size
            mine = float(SO.f_measure(sets[0].double()[None], y.double(), beta).mean())
            assert abs(mine - best) <= 1e-12
            order = torch.sort(all_ef, descending=True).values
            if len(order) == 1 or float(order[0] - order[1]) > 1e-9:
                assert torch.equal(sets[0], hs[int(all_ef.argmax())])


def test_the_issue_example_three_groups():
    """Rows with exactly one of three groups of three labels (each with probability 0.3) or none: every marginal is 0.3,
    thresholding at 0.5 predicts nothing and scores 0.1; all nine labels score 0.9 * 6 / 12 = 0.45, the optimum."""
    y = torch.zeros(10, 9)
    for i, g in enumerate([0, 0, 0, 1, 1, 1, 2, 2, 2]):
        y[i, 3 * g:3 * g + 3] = 1
    sets, ef, size = SO.gfm(y[None])
    assert int(size[0]) == 9 and bool(sets[0].all())
    assert abs(float(ef[0]) - 0.45) < 1e-15
    assert abs(float(SO.f_measure(torch.zeros(9)[None], y).mean()) - 0.1) < 1e-15


@pytest.mark.parametrize("stable", [False, True])
def test_sampler_oracle_is_u_below_predicts_e(stable):
    """The oracle's per-sample E averages to predict_oracle.predict's bits, and its samples are U < E, cell for cell."""
    g = torch.Generator().manual_seed(3)
    S, B, L, Z = 9, 5, 37, 6
    fx = torch.randn(B, L, generator=g) * 2
    r = torch.randn(L, Z, generator=g, dtype=torch.float64) * 0.5
    noise = torch.randn(S, B, Z, generator=g)
    E = SO.sample_E(fx, r, noise, stable)
    assert torch.equal(torch.mean(E, dim=0), PO.predict(fx, r, noise, stable))
    U = torch.rand(S, B, L, generator=g)
    y = SO.sample(E, U)
    assert torch.equal(y, U.double() < E.double())
    assert (y.double().mean(0) - E.double().mean(0)).abs().max() < 1.0


def test_library_uniforms_are_inside_the_open_interval_and_shard_invariant():
    U = SO.library_uniform(40, 6, 37, seed=4242, offset=6)
    assert float(U.min()) > 0.0 and float(U.max()) < 1.0
    assert abs(float(U.mean()) - 0.5) < 0.02
    # rows [2, 5) of a 6-row batch are the same draws when computed alone (global-row keys)
    part = SO.library_uniform(40, 3, 37, seed=4242, offset=6, b_global=6, row0=2)
    assert torch.equal(part, U[:, 2:5])
    assert not torch.equal(SO.library_uniform(40, 6, 37, seed=4242, offset=7), U)


def test_pack_is_pack_labels_bit_order_and_unpack_inverts_it():
    from mpvae_b200.mpvae import unpack_label_samples
    from mpvae_b200.train import pack_labels
    g = torch.Generator().manual_seed(1)
    for L in (1, 31, 32, 33, 70):
        y = torch.rand(4, 3, L, generator=g) < 0.4
        bits = SO.pack(y)
        assert bits.shape == (4, 3, (L + 31) // 32) and bits.dtype == torch.int32
        assert torch.equal(unpack_label_samples(bits, L), y)
        as_bytes = bits.numpy().view(np.uint8).reshape(12, -1)[:, :(L + 7) // 8]
        assert np.array_equal(as_bytes, pack_labels(y.reshape(12, L).int()).numpy())


def test_header_declares_and_library_exports_set_prediction(lib):
    from mpvae_b200 import _lib
    from tests.test_lib_cpu import declared_symbols
    for s in ("mpvae_probit_sample_labels", "mpvae_f1_sets_workspace_bytes", "mpvae_f1_sets"):
        assert s in declared_symbols() and s in _lib.EXPORTS and hasattr(lib, s)


def test_entry_points_validate_arguments(lib):
    """Refused before anything touches the device (the non-NULL pointers below are never dereferenced)."""
    from mpvae_b200 import _lib
    err = lambda: lib.mpvae_last_error().decode()
    d = C.c_void_p(256)
    ws = int(lib.mpvae_f1_sets_workspace_bytes(4, 8, 40))
    assert ws >= 4 * 8 * 12 + 4 * 40 * 12 and lib.mpvae_f1_sets_workspace_bytes(0, 8, 40) == 256
    call = lambda B=4, S=8, L=40, beta=1.0, ms=40, ptr=d, nbytes=ws: lib.mpvae_f1_sets(
        ptr, B, S, L, beta, ms, d, d, d, d, nbytes, None)
    assert call(B=0) == 1 and "bad sizes" in err()
    assert call(S=0) == 1 and "bad sizes" in err()
    assert call(beta=0.0) == 1 and "beta" in err()
    assert call(beta=-1.0) == 1 and "beta" in err()
    assert call(beta=float("nan")) == 1 and "beta" in err()
    assert call(beta=float("inf")) == 1 and "beta" in err()
    assert call(beta=1e155) == 1 and "finite square" in err()      # finite, but beta^2 overflows
    assert call(ms=-1) == 1 and "max_size" in err()
    assert call(ptr=None) == 1 and "NULL" in err()
    assert call(nbytes=ws - 1) == 1 and "too small" in err()
    p = _lib.ProbitParams()
    p.struct_bytes = C.sizeof(_lib.ProbitParams)
    p.S, p.B, p.L, p.Z = 4, 3, 10, 5
    p.fx_out = p.r = p.workspace = d
    p.workspace_bytes = 1 << 30
    p.noise_b_global, p.noise_row0 = 3, 0
    assert lib.mpvae_probit_sample_labels(C.byref(p), None, None, None) == 1 and "bits" in err()
    p.noise = d
    p.noise_b_global, p.noise_row0 = 2, 0
    assert lib.mpvae_probit_sample_labels(C.byref(p), None, d, None) == 1 and "label draws" in err()
    p.B = 0
    assert lib.mpvae_probit_sample_labels(C.byref(p), None, d, None) == 1 and "bad sizes" in err()


def test_python_refusals():
    from mpvae_b200 import mpvae
    args = types.SimpleNamespace(n_test_sample=4, z_dim=3, noise_seed=1, noise_offset=0, mpvae_flags=0)
    fx, r = torch.zeros(2, 40), torch.zeros(40, 3, dtype=torch.float64)
    with pytest.raises(RuntimeError, match="needs CUDA tensors"):
        mpvae.sample_labels(fx, r, args)
    with pytest.raises(RuntimeError, match="needs CUDA tensors"):
        mpvae.predict_sets(fx, r, args)
    bits = torch.zeros(2, 4, 2, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="needs CUDA tensors"):
        mpvae.f1_optimal_sets(bits, 40)
    from mpvae_b200.probit import f1_sets
    with pytest.raises(ValueError, match="expected"):
        f1_sets(torch.zeros(2, 4, 3, dtype=torch.int32), 40)
    with pytest.raises(ValueError, match="expected"):
        f1_sets(torch.zeros(2, 4, dtype=torch.int32), 40)
    with pytest.raises(TypeError, match="int32"):
        f1_sets(torch.zeros(2, 4, 2, dtype=torch.int64), 40)
    for beta in (0.0, -1.0, float("inf"), float("nan"), 1e155):
        with pytest.raises(ValueError, match="beta"):
            f1_sets(bits, 40, beta=beta)
    with pytest.raises(ValueError, match="max_size"):
        f1_sets(bits, 40, max_size=-1)
    with pytest.raises(ValueError, match="beta"):
        mpvae.predict_sets(fx, r, args, beta=0.0)
    with pytest.raises(ValueError, match="max_size"):
        mpvae.predict_sets(fx, r, args, max_size=-2)
    # refused before the noise plan: no offset is consumed
    from mpvae_b200.mpvae import _state
    args.noise_offset = None
    before = _state["offset"]
    for beta in (float("inf"), 1e155):
        with pytest.raises(ValueError, match="beta"):
            mpvae.predict_sets(fx, r, args, beta=beta)
    assert _state["offset"] == before
