"""CPU-side checks of the boundary: the C-ABI library loads, exports every symbol include/*.h declares,
validates its arguments before touching CUDA, and the host mirror refuses to run without CUDA."""
import ctypes as C
import hashlib
import json
import os
import re

import numpy as np
import pytest
import torch

from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as entry
    entry.build()
    from mpvae_b200 import _lib
    return _lib.lib()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "mpvae_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mpvae_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    from mpvae_b200 import _lib
    syms = declared_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), s
    assert sorted(_lib.EXPORTS) == syms
    assert lib.mpvae_abi_version() == _lib.ABI_VERSION


def test_params_struct_matches_header(lib):
    """struct_bytes guard: a wrong size is rejected, the right size gets past it to the pointer checks."""
    from mpvae_b200 import _lib
    p = _lib.ProbitParams()
    p.struct_bytes = 8
    assert lib.mpvae_probit_forward(C.byref(p), None) == 1
    assert b"struct_bytes" in lib.mpvae_last_error()
    p.struct_bytes = C.sizeof(_lib.ProbitParams)
    p.S, p.B, p.L, p.Z, p.D = 10, 4, 14, 14, 50
    assert lib.mpvae_probit_forward(C.byref(p), None) == 1
    assert b"NULL input pointer" in lib.mpvae_last_error()
    p.B = 0
    assert lib.mpvae_probit_forward(C.byref(p), None) == 1
    assert b"bad sizes" in lib.mpvae_last_error()


def test_workspace_sizes(lib):
    S, B, L, Z = 10, 128, 38, 38
    fwd = lib.mpvae_workspace_bytes(S, B, L, Z, 0, 0)
    both = lib.mpvae_workspace_bytes(S, B, L, Z, 1, 0)
    cube = S * B * L * 4
    assert fwd >= cube and both >= fwd + cube
    assert both < 6 * cube + (2 << 20)        # nr, E_l, E_x, gxs, fp32 noise + the per-row g_R shares and statistics
    assert lib.mpvae_workspace_bytes(10, 1024, 3993, 3993, 1, 0) < 2 << 30
    assert lib.mpvae_workspace_bytes(0, 0, 0, 0, 1, 0) == 256


def test_no_cpu_fallback():
    from mpvae_b200.mpvae import compute_loss
    from oracle import probit_elbo_oracle as orc
    case = H.load_golden("yeast_b16")
    t = H.to_torch(case["inputs"])
    args = orc.make_args(case["L"], case["Z"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                     t["r_sqrt_sigma"], args)


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from mpvae_b200 import _lib
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(_lib.LibraryMissing):
        _lib.lib()


def test_vae_state_dict_layout():
    """Checkpoint interchange (SURVEY section 5): keys, shapes, dtypes; r_sqrt_sigma float64 (L, Z); the shared
    decoder trunk appears under both names."""
    from types import SimpleNamespace
    from mpvae_b200.mpvae import VAE
    args = SimpleNamespace(feature_dim=20, label_dim=7, latent_dim=5, z_dim=3, keep_prob=0.5, scale_coeff=1.0,
                           residue_sigma="")
    np.random.seed(4)
    vae = VAE(args)
    sd = vae.state_dict()
    assert sd["r_sqrt_sigma"].dtype == torch.float64 and sd["r_sqrt_sigma"].shape == (7, 3)
    for a, b in (("fd1", "fd_x1"), ("fd2", "fd_x2")):
        assert sd[a + ".weight"].data_ptr() == sd[b + ".weight"].data_ptr()
    assert vae.r_sqrt_sigma.requires_grad
    args.residue_sigma = "random"
    assert not VAE(args).r_sqrt_sigma.requires_grad
    args.residue_sigma = "zero"
    assert float(VAE(args).r_sqrt_sigma.abs().sum()) == 0.0
    # the reference class's seeded initialisation and forward, as tests/golden/make_golden_vae.py records them from the
    # reference's mpvae.py (the record's `source` says what produced it): the weights bit for bit (SHA-256), the forward
    # within a few fp32 ulps (CPU BLAS kernels round differently per instruction set: up to 5.5e-7 seen between AVX2 and
    # AVX-512).  Where the reference's copy is installed (oracle/make_ref.py), the reference class is held to the record
    # as well, so the record itself is checked against the reference.
    from oracle import make_ref
    with open(os.path.join(H.GOLDEN_DIR, "vae_init_forward.json")) as f:
        gold = json.load(f)
    ref = make_ref.load()
    x = torch.tensor(gold["x"], dtype=torch.float32)
    y = torch.tensor(gold["y"], dtype=torch.float32)
    args.residue_sigma = ""
    for cls in [VAE] + ([ref.VAE] if ref is not None else []):
        who = cls.__module__
        np.random.seed(4); torch.manual_seed(0)
        vae = cls(args)
        sd = vae.state_dict()
        assert list(sd.keys()) == [e["key"] for e in gold["state_dict"]], who
        for e in gold["state_dict"]:
            t = sd[e["key"]]
            assert str(t.dtype) == e["dtype"] and list(t.shape) == e["shape"], (who, e["key"])
            assert hashlib.sha256(t.detach().contiguous().numpy().tobytes()).hexdigest() == e["sha256"], (who, e["key"])
        torch.manual_seed(1); out = vae(y, x)
        assert len(out) == len(gold["forward"]), who
        for v, want in zip(out, gold["forward"]):
            want = np.array(want, dtype=np.float32)
            assert v.dtype == torch.float32 and v.shape == want.shape, who
            assert H.rel_err(v.detach().numpy(), want) <= 5e-6, who


def test_new_entry_points_validate_arguments(lib):
    """The optimizer / staged-engine / metrics / peer entry points reject bad arguments before touching the device."""
    assert lib.mpvae_grad_norm(None, 10, 1.0, 1.0, None, 1e-3, 0.9, 0.999, None, None, 0, None) == 1
    assert b"grad_norm" in lib.mpvae_last_error()
    assert lib.mpvae_adam_step(None, 0, None, None, None, None, 10, None, 0.9, 0.999, 1e-8, 0.0, None) == 1
    assert b"adam_step" in lib.mpvae_last_error()
    assert lib.mpvae_tc_split(None, 4, 64, None, None, None) == 1
    assert lib.mpvae_tc_gemm_nt(None, None, None, 1, 1, 1, 0, None, None, 0, None, 0, None) == 1
    assert lib.mpvae_tc_gemm_tn(None, None, None, 1, 1, 1, None, None, None, 0, None) == 1
    assert lib.mpvae_label_curves(None, None, 4, 4, 0.5, None, None) == 1
    assert b"label_curves" in lib.mpvae_last_error()
    assert lib.mpvae_peer_allreduce(None, None, None, 2, 0, 1, 16, None) == 1
    assert b"peer_allreduce" in lib.mpvae_last_error()
    assert lib.mpvae_tc_planes_bytes(1024, 3993) >= 2 * 1024 * 3993 * 2
    assert lib.mpvae_peer_flag_bytes() >= 17 * 4
    assert lib.mpvae_grad_norm_workspace() > 0


def test_host_wrappers_have_no_cpu_path():
    """The device-side replacements refuse CPU tensors; only the small-layer fallback of dense.linear (plain torch.nn,
    which the design keeps for the MLP) runs anywhere."""
    from mpvae_b200 import metrics
    from mpvae_b200.dense import linear, uses_tensor_engine
    from mpvae_b200.optim import FusedAdam
    p, y = torch.rand(4, 6), (torch.rand(4, 6) < 0.5).float()
    for fn in (metrics.batch_metrics, metrics.label_curves):
        with pytest.raises(RuntimeError, match="CUDA tensors only"):
            fn(p, y)
    w = torch.nn.Parameter(torch.randn(3, 3))
    w.grad = torch.randn(3, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        FusedAdam([w], lr=1e-3).step()
    layer, x = torch.nn.Linear(2048, 1024), torch.randn(256, 2048)
    assert not uses_tensor_engine(layer, x)
    assert torch.equal(linear(layer, x), layer(x))


def _integration_stub_source():
    """The ```python block of INTEGRATION.md section 2 (the binding a reference maintainer would paste into mpvae.py)."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    sec = text[text.index("## 2. Raw C-ABI"):]
    block = sec[sec.index("```python") + len("```python"):]
    block = block[:block.index("```")]
    from mpvae_b200 import _lib
    return block.replace('"libmpvae_b200.so"', repr(_lib.LIB_PATH))


def test_integration_stub_struct_matches_the_header(lib):
    """The stub's struct is a PREFIX of mpvae_probit_params (it stops before the peer_* fields): its size must be the
    MPVAE_PARAMS_BASE_BYTES the library accepts, field by field the same offsets as the maintained binding."""
    import ctypes as C
    from mpvae_b200 import _lib
    ns = {}
    exec(_integration_stub_source(), ns)           # defines P, _ProbitELBO, compute_loss against the built library
    P = ns["P"]
    assert C.sizeof(P) == _lib.PARAMS_BASE_BYTES
    full = {n: getattr(_lib.ProbitParams, n).offset for n, _ in _lib.ProbitParams._fields_}
    for name, _ in P._fields_:
        assert getattr(P, name).offset == full[name], name
    # the library takes exactly the two sizes: a params block of any other size is refused before anything is launched
    p = _lib.ProbitParams()
    p.struct_bytes = _lib.PARAMS_BASE_BYTES - 8
    assert lib.mpvae_probit_forward(C.byref(p), None) == 1
    assert b"struct_bytes" in lib.mpvae_last_error()
