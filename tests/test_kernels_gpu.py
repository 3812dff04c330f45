"""GPU tests of the individual kernels behind the C-ABI: Philox noise, the contraction engines, and
size-independent properties of the full path at BASELINE.json's large shapes."""
import os

import numpy as np
import pytest
import torch

from oracle import probit_elbo_oracle as orc
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ----------------------------------------------------------------------------- Philox noise
def philox4x32_10_numpy(counter, offset, seed):
    """Reference Philox4x32-10 (Salmon et al. 2011) in numpy uint64 arithmetic, vectorised over counters."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    mask = np.uint64(0xFFFFFFFF)
    c = [(counter & mask), (counter >> np.uint64(32)) & mask,
         np.full_like(counter, offset & 0xFFFFFFFF), np.full_like(counter, (offset >> 32) & 0xFFFFFFFF)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(W0)) & mask
        k1 = (k1 + np.uint64(W1)) & mask
    return c


def philox_normals_numpy(n, seed, offset):
    ctr = np.arange((n + 3) // 4, dtype=np.uint64)
    r = philox4x32_10_numpy(ctr, offset, seed)
    def bm(a, b):
        u1 = ((a >> np.uint64(9)).astype(np.float64) + 0.5) / 8388608.0
        u2 = ((b >> np.uint64(9)).astype(np.float64) + 0.5) / 8388608.0
        rad = np.sqrt(-2.0 * np.log(u1))
        return rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)
    n0, n1 = bm(r[0], r[1])
    n2, n3 = bm(r[2], r[3])
    return np.stack([n0, n1, n2, n3], axis=1).reshape(-1)[:n]


def test_philox_matches_numpy_reference():
    from mpvae_b200.probit import philox_normal
    S, B, Z = 3, 7, 13
    got = philox_normal(S, B, Z, seed=1234567890123, offset=5, device=DEV).cpu().numpy()
    want = philox_normals_numpy(S * B * Z, 1234567890123, 5).reshape(S, B, Z)
    # the library's noise is defined on the fp16 grid (philox.cuh): Box-Muller on the SFU, then round-to-nearest fp16
    assert np.array_equal(got, got.astype(np.float16).astype(np.float32))
    want16 = want.astype(np.float16).astype(np.float32)
    # the special-function unit (lg2/sqrt/sin/cos.approx, ~1e-6) vs numpy can move a value across an fp16 rounding
    # boundary: rare, and then by one step
    assert (got != want16).mean() <= 0.02
    np.testing.assert_allclose(got, want, rtol=2.0 ** -11, atol=2e-5)


def test_philox_is_shard_invariant_and_deterministic():
    """Rows [row0, row0+B) of a global draw equal the same rows drawn on one device (SURVEY 8e)."""
    from mpvae_b200.probit import philox_normal
    S, Bg, Z = 10, 64, 38
    full = philox_normal(S, Bg, Z, seed=99, offset=3, device=DEV)
    again = philox_normal(S, Bg, Z, seed=99, offset=3, device=DEV)
    assert torch.equal(full, again)
    for row0, B in ((0, 16), (16, 16), (40, 24), (63, 1)):
        part = philox_normal(S, B, Z, seed=99, offset=3, device=DEV, global_batch=Bg, row0=row0)
        assert torch.equal(part, full[:, row0:row0 + B, :]), (row0, B)
    other = philox_normal(S, Bg, Z, seed=99, offset=4, device=DEV)
    assert not torch.equal(full, other)


def test_philox_moments():
    from mpvae_b200.probit import philox_normal
    x = philox_normal(10, 1024, 1001, seed=7, device=DEV).double()
    n = x.numel()
    assert abs(x.mean().item()) < 5 / np.sqrt(n)
    assert abs(x.var().item() - 1.0) < 5 * np.sqrt(2.0 / n)
    assert abs((x ** 3).mean().item()) < 5 * np.sqrt(15.0 / n)
    assert abs((x ** 4).mean().item() - 3.0) < 5 * np.sqrt(96.0 / n)
    assert x.abs().max().item() < 6.0
    # consecutive elements are uncorrelated
    flat = x.flatten()
    assert abs((flat[:-1] * flat[1:]).mean().item()) < 5 / np.sqrt(n)


def test_philox_noise_fed_to_oracle():
    """Philox mode is validated by dumping its noise and giving the same tensor to the oracle (SURVEY 7-6)."""
    from mpvae_b200 import synth
    from mpvae_b200.mpvae import compute_loss
    from mpvae_b200.probit import philox_normal
    L, Z, B, S = 38, 38, 64, 10
    inp = synth.loss_inputs(L, Z, B, S, seed=21, with_noise=False)
    args = orc.make_args(L, Z, n_train_sample=S, noise_seed=4242, noise_offset=17)
    t = {k: torch.from_numpy(v).to(DEV).requires_grad_(k != "y") for k, v in inp.items()}
    out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                       t["r_sqrt_sigma"], args)
    out[0].backward()
    noise = philox_normal(S, B, Z, seed=4242, offset=17, device=DEV)
    # same-device oracle (the reference's torch ops on cuda): strict bar, see test_parity_gpu.py
    ref, ref_g = orc.probit_elbo_with_grads({k: torch.from_numpy(v).to(DEV) for k, v in inp.items()}, noise, 0.5, 10.0)
    for i, k in enumerate(H.SCALAR_KEYS):
        assert H.rel_err(out[i].item(), getattr(ref, k).item()) <= 1e-5, k
    for k in H.GRAD_KEYS:
        assert H.rel_err(t[k].grad.cpu().numpy(), ref_g[k].cpu().numpy()) <= 1e-5, k


def test_log_normal_bits():
    """csrc/probit_math.cuh::log_normal (libdevice's logf main path without the denormal / inf / zero blocks) must equal
    logf BIT FOR BIT on the domain the loss evaluates it on: every fp32 value of [4.7e-7, 1] is checked (115 M of them)."""
    import ctypes as C
    from mpvae_b200 import _lib
    lo = np.array([4.7e-7], dtype=np.float32).view(np.int32)[0]
    hi = np.array([1.0], dtype=np.float32).view(np.int32)[0]
    bits = torch.arange(int(lo), int(hi) + 1, dtype=torch.int32, device=DEV)
    x = bits.view(torch.float32)
    out, ref = torch.empty_like(x), torch.empty_like(x)
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    _lib.check(_lib.lib().mpvae_test_log_normal(C.c_void_p(x.data_ptr()), C.c_void_p(out.data_ptr()), C.c_void_p(ref.data_ptr()),
                                                x.numel(), stream), "mpvae_test_log_normal")
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), ref.view(torch.int32)), int((out.view(torch.int32) != ref.view(torch.int32)).sum())
    assert torch.allclose(ref.double(), torch.log(x.double()), rtol=3e-7, atol=1e-7)      # and logf itself is logf


# ----------------------------------------------------------------------------- contraction engines
@pytest.mark.parametrize("M,N,K", [(1280, 38, 38), (1280, 14, 14), (12800, 81, 81), (333, 130, 5), (1280, 983, 10),
                                   (1280, 983, 983), (257, 129, 127), (64, 3993, 10)])
def test_contract_nt_fma(M, N, K):
    from mpvae_b200.probit import contract_nt
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g) * 0.1
    got = contract_nt(a.to(DEV), b.to(DEV), engine=1).cpu()
    want = (a.double() @ b.double().T)
    assert H.rel_err(got.numpy(), want.numpy()) <= 2e-6


@pytest.mark.parametrize("M,N1,N2", [(1280, 38, 38), (1280, 14, 14), (333, 130, 5), (10240, 983, 10),
                                     (1280, 983, 983), (257, 129, 127), (10240, 3993, 10)])
def test_contract_tn_fma(M, N1, N2):
    from mpvae_b200.probit import contract_tn
    g = torch.Generator(device="cpu").manual_seed(M * 3 + N1)
    a = torch.randn(M, N1, generator=g) * 0.01
    b = torch.randn(M, N2, generator=g)
    got = contract_tn(a.to(DEV), b.to(DEV), engine=1)
    again = contract_tn(a.to(DEV), b.to(DEV), engine=1)
    assert torch.equal(got, again)          # split-K partials are reduced in a fixed order
    want = (a.double().T @ b.double())
    assert H.rel_err(got.cpu().numpy(), want.numpy()) <= 5e-6


# ----------------------------------------------------------------------------- full-size properties
def _run(inp, noise, args, scale=None, rows=None):
    """`noise` None = the library's own Philox draw (args carries seed / offset); a row slice then draws the rows of the
    GLOBAL batch it covers (dp_global_batch / dp_row0), exactly as a data-parallel rank would."""
    import copy
    from mpvae_b200.mpvae import compute_loss
    sel = (lambda v: v) if rows is None else (lambda v: v[rows])
    t = {k: (torch.from_numpy(sel(v)) if k != "r_sqrt_sigma" else torch.from_numpy(v)).to(DEV).requires_grad_(k != "y")
         for k, v in inp.items()}
    kw = {}
    if noise is not None:
        kw["noise"] = torch.from_numpy(noise if rows is None else noise[:, rows]).to(DEV)
    else:
        args = copy.copy(args)
        args.dp_global_batch = inp["y"].shape[0]
        args.dp_row0 = 0 if rows is None else rows.start
    out = compute_loss(t["y"], t["fe_out"], t["fe_mu"], t["fe_logvar"], t["fx_out"], t["fx_mu"], t["fx_logvar"],
                       t["r_sqrt_sigma"], args, **kw)
    (out[0] * (1.0 if scale is None else scale)).backward()
    return out, {k: t[k].grad for k in H.GRAD_KEYS}


@pytest.mark.parametrize("name,L,Z,B,library_noise", [("eurlex_z10", 3993, 10, 1024, False),
                                                      ("delicious", 983, 983, 128, False),
                                                      ("delicious_philox", 983, 983, 128, True),
                                                      ("eurlex_philox", 3993, 3993, 1024, True)])
def test_full_size_properties(name, L, Z, B, library_noise):
    """BASELINE.json full sizes, through properties that need no O(L^2) oracle:
      * every loss term is a mean over rows => halves recombine: term = (term_A + term_B) / 2, grads likewise
      * the backward is linear in the upstream cotangent
      * predictions are probabilities inside the clamp [eps/2, 1 - eps/2]
    `eurlex_philox` is bench.py's headline configuration exactly: S10 B1024 L3993 Z3993, library Philox noise, two-pass
    tensor product, then the row forward."""
    from mpvae_b200 import synth
    S = 10
    inp = synth.loss_inputs(L, Z, B, S, seed=3, label_rate=20.0 / L, with_noise=not library_noise)
    noise = None if library_noise else inp.pop("noise")
    args = orc.make_args(L, Z, n_train_sample=S, noise_seed=777, noise_offset=5)
    full, g_full = _run(inp, noise, args)
    half = B // 2
    a, g_a = _run(inp, noise, args, rows=slice(0, half))
    b, g_b = _run(inp, noise, args, rows=slice(half, B))
    for i in range(6):
        assert H.rel_err(full[i].item(), 0.5 * (a[i].item() + b[i].item())) <= 2e-6, i
    assert torch.equal(full[6][:half], a[6]) and torch.equal(full[6][half:], b[6])
    recombined = 0.5 * (g_a["r_sqrt_sigma"] + g_b["r_sqrt_sigma"])
    err_r = H.rel_err(g_full["r_sqrt_sigma"].cpu().numpy(), recombined.cpu().numpy())
    _tc_report(test="halves_recombine", name=name, err_g_r=err_r)
    assert err_r <= 1e-5
    assert H.rel_err(g_full["fe_out"][:half].cpu().numpy(), 0.5 * g_a["fe_out"].cpu().numpy()) <= 1e-6
    _, g_scaled = _run(inp, noise, args, scale=-2.5)
    for k in H.GRAD_KEYS:
        assert H.rel_err(g_scaled[k].cpu().numpy(), -2.5 * g_full[k].cpu().numpy()) <= 2e-6, k
    p = full[6]
    assert float(p.min()) >= 5e-7 * 0.99 and float(p.max()) <= 1.0 - 4.7e-7
    assert all(torch.isfinite(g).all() for g in g_full.values())


# ----------------------------------------------------------------------------- tcgen05 split-precision engine
def _tc_report(**kw):
    import json, os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "tc_report.jsonl")
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "a") as f:
            f.write(json.dumps(kw) + "\n")
    except OSError:
        pass


@pytest.mark.parametrize("M,N,K", [(128, 256, 32), (128, 256, 64), (256, 512, 256), (300, 500, 200), (1280, 983, 983),
                                   (10240, 983, 983), (640, 3993, 3993)])
def test_contract_nt_tensor(M, N, K):
    """The split-precision product on tcgen05 must agree with the exact product to fp32-SGEMM accuracy (parity needs ~1e-6)."""
    from mpvae_b200.probit import contract_nt
    g = torch.Generator(device="cpu").manual_seed(M + 3 * N + 7 * K)
    a = torch.randn(M, K, generator=g)
    b = (torch.rand(N, K, generator=g) - 0.5) * 0.06
    got = contract_nt(a.to(DEV), b.to(DEV), engine=2)
    want = a.to(DEV).double() @ b.to(DEV).double().T
    fma = contract_nt(a.to(DEV), b.to(DEV), engine=1)
    err = ((got.double() - want).abs().max() / want.abs().max()).item()
    err_fma = ((fma.double() - want).abs().max() / want.abs().max()).item()
    _tc_report(test="nt", M=M, N=N, K=K, err=err, err_fma=err_fma)
    assert err <= 3e-6, (err, err_fma)


@pytest.mark.parametrize("M,N,K", [(300, 500, 200), (1280, 983, 983), (10240, 983, 983), (640, 3993, 3993)])
def test_contract_with_fp16_grid_noise_operand(M, N, K):
    """Engines 4/5: the noise operand (A of nt, B of tn) lies on the fp16 grid like the library's Philox noise, so it
    is a single operand piece and the product takes two MMA passes.  Same accuracy bar as the three-pass product."""
    from mpvae_b200.probit import contract_nt, contract_tn
    g = torch.Generator(device="cpu").manual_seed(M + 5 * N + 11 * K)
    noise = torch.randn(M, K, generator=g).half().float().to(DEV)
    r = ((torch.rand(N, K, generator=g) - 0.5) * 0.06).to(DEV)
    got = contract_nt(noise, r, engine=4)
    want = noise.double() @ r.double().T
    err = ((got.double() - want).abs().max() / want.abs().max()).item()
    _tc_report(test="nt_exact", M=M, N=N, K=K, err=err)
    assert err <= 3e-6, err
    gx = (torch.randn(M, N, generator=g) * 1e-4).to(DEV)
    got_t = contract_tn(gx, noise, engine=4)
    want_t = gx.double().T @ noise.double()
    err_t = ((got_t.double() - want_t).abs().max() / want_t.abs().max()).item()
    _tc_report(test="tn_exact", M=M, N=N, K=K, err=err_t)
    assert err_t <= 3e-6, err_t
    assert torch.equal(got, contract_nt(noise, r, engine=4))          # reproducible, K-sliced tail wave included


@pytest.mark.parametrize("engine", [1, 2, 4])
def test_contract_nt_pitched_rows(engine):
    """The loss kernels keep noise.R^T in rows padded to 16 bytes; the padded and the dense store paths agree bit for bit."""
    from mpvae_b200.probit import contract_nt
    g = torch.Generator(device="cpu").manual_seed(77)
    a = torch.randn(1280, 983, generator=g).half().float().to(DEV)
    b = ((torch.rand(983, 983, generator=g) - 0.5) * 0.06).to(DEV)
    dense = contract_nt(a, b, engine=engine)
    padded = contract_nt(a, b, engine=engine, pitched=True)
    assert padded.stride(0) == 984 and torch.equal(dense, padded)


@pytest.mark.parametrize("M,N1,N2", [(32, 128, 256), (64, 128, 256), (256, 256, 512), (200, 300, 500), (1280, 983, 983),
                                     (10240, 983, 983), (1280, 3993, 3993)])
def test_contract_tn_tensor(M, N1, N2):
    from mpvae_b200.probit import contract_tn
    g = torch.Generator(device="cpu").manual_seed(M + 3 * N1 + 7 * N2)
    a = torch.randn(M, N1, generator=g) * 0.01
    b = torch.randn(M, N2, generator=g)
    got = contract_tn(a.to(DEV), b.to(DEV), engine=2)
    want = a.to(DEV).double().T @ b.to(DEV).double()
    err = ((got.double() - want).abs().max() / want.abs().max()).item()
    _tc_report(test="tn", M=M, N1=N1, N2=N2, err=err)
    assert err <= 3e-6, err
