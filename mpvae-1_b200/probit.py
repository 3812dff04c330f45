"""Host side of the probit-ELBO boundary: one `torch.autograd.Function` over the C-ABI.

Mirrors the autograd contract of the reference's `compute_loss` (mpvae.py:145-210, SURVEY.md 8b):
differentiable w.r.t. fe_out, fx_out, the four encoder outputs and R; cotangents may arrive on any of
the 8 outputs (total_loss from train.py:125, indiv_prob / indiv_prob_label from the fairness
regulariser, fairsoft_train.py:76-140).  PyTorch is used for device memory and the stream only.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib

_NAMES = ("input_label", "fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma", "noise")


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _check_tensors(names, tensors):
    dev = tensors[0].device
    for name, t in zip(names, tensors):
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(f"mpvae_b200: {name} is on {t.device}; the probit ELBO runs on CUDA only "
                               "(there is no CPU fallback)")
        if t.device != dev:
            raise RuntimeError(f"mpvae_b200: {name} is on {t.device}, expected {dev}")
        if t.dtype != torch.float32:
            raise TypeError(f"mpvae_b200: {name} must be float32, got {t.dtype}")


def _check_inputs(y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise, noise_spec):
    _check_tensors(_NAMES, (y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise))
    B, L = fe_out.shape
    D = fe_mu.shape[1]
    if noise is not None:
        S, Bn, Z = noise.shape
    else:
        S, Bn, Z = int(noise_spec[0]), B, r32.shape[1]
    if y.shape != (B, L) or fx_out.shape != (B, L):
        raise ValueError(f"label / logit shapes disagree: {tuple(y.shape)}, {tuple(fe_out.shape)}, {tuple(fx_out.shape)}")
    for name, t in (("fe_mu", fe_mu), ("fe_logvar", fe_logvar), ("fx_mu", fx_mu), ("fx_logvar", fx_logvar)):
        if t.shape != (B, D):
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {(B, D)}")
    if r32.shape != (L, Z):
        raise ValueError(f"r_sqrt_sigma has shape {tuple(r32.shape)}, expected {(L, Z)} (label_dim, z_dim)")
    if Bn != B:
        raise ValueError(f"noise has {Bn} rows, batch has {B}")
    return S, B, L, Z, D


def _set_noise_spec(p, spec, B):
    p.noise_offset_dev = None
    if spec is None:
        p.noise_seed = p.noise_offset = 0
        p.noise_b_global, p.noise_row0 = B, 0
        return
    _, seed, offset, b_global, row0 = spec[:5]
    if len(spec) > 5 and spec[5] is not None:     # device-side int64 counter added to the offset (CUDA graphs)
        counter = spec[5]
        if not (counter.is_cuda and counter.dtype == torch.int64 and counter.numel() == 1):
            raise TypeError("noise offset counter must be a 1-element int64 CUDA tensor")
        p.noise_offset_dev = counter.data_ptr()
    p.noise_seed = int(seed) & (2 ** 64 - 1)
    p.noise_offset = int(offset) & (2 ** 64 - 1)
    p.noise_b_global = int(b_global if b_global is not None else B)
    p.noise_row0 = int(row0)


class ProbitELBO(torch.autograd.Function):
    """(y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, R32, noise) -> the 8-tuple of mpvae.py:210.

    `noise` is either the (S, B, Z) tensor or None, in which case `noise_spec` = (S, seed, offset, B_global, row0)
    and the library draws the Philox normals itself, straight into the contraction engine's operand layout."""

    @staticmethod
    def forward(ctx, y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise, nll_coeff, c_coeff, flags,
                noise_spec=None, peer=None):
        lib = _lib.lib()
        y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32 = (
            t.contiguous() for t in (y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32))
        if noise is not None:
            noise = noise.contiguous()
        elif noise_spec is None:
            raise ValueError("ProbitELBO needs either a noise tensor or a noise_spec")
        S, B, L, Z, D = _check_inputs(y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise, noise_spec)
        dev = y.device
        want_bwd = any(ctx.needs_input_grad)
        with torch.cuda.device(dev):
            ws_bytes = int(lib.mpvae_workspace_bytes(S, B, L, Z, 1 if want_bwd else 0, flags))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            scalars = [torch.empty((), dtype=torch.float32, device=dev) for _ in range(6)]
            prob = torch.empty((B, L), dtype=torch.float32, device=dev)
            prob_label = torch.empty((B, L), dtype=torch.float32, device=dev)
            if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
                # test hook (compute-sanitizer --tool initcheck is closed on this pool): every scratch / output byte starts
                # as 0xFF (NaN as fp16 / fp32 / fp64, huge as a counter), so anything the kernels read before writing shows
                ws.fill_(255)
                for t in [prob, prob_label] + scalars:
                    t.fill_(float("nan"))
            p = _lib.ProbitParams()
            p.struct_bytes = C.sizeof(_lib.ProbitParams)
            p.flags = flags
            p.S, p.B, p.L, p.Z, p.D = S, B, L, Z, D
            p.nll_coeff, p.c_coeff = float(nll_coeff), float(c_coeff)
            p.y, p.fe_out, p.fx_out = _ptr(y), _ptr(fe_out), _ptr(fx_out)
            p.fe_mu, p.fe_logvar, p.fx_mu, p.fx_logvar = _ptr(fe_mu), _ptr(fe_logvar), _ptr(fx_mu), _ptr(fx_logvar)
            p.r, p.noise = _ptr(r32), _ptr(noise)
            _set_noise_spec(p, noise_spec, B)
            for i in range(6):
                p.scalars[i] = scalars[i].data_ptr()
            p.indiv_prob, p.indiv_prob_label = _ptr(prob), _ptr(prob_label)
            p.workspace, p.workspace_bytes = _ptr(ws), ws_bytes
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(lib.mpvae_probit_forward(C.byref(p), stream), "mpvae_probit_forward")
        if want_bwd:
            ctx.has_noise = noise is not None
            ctx.noise_spec = noise_spec
            # data-parallel g_R over peer memory (peer.py): the backward then returns the SUM over all ranks
            ctx.peer = peer if (peer is not None and peer.applies(S, B, L, Z, flags)) else None
            ctx.save_for_backward(y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, ws,
                                  *([noise] if noise is not None else []))
            ctx.dims = (S, B, L, Z, D)
            ctx.coeffs = (float(nll_coeff), float(c_coeff), int(flags))
            ctx.set_materialize_grads(False)
        return (*scalars, prob, prob_label)

    @staticmethod
    def backward(ctx, g_total, g_nll, g_nll_x, g_c, g_c_x, g_kl, g_prob, g_prob_label):
        lib = _lib.lib()
        y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, ws = ctx.saved_tensors[:9]
        noise = ctx.saved_tensors[9] if ctx.has_noise else None
        S, B, L, Z, D = ctx.dims
        nll_coeff, c_coeff, flags = ctx.coeffs
        dev = y.device
        need_r = ctx.needs_input_grad[7]

        def as_f32(g, shape=None):
            if g is None:
                return None
            g = g.to(device=dev, dtype=torch.float32)
            if shape is not None:
                g = g.expand(shape)
            return g.contiguous()

        g_scal = [as_f32(g) for g in (g_total, g_nll, g_nll_x, g_c, g_c_x, g_kl)]
        g_prob = as_f32(g_prob, (B, L))
        g_prob_label = as_f32(g_prob_label, (B, L))
        with torch.cuda.device(dev):
            g_fe_out = torch.empty_like(fe_out)
            g_fx_out = torch.empty_like(fx_out)
            g_mulv = [torch.empty_like(fe_mu) for _ in range(4)]
            if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
                for t in [g_fe_out, g_fx_out] + g_mulv:
                    t.fill_(float("nan"))
            peer = ctx.peer if need_r else None
            g_r = (torch.empty_like(r32) if peer is None else None) if need_r else None
            p = _lib.ProbitParams()
            p.struct_bytes = C.sizeof(_lib.ProbitParams)
            p.flags = flags
            p.S, p.B, p.L, p.Z, p.D = S, B, L, Z, D
            p.nll_coeff, p.c_coeff = nll_coeff, c_coeff
            p.y, p.fe_out, p.fx_out = _ptr(y), _ptr(fe_out), _ptr(fx_out)
            p.fe_mu, p.fe_logvar, p.fx_mu, p.fx_logvar = _ptr(fe_mu), _ptr(fe_logvar), _ptr(fx_mu), _ptr(fx_logvar)
            p.r, p.noise = _ptr(r32), _ptr(noise)
            _set_noise_spec(p, ctx.noise_spec, B)
            for i in range(6):
                p.g_scalars[i] = g_scal[i].data_ptr() if g_scal[i] is not None else None
            p.g_indiv_prob, p.g_indiv_prob_label = _ptr(g_prob), _ptr(g_prob_label)
            p.g_fe_out, p.g_fx_out = _ptr(g_fe_out), _ptr(g_fx_out)
            p.g_fe_mu, p.g_fe_logvar, p.g_fx_mu, p.g_fx_logvar = (_ptr(t) for t in g_mulv)
            if peer is not None:
                g_r = peer.fill(p)               # the ring's own buffer; every rank writes its slab of the sum into it
            p.g_r = _ptr(g_r)
            p.workspace, p.workspace_bytes = _ptr(ws), ws.numel()
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(lib.mpvae_probit_backward(C.byref(p), stream), "mpvae_probit_backward")
        #       y     fe_out    fe_mu      fe_logvar  fx_out    fx_mu      fx_logvar  r32  noise nll_c c_c flags spec
        return (None, g_fe_out, g_mulv[0], g_mulv[1], g_fx_out, g_mulv[2], g_mulv[3], g_r, None, None, None, None, None,
                None)


def probit_predict(fx_out, r32, S, *, noise=None, noise_spec=None, flags=0):
    """indiv_prob (B, L) = mean over S samples of clamp(Phi(fx_out + noise.R^T)) (mpvae.py:170,180,203): the prediction
    of the feature branch, without labels and without the loss.  Bit-equal to `ProbitELBO`'s indiv_prob on the same
    fx_out, R and noise.  `noise` / `noise_spec` as for `ProbitELBO`; inference only (no autograd graph)."""
    if noise is None and noise_spec is None:
        raise ValueError("probit_predict needs either a noise tensor or a noise_spec")
    if fx_out.dim() != 2:
        raise ValueError(f"fx_out must be (batch, label_dim), got {tuple(fx_out.shape)}")
    B, L = fx_out.shape
    S = int(S)
    if S < 1:
        raise ValueError(f"n_sample must be positive, got {S}")
    if r32.dim() != 2 or r32.shape[0] != L:
        raise ValueError(f"r_sqrt_sigma has shape {tuple(r32.shape)}, expected ({L}, z_dim)")
    Z = r32.shape[1]
    if noise is not None and noise.shape != (S, B, Z):
        raise ValueError(f"noise has shape {tuple(noise.shape)}, expected {(S, B, Z)} (n_sample, batch, z_dim)")
    _check_tensors(("fx_out", "r_sqrt_sigma", "noise"), (fx_out, r32, noise))
    lib = _lib.lib()
    fx_out, r32 = fx_out.contiguous(), r32.contiguous()
    if noise is not None:
        noise = noise.contiguous()
    dev = fx_out.device
    with torch.cuda.device(dev):
        ws_bytes = int(lib.mpvae_workspace_bytes(S, B, L, Z, 0, flags))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        prob = torch.empty((B, L), dtype=torch.float32, device=dev)
        if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
            # test hook: see ProbitELBO.forward
            ws.fill_(255)
            prob.fill_(float("nan"))
        p = _lib.ProbitParams()
        p.struct_bytes = C.sizeof(_lib.ProbitParams)
        p.flags = flags
        p.S, p.B, p.L, p.Z = S, B, L, Z
        p.fx_out, p.r, p.noise = _ptr(fx_out), _ptr(r32), _ptr(noise)
        _set_noise_spec(p, noise_spec, B)
        p.indiv_prob = _ptr(prob)
        p.workspace, p.workspace_bytes = _ptr(ws), ws_bytes
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.mpvae_probit_predict(C.byref(p), stream), "mpvae_probit_predict")
    return prob


# ---- closed-form prediction (csrc/predictive.cu): the S -> infinity limit of probit_predict ----

def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _check_f64(name, t, n, dev):
    if not t.is_cuda or t.device != dev:
        raise RuntimeError(f"mpvae_b200: {name} is on {t.device}, expected {dev} (CUDA only, no CPU fallback)")
    if t.dtype != torch.float64 or t.shape != (n,):
        raise TypeError(f"mpvae_b200: {name} must be a float64 ({n},) tensor, got {t.dtype} {tuple(t.shape)}")


def label_pairs(pairs, L, device=None):
    """(P, 2) label index pairs as the contiguous int32 tensor the kernels read, on `device`.  Indices are checked
    against [0, L) here on the host (ValueError); the kernels still return NaN for a pair outside it."""
    p = torch.as_tensor(pairs)
    if p.dim() != 2 or p.shape[1] != 2:
        raise ValueError(f"pairs must be (P, 2), got {tuple(p.shape)}")
    if p.dtype.is_floating_point or p.dtype.is_complex or p.dtype == torch.bool:
        raise TypeError(f"pairs must be integers, got {p.dtype}")
    if p.shape[0] > 0:
        lo, hi = int(p.min()), int(p.max())
        if lo < 0 or hi >= L:
            raise ValueError(f"pairs hold label indices in [{lo}, {hi}], outside [0, {L})")
    if p.shape[0] >= 2 ** 31:
        raise ValueError(f"{p.shape[0]} pairs do not fit int32")
    return p.to(device=device if device is not None else p.device, dtype=torch.int32).contiguous()


def predictive_scale(r32):
    """(L,) fp64 scale_l = 1 / sqrt(1 + sum_z R[l, z]^2) of the fp32 R (mpvae_predictive_scale)."""
    if r32.dim() != 2:
        raise ValueError(f"r_sqrt_sigma must be (label_dim, z_dim), got {tuple(r32.shape)}")
    _check_tensors(("r_sqrt_sigma",), (r32,))
    r32 = r32.contiguous()
    L, Z = r32.shape
    dev = r32.device
    scale = torch.empty(L, dtype=torch.float64, device=dev)
    if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
        scale.fill_(float("nan"))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().mpvae_predictive_scale(_ptr(r32), L, Z, _ptr(scale), _stream(dev)), "mpvae_predictive_scale")
    return scale


def predictive_rho(r32, scale, pairs):
    """(P,) fp64 correlation R_i . R_j * scale_i * scale_j of each (i, j) label pair of the probit predictive
    distribution (mpvae_predictive_rho): P * Z fp64 FMAs, so compute it once per R and pair list."""
    if r32.dim() != 2:
        raise ValueError(f"r_sqrt_sigma must be (label_dim, z_dim), got {tuple(r32.shape)}")
    L, Z = r32.shape
    pairs = label_pairs(pairs, L, r32.device)
    _check_tensors(("r_sqrt_sigma",), (r32,))
    dev = r32.device
    _check_f64("scale", scale, L, dev)
    r32 = r32.contiguous()
    P = pairs.shape[0]
    rho = torch.empty(P, dtype=torch.float64, device=dev)
    if P == 0:
        return rho
    if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
        rho.fill_(float("nan"))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().mpvae_predictive_rho(_ptr(r32), L, Z, _ptr(scale), _ptr(pairs), P, _ptr(rho), _stream(dev)),
                   "mpvae_predictive_rho")
    return rho


def predict_exact(fx_out, scale, flags=0):
    """(B, L) fp32 P(y = 1) = E(x'), x' = fp32(fx_out * scale) (mpvae_predict_exact): the S -> infinity limit of
    probit_predict's indiv_prob for the R that `scale` came from.  Only MPVAE_FLAG_STABLE_CDF in `flags` matters."""
    if fx_out.dim() != 2:
        raise ValueError(f"fx_out must be (batch, label_dim), got {tuple(fx_out.shape)}")
    B, L = fx_out.shape
    _check_tensors(("fx_out",), (fx_out,))
    dev = fx_out.device
    _check_f64("scale", scale, L, dev)
    fx_out = fx_out.contiguous()
    prob = torch.empty((B, L), dtype=torch.float32, device=dev)
    if B == 0:
        return prob
    if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
        prob.fill_(float("nan"))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().mpvae_predict_exact(_ptr(fx_out), B, L, _ptr(scale), int(flags), _ptr(prob), _stream(dev)),
                   "mpvae_predict_exact")
    return prob


def predict_exact_from_r(fx_out, r32, flags=0):
    """predictive_scale(r32) then predict_exact(fx_out, scale, flags) in one host pass: one check, one stream lookup and
    no device switch when fx_out's device is current.  Small batches are bound by the host's time per call, and this is
    what mpvae.predict_exact runs on every batch."""
    if fx_out.dim() != 2:
        raise ValueError(f"fx_out must be (batch, label_dim), got {tuple(fx_out.shape)}")
    B, L = fx_out.shape
    if r32.dim() != 2 or r32.shape[0] != L:
        raise ValueError(f"r_sqrt_sigma has shape {tuple(r32.shape)}, expected ({L}, z_dim)")
    _check_tensors(("fx_out", "r_sqrt_sigma"), (fx_out, r32))
    fx_out, r32 = fx_out.contiguous(), r32.contiguous()
    dev = fx_out.device
    scale = fx_out.new_empty(L, dtype=torch.float64)
    prob = fx_out.new_empty((B, L))
    if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
        scale.fill_(float("nan"))
        prob.fill_(float("nan"))
    lib = _lib.lib()

    def launch():
        # the raw handle of the current stream, without building a torch.cuda.Stream object on every batch
        stream = C.c_void_p(torch._C._cuda_getCurrentRawStream(dev.index))
        _lib.check(lib.mpvae_predictive_scale(_ptr(r32), L, r32.shape[1], _ptr(scale), stream), "mpvae_predictive_scale")
        if B:
            _lib.check(lib.mpvae_predict_exact(_ptr(fx_out), B, L, _ptr(scale), int(flags), _ptr(prob), stream),
                       "mpvae_predict_exact")

    if dev.index == torch.cuda.current_device():
        launch()
    else:
        with torch.cuda.device(dev):
            launch()
    return prob


def predict_pairs(fx_out, scale, pairs, rho, flags=0):
    """(B, P) fp32 P(y_i = 1, y_j = 1) of each label pair (mpvae_predict_pairs), `rho` from predictive_rho for the same
    pairs.  A pair (i, i) returns predict_exact's P(y_i = 1) bit for bit under the same flags.  The range check of
    `pairs` reads them on the host (a device synchronisation when they live on the GPU)."""
    if fx_out.dim() != 2:
        raise ValueError(f"fx_out must be (batch, label_dim), got {tuple(fx_out.shape)}")
    B, L = fx_out.shape
    pairs = label_pairs(pairs, L, fx_out.device)
    P = pairs.shape[0]
    _check_tensors(("fx_out",), (fx_out,))
    dev = fx_out.device
    _check_f64("scale", scale, L, dev)
    _check_f64("rho", rho, P, dev)
    fx_out = fx_out.contiguous()
    out = torch.empty((B, P), dtype=torch.float32, device=dev)
    if B == 0 or P == 0:
        return out
    if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
        out.fill_(float("nan"))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().mpvae_predict_pairs(_ptr(fx_out), B, L, _ptr(scale), _ptr(pairs), _ptr(rho), P, int(flags),
                                                  _ptr(out), _stream(dev)), "mpvae_predict_pairs")
    return out


def philox_normal(S, B, Z, *, seed, offset=0, device="cuda", global_batch=None, row0=0):
    """Standard-normal (S, B, Z) noise from the library's counter-based generator (mpvae.py:162 stand-in).
    Rows [row0, row0+B) of a `global_batch`-row draw: independent of how the batch is sharded."""
    lib = _lib.lib()
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("mpvae_b200.philox_normal runs on CUDA only")
    out = torch.empty((S, B, Z), dtype=torch.float32, device=dev)
    if out.numel() == 0:
        return out
    with torch.cuda.device(dev):
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.mpvae_philox_normal(_ptr(out), S, B, Z, int(global_batch if global_batch is not None else B),
                                           int(row0), C.c_uint64(seed & (2 ** 64 - 1)), C.c_uint64(offset), stream),
                   "mpvae_philox_normal")
    return out


def contract_nt(a, b, engine=0, ws=None, pitched=False):
    """C[M,N] = A[M,K] . B[N,K]^T through the library (the product of mpvae.py:168).  `ws` (a uint8 tensor from a
    previous call, see `contract_workspace`) lets engine 3 reuse the operand planes engine 2 prepared.  `pitched`
    stores C with rows padded to 16 bytes, as the loss kernels keep it, and returns the (M, N) view."""
    lib = _lib.lib()
    a, b = a.contiguous(), b.contiguous()
    M, K = a.shape
    N = b.shape[0]
    assert b.shape[1] == K and a.is_cuda and b.is_cuda and a.dtype == b.dtype == torch.float32
    ldc = (N + 3) & ~3 if pitched else N
    out = torch.empty((M, ldc), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        nbytes = int(lib.mpvae_contract_workspace_bytes(M, N, K, engine))
        if ws is None:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=a.device)
        stream = C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)
        _lib.check(lib.mpvae_contract_nt_pitched(_ptr(a), _ptr(b), _ptr(out), M, N, K, ldc, engine, _ptr(ws), nbytes, stream),
                   "mpvae_contract_nt_pitched")
    return out[:, :N] if pitched else out


def contract_workspace(M, N, K, device, engine=2):
    """Scratch for contract_nt / contract_tn that can be handed back in to reuse the prepared operand planes."""
    nbytes = int(_lib.lib().mpvae_contract_workspace_bytes(M, N, K, engine))
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def contract_tn(a, b, engine=0):
    """C[N1,N2] = A[M,N1]^T . B[M,N2] through the library (g_R = gx^T . noise)."""
    lib = _lib.lib()
    a, b = a.contiguous(), b.contiguous()
    M, N1 = a.shape
    N2 = b.shape[1]
    assert b.shape[0] == M and a.is_cuda and b.is_cuda and a.dtype == b.dtype == torch.float32
    out = torch.empty((N1, N2), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        nbytes = int(lib.mpvae_contract_workspace_bytes(M, N1, N2, engine))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=a.device)
        stream = C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)
        _lib.check(lib.mpvae_contract_tn(_ptr(a), _ptr(b), _ptr(out), M, N1, N2, engine, _ptr(ws), nbytes, stream),
                   "mpvae_contract_tn")
    return out
