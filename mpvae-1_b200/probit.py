"""Host side of the probit-ELBO boundary: one `torch.autograd.Function` over the C-ABI.

Mirrors the autograd contract of the reference's `compute_loss` (mpvae.py:145-210, SURVEY.md 8b):
differentiable w.r.t. fe_out, fx_out, the four encoder outputs and R; cotangents may arrive on any of
the 8 outputs (total_loss from train.py:125, indiv_prob / indiv_prob_label from the fairness
regulariser, fairsoft_train.py:76-140).  PyTorch is used for device memory and the stream only.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from collections import namedtuple

import torch

from . import _lib

_NAMES = ("input_label", "fe_out", "fe_mu", "fe_logvar", "fx_out", "fx_mu", "fx_logvar", "r_sqrt_sigma", "noise")


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(dev):
    # the raw handle of the current stream, without building a torch.cuda.Stream object on every call: small batches
    # are bound by the host's time per call
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(dev.index))


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


def _check_label_mask(label_mask, B, L, device):
    """The (B, L) label mask as contiguous uint8 (nonzero = observed), refused before any launch when it is not a bool or
    uint8 tensor of that shape on the batch's device."""
    if not isinstance(label_mask, torch.Tensor) or label_mask.dtype not in (torch.bool, torch.uint8):
        raise TypeError(f"label_mask must be a bool or uint8 tensor, got {getattr(label_mask, 'dtype', type(label_mask))}")
    if label_mask.shape != (B, L):
        raise ValueError(f"label_mask has shape {tuple(label_mask.shape)}, expected {(B, L)} (batch, label_dim)")
    if label_mask.device != device:
        raise ValueError(f"label_mask is on {label_mask.device}, expected {device}")
    return label_mask.contiguous().view(torch.uint8)


def _check_row_weight(row_weight, B, device):
    """The (B,) row weights as a contiguous fp32 tensor, refused before any launch when they are not a floating tensor of
    that shape on the batch's device, or when they require grad: the loss returns no gradient for them, and a silent
    zero would mislead.  The values are not checked (that would synchronise with the host)."""
    if not isinstance(row_weight, torch.Tensor) or not row_weight.is_floating_point():
        raise TypeError(f"row_weight must be a floating tensor, got {getattr(row_weight, 'dtype', type(row_weight))}")
    if row_weight.requires_grad:
        raise ValueError("row_weight requires grad, but the loss returns no gradient for it: pass row_weight.detach()")
    if row_weight.shape != (B,):
        raise ValueError(f"row_weight has shape {tuple(row_weight.shape)}, expected {(B,)} (batch,)")
    if row_weight.device != device:
        raise ValueError(f"row_weight is on {row_weight.device}, expected {device}")
    return row_weight.to(torch.float32).contiguous()


def _check_label_weight(pos_weight, neg_weight, L, device):
    """The (L,) weights of the y == 1 and y == 0 cells packed as one contiguous (2, L) fp32 tensor [neg_weight;
    pos_weight] (None for either = all ones), or None when both are None.  Refused before any launch, like row_weight,
    when a weight is not a floating tensor of that shape on the batch's device or requires grad.  The values are not
    checked (that would synchronise with the host)."""
    if pos_weight is None and neg_weight is None:
        return None
    for name, w in (("neg_weight", neg_weight), ("pos_weight", pos_weight)):
        if w is None:
            continue
        if not isinstance(w, torch.Tensor) or not w.is_floating_point():
            raise TypeError(f"{name} must be a floating tensor, got {getattr(w, 'dtype', type(w))}")
        if w.requires_grad:
            raise ValueError(f"{name} requires grad, but the loss returns no gradient for it: pass {name}.detach()")
        if w.shape != (L,):
            raise ValueError(f"{name} has shape {tuple(w.shape)}, expected {(L,)} (label_dim,)")
        if w.device != device:
            raise ValueError(f"{name} is on {w.device}, expected {device}")
    return torch.stack([torch.ones(L, dtype=torch.float32, device=device) if w is None else w.to(torch.float32)
                        for w in (neg_weight, pos_weight)]).contiguous()


def _check_observed(observed, shape, device):
    """Refuses an `observed` argument that is not an int8 tensor of `shape` (batch, label_dim) on `device`."""
    if not isinstance(observed, torch.Tensor) or observed.dtype != torch.int8:
        raise TypeError(f"observed must be an int8 tensor, got {getattr(observed, 'dtype', type(observed))}")
    if observed.shape != shape:
        raise ValueError(f"observed has shape {tuple(observed.shape)}, expected {tuple(shape)} (batch, label_dim)")
    if observed.device != device:
        raise ValueError(f"observed is on {observed.device}, expected {device}")


def _poison(*tensors):
    """Test hook (MPVAE_POISON_WORKSPACE=1): every scratch byte starts as 0xFF (NaN as fp16 / fp32 / fp64, huge as a
    counter) and every output as NaN, so anything the kernels read before writing, or leave unwritten, shows."""
    if os.environ.get("MPVAE_POISON_WORKSPACE") == "1":
        for t in tensors:
            t.fill_(255 if t.dtype == torch.uint8 else float("nan") if t.is_floating_point() else -1)


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
    and the library draws the Philox normals itself, straight into the contraction engine's operand layout.

    `label_mask` (B, L) bool / uint8 on the batch's device, or None: nonzero = the label is observed.  The
    log-likelihood and the ranking loss then run over the observed labels only (mpvae_probit_forward_masked); y is not
    read where the mask is 0.  None runs the unmasked entry points.

    `row_weight` (B,) floating on the batch's device, or None: the weight of each row's loss terms
    (mpvae_probit_forward_weighted, semantics in mpvae.compute_loss).  It receives no gradient.

    `label_weight` (2, L) fp32 on the batch's device (`_check_label_weight`: row 0 weighs the y == 0 cells, row 1 the
    y == 1 cells), or None: the label weights of the cell log-likelihoods (mpvae_probit_forward_label_weighted,
    semantics in mpvae.compute_loss).  It receives no gradient.

    `per_row` (reduction 'none'): the six loss outputs are (B,) tensors of every row's terms, and their cotangents are
    (B,) per row (mpvae_probit_forward_rows / _backward_rows, semantics in mpvae.compute_loss)."""

    @staticmethod
    def forward(ctx, y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise, nll_coeff, c_coeff, flags,
                noise_spec=None, peer=None, label_mask=None, row_weight=None, label_weight=None, per_row=False):
        lib = _lib.lib()
        y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32 = (
            t.contiguous() for t in (y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32))
        if noise is not None:
            noise = noise.contiguous()
        elif noise_spec is None:
            raise ValueError("ProbitELBO needs either a noise tensor or a noise_spec")
        S, B, L, Z, D = _check_inputs(y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, noise, noise_spec)
        dev = y.device
        if label_mask is not None:
            label_mask = _check_label_mask(label_mask, B, L, dev)
        if row_weight is not None:
            row_weight = _check_row_weight(row_weight, B, dev)
        if label_weight is not None and (not isinstance(label_weight, torch.Tensor) or label_weight.shape != (2, L) or
                                         label_weight.dtype != torch.float32 or label_weight.device != dev or
                                         label_weight.requires_grad):
            raise ValueError(f"label_weight must be a (2, {L}) fp32 tensor on {dev} without grad (_check_label_weight)")
        if label_weight is not None:
            label_weight = label_weight.contiguous()
        want_bwd = any(ctx.needs_input_grad)
        with torch.cuda.device(dev):
            ws_bytes = int(lib.mpvae_workspace_bytes(S, B, L, Z, 1 if want_bwd else 0, flags))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            scalars = [torch.empty((B,) if per_row else (), dtype=torch.float32, device=dev) for _ in range(6)]
            prob = torch.empty((B, L), dtype=torch.float32, device=dev)
            prob_label = torch.empty((B, L), dtype=torch.float32, device=dev)
            _poison(ws, prob, prob_label, *scalars)
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
            if per_row:
                _lib.check(lib.mpvae_probit_forward_rows(C.byref(p), _ptr(label_mask), _ptr(row_weight),
                                                         _ptr(label_weight), stream), "mpvae_probit_forward_rows")
            elif label_weight is not None:
                _lib.check(lib.mpvae_probit_forward_label_weighted(C.byref(p), _ptr(label_mask), _ptr(row_weight),
                                                                   _ptr(label_weight), stream),
                           "mpvae_probit_forward_label_weighted")
            elif row_weight is not None:
                _lib.check(lib.mpvae_probit_forward_weighted(C.byref(p), _ptr(label_mask), _ptr(row_weight), stream),
                           "mpvae_probit_forward_weighted")
            elif label_mask is None:
                _lib.check(lib.mpvae_probit_forward(C.byref(p), stream), "mpvae_probit_forward")
            else:
                _lib.check(lib.mpvae_probit_forward_masked(C.byref(p), _ptr(label_mask), stream),
                           "mpvae_probit_forward_masked")
        if want_bwd:
            ctx.has_noise = noise is not None
            ctx.noise_spec = noise_spec
            # data-parallel g_R over peer memory (peer.py): the backward then returns the SUM over all ranks
            ctx.peer = peer if (peer is not None and peer.applies(S, B, L, Z, flags)) else None
            ctx.has_mask = label_mask is not None
            ctx.has_weight = row_weight is not None
            ctx.has_label_weight = label_weight is not None
            ctx.save_for_backward(y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, ws,
                                  *([noise] if noise is not None else []),
                                  *([label_mask] if label_mask is not None else []),
                                  *([row_weight] if row_weight is not None else []),
                                  *([label_weight] if label_weight is not None else []))
            ctx.dims = (S, B, L, Z, D)
            ctx.coeffs = (float(nll_coeff), float(c_coeff), int(flags))
            ctx.per_row = bool(per_row)
            ctx.set_materialize_grads(False)
        return (*scalars, prob, prob_label)

    @staticmethod
    def backward(ctx, g_total, g_nll, g_nll_x, g_c, g_c_x, g_kl, g_prob, g_prob_label):
        lib = _lib.lib()
        y, fe_out, fe_mu, fe_logvar, fx_out, fx_mu, fx_logvar, r32, ws = ctx.saved_tensors[:9]
        rest = list(ctx.saved_tensors[9:])
        noise = rest.pop(0) if ctx.has_noise else None
        label_mask = rest.pop(0) if ctx.has_mask else None
        row_weight = rest.pop(0) if ctx.has_weight else None
        label_weight = rest.pop(0) if ctx.has_label_weight else None
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

        g_scal = [as_f32(g, (B,) if ctx.per_row else None) for g in (g_total, g_nll, g_nll_x, g_c, g_c_x, g_kl)]
        g_prob = as_f32(g_prob, (B, L))
        g_prob_label = as_f32(g_prob_label, (B, L))
        with torch.cuda.device(dev):
            g_fe_out = torch.empty_like(fe_out)
            g_fx_out = torch.empty_like(fx_out)
            g_mulv = [torch.empty_like(fe_mu) for _ in range(4)]
            _poison(g_fe_out, g_fx_out, *g_mulv)
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
            if ctx.per_row:
                _lib.check(lib.mpvae_probit_backward_rows(C.byref(p), _ptr(label_mask), _ptr(row_weight),
                                                          _ptr(label_weight), stream), "mpvae_probit_backward_rows")
            elif label_weight is not None:
                _lib.check(lib.mpvae_probit_backward_label_weighted(C.byref(p), _ptr(label_mask), _ptr(row_weight),
                                                                    _ptr(label_weight), stream),
                           "mpvae_probit_backward_label_weighted")
            elif row_weight is not None:
                _lib.check(lib.mpvae_probit_backward_weighted(C.byref(p), _ptr(label_mask), _ptr(row_weight), stream),
                           "mpvae_probit_backward_weighted")
            elif label_mask is None:
                _lib.check(lib.mpvae_probit_backward(C.byref(p), stream), "mpvae_probit_backward")
            else:
                _lib.check(lib.mpvae_probit_backward_masked(C.byref(p), _ptr(label_mask), stream),
                           "mpvae_probit_backward_masked")
        #       y     fe_out    fe_mu      fe_logvar  fx_out    fx_mu      fx_logvar  r32  noise nll_c c_c flags spec
        return (None, g_fe_out, g_mulv[0], g_mulv[1], g_fx_out, g_mulv[2], g_mulv[3], g_r, None, None, None, None, None,
                None, None, None, None, None)   # peer, label_mask, row_weight, label_weight, per_row


def _predict_dims(name, fx_out, r32, S, noise, noise_spec):
    """The shape checks of a sampled prediction's inputs: (S, B, L, Z)."""
    if noise is None and noise_spec is None:
        raise ValueError(f"{name} needs either a noise tensor or a noise_spec")
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
    return S, B, L, Z


def _predict_tensors(fx_out, r32, noise, *optional):
    """The device and dtype checks of a sampled prediction's tensors, after the shape of each optional input:
    `optional` holds (name, tensor or None, expected shape) triples.  Returns fx_out, r32, noise and the optional
    tensors, contiguous (None stays None)."""
    names, tensors = ["fx_out", "r_sqrt_sigma", "noise"], [fx_out, r32, noise]
    for name, t, shape in optional:
        if t is not None and tuple(t.shape) != shape:
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {shape}")
        names.append(name)
        tensors.append(t)
    _check_tensors(names, tensors)
    return [t.contiguous() if t is not None else None for t in tensors]


def _predict_inputs(name, fx_out, r32, S, noise, noise_spec):
    """The checks of mpvae_probit_predict's inputs: (fx_out, r32, noise) contiguous, and (S, B, L, Z)."""
    dims = _predict_dims(name, fx_out, r32, S, noise, noise_spec)
    return (*_predict_tensors(fx_out, r32, noise), dims)


Out = namedtuple("Out", ["shape", "dtype"])     # an output of a sampled-prediction entry point, for _run_predict
Scratch = namedtuple("Scratch", ["nbytes"])     # a scratch block of one, besides the params' workspace


def _run_predict(entry, fx_out, r32, noise, noise_spec, flags, dims, *args, prob=True):
    """Runs the sampled-prediction entry point `entry` of the library: `args` are its C arguments between the params and
    the stream, in order.  Each Out(shape, dtype) is allocated on fx_out's device and passed as its pointer, each
    Scratch(nbytes) as its pointer and byte count; anything else is passed as is.  Outputs and scratch are poisoned under
    MPVAE_POISON_WORKSPACE=1.  `prob`: the entry point writes params.indiv_prob, a (B, L) fp32 output that comes first.
    Returns the outputs, in order.  With B == 0 they are returned with zero rows, and the library is not called."""
    S, B, L, Z = dims
    dev = fx_out.device
    with torch.cuda.device(dev):
        outs = [torch.empty((B, L), dtype=torch.float32, device=dev)] if prob else []
        blocks, c_args = [], []
        for a in args:
            if isinstance(a, Out):
                outs.append(torch.empty(a.shape, dtype=a.dtype, device=dev))
                c_args.append(_ptr(outs[-1]))
            elif isinstance(a, Scratch):
                blocks.append(torch.empty(a.nbytes, dtype=torch.uint8, device=dev))
                c_args += (_ptr(blocks[-1]), a.nbytes)
            else:
                c_args.append(a)
        if B == 0:
            return outs
        lib = _lib.lib()
        ws = torch.empty(int(lib.mpvae_workspace_bytes(S, B, L, Z, 0, flags)), dtype=torch.uint8, device=dev)
        _poison(ws, *blocks, *outs)
        p = _lib.ProbitParams()
        p.struct_bytes = C.sizeof(_lib.ProbitParams)
        p.flags = flags
        p.S, p.B, p.L, p.Z = S, B, L, Z
        p.fx_out, p.r, p.noise = _ptr(fx_out), _ptr(r32), _ptr(noise)
        _set_noise_spec(p, noise_spec, B)
        p.indiv_prob = _ptr(outs[0]) if prob else None
        p.workspace, p.workspace_bytes = _ptr(ws), ws.numel()
        _lib.check(getattr(lib, entry)(C.byref(p), *c_args, _stream(dev)), entry)
    return outs


def probit_predict(fx_out, r32, S, *, noise=None, noise_spec=None, flags=0):
    """indiv_prob (B, L) = mean over S samples of clamp(Phi(fx_out + noise.R^T)) (mpvae.py:170,180,203): the prediction
    of the feature branch, without labels and without the loss.  Bit-equal to `ProbitELBO`'s indiv_prob on the same
    fx_out, R and noise.  `noise` / `noise_spec` as for `ProbitELBO`; inference only (no autograd graph)."""
    fx_out, r32, noise, dims = _predict_inputs("probit_predict", fx_out, r32, S, noise, noise_spec)
    return _run_predict("mpvae_probit_predict", fx_out, r32, noise, noise_spec, flags, dims)[0]


def probit_predict_conditional(fx_out, r32, observed, S, *, noise=None, noise_spec=None, flags=0):
    """(prob (B, L), log_evidence (B,), ess (B,)): P(y_l = 1 | the row's observed labels, x) by importance-weighting
    probit_predict's S samples with the likelihood of the observed labels (mpvae_probit_predict_conditional).
    `observed` is an int8 (B, L) tensor on fx_out's device: 0 or 1 = observed with that value, any other value =
    unobserved; it is not read on the host.  Observed cells return their value; with nothing observed prob is
    probit_predict's bit for bit.  `noise` / `noise_spec` / `flags` as for probit_predict; inference only."""
    fx_out, r32, noise, dims = _predict_inputs("probit_predict_conditional", fx_out, r32, S, noise, noise_spec)
    S, B, L, Z = dims
    _check_observed(observed, (B, L), fx_out.device)
    observed = observed.contiguous()
    return tuple(_run_predict("mpvae_probit_predict_conditional", fx_out, r32, noise, noise_spec, flags, dims,
                              _ptr(observed), Out((B,), torch.float32), Out((B,), torch.float32)))


def ghk_workspace_bytes(S, B, L, Z, max_observed, flags=0):
    """Bytes of the GHK sampler's own scratch block (G, the per-row factors and index lists, the per-sample vectors)."""
    return int(_lib.lib().mpvae_ghk_workspace_bytes(S, B, L, Z, max_observed, flags))


def probit_predict_conditional_ghk(fx_out, r32, observed, S, max_observed, *, noise=None, noise_spec=None, flags=0,
                                   gram=None, zeta=None, uniform=None):
    """(prob (B, L), log_evidence (B,), ess (B,)): probit_predict_conditional's outputs from the GHK sampler
    (mpvae_probit_predict_conditional_ghk).  `max_observed` bounds every row's observed count (a row with more gets
    NaN outputs).  `gram`: the (L, L) fp32 R R^T of `contract_nt(r32, r32)` with the engine mpvae.label_gram picks, or
    None.  `zeta` / `uniform`: optional (S, B, L) fp32 draws for the observed cells (uniform in (0, 1)); None = the
    library's Philox stream.  `noise` / `noise_spec` / `flags` as for probit_predict; inference only."""
    dims = _predict_dims("probit_predict_conditional_ghk", fx_out, r32, S, noise, noise_spec)
    S, B, L, Z = dims
    _check_observed(observed, (B, L), fx_out.device)
    max_observed = int(max_observed)
    if not 0 <= max_observed <= L:
        raise ValueError(f"max_observed={max_observed} outside [0, {L}]")
    fx_out, r32, noise, gram, zeta, uniform = _predict_tensors(
        fx_out, r32, noise, ("gram", gram, (L, L)), ("zeta", zeta, (S, B, L)), ("uniform", uniform, (S, B, L)))
    observed = observed.contiguous()
    return tuple(_run_predict("mpvae_probit_predict_conditional_ghk", fx_out, r32, noise, noise_spec, flags, dims,
                              _ptr(observed), _ptr(gram), _ptr(zeta), _ptr(uniform),
                              Scratch(ghk_workspace_bytes(S, B, L, Z, max_observed, flags)), max_observed,
                              Out((B,), torch.float32), Out((B,), torch.float32)))


def probit_sample_labels(fx_out, r32, S, *, noise=None, noise_spec=None, flags=0, uniform=None):
    """(B, S, ceil(L / 32)) int32 bits of S joint label samples per row, y = (U < E) with E the clamped probit that
    probit_predict averages, on its noise (mpvae_probit_sample_labels): label l of sample s is bit l % 32 of word l / 32.
    `uniform`: optional (S, B, L) fp32 U in (0, 1); None = the library's own Philox stream, keyed by global row.
    `noise` / `noise_spec` / `flags` as for probit_predict; inference only."""
    dims = _predict_dims("probit_sample_labels", fx_out, r32, S, noise, noise_spec)
    S, B, L, Z = dims
    fx_out, r32, noise, uniform = _predict_tensors(fx_out, r32, noise, ("uniform", uniform, (S, B, L)))
    return _run_predict("mpvae_probit_sample_labels", fx_out, r32, noise, noise_spec, flags, dims, _ptr(uniform),
                        Out((B, S, (L + 31) // 32), torch.int32), prob=False)[0]


def check_set_args(beta, max_size):
    """beta as a float, refused unless it is positive with a finite square (beta^2 enters every weight of the F-measure
    decoder); max_size refused below 0 (None: no bound)."""
    beta = float(beta)
    if not (beta > 0.0 and math.isfinite(beta * beta)):
        raise ValueError(f"beta must be positive with a finite square, got {beta}")
    if max_size is not None and int(max_size) < 0:
        raise ValueError(f"max_size must be >= 0 (None for no bound), got {max_size}")
    return beta


def f1_sets(bits, L, beta=1.0, max_size=None):
    """(sets (B, L) bool, expected_f (B,) fp64, size (B,) int32): per row, the set of at most `max_size` labels (None:
    no bound) that maximises the expected F_beta over the row's S label samples in `bits` ((B, S, ceil(L / 32)) int32,
    probit_sample_labels' layout), by the GFM algorithm (mpvae_f1_sets).  One launch; no host synchronisation."""
    if not isinstance(bits, torch.Tensor) or bits.dtype != torch.int32:
        raise TypeError(f"bits must be an int32 tensor, got {getattr(bits, 'dtype', type(bits))}")
    L = int(L)
    if L < 1:
        raise ValueError(f"label_dim must be positive, got {L}")
    W = (L + 31) // 32
    if bits.dim() != 3 or bits.shape[2] != W or bits.shape[1] < 1:
        raise ValueError(f"bits has shape {tuple(bits.shape)}, expected (batch, n_sample >= 1, {W}) for {L} labels")
    beta = check_set_args(beta, max_size)
    max_size = L if max_size is None else int(max_size)
    max_size = min(max_size, L)
    if not bits.is_cuda:
        raise RuntimeError(f"mpvae_b200: bits is on {bits.device}; the F-measure decoder runs on CUDA only "
                           "(there is no CPU fallback)")
    B, S = bits.shape[0], bits.shape[1]
    dev = bits.device
    sets = torch.empty((B, L), dtype=torch.uint8, device=dev)
    expected_f = torch.empty(B, dtype=torch.float64, device=dev)
    size = torch.empty(B, dtype=torch.int32, device=dev)
    if B == 0:
        return sets.view(torch.bool), expected_f, size
    bits = bits.contiguous()
    lib = _lib.lib()
    with torch.cuda.device(dev):
        ws_bytes = int(lib.mpvae_f1_sets_workspace_bytes(B, S, L))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _poison(ws, sets, expected_f, size)
        _lib.check(lib.mpvae_f1_sets(_ptr(bits), B, S, L, beta, max_size, _ptr(sets), _ptr(expected_f), _ptr(size),
                                     _ptr(ws), ws_bytes, _stream(dev)), "mpvae_f1_sets")
    return sets.view(torch.bool), expected_f, size


def check_set_bits(bits, B, L, device):
    """Refuses `bits` that are not an int32 (B, C >= 1, ceil(L / 32)) tensor on `device` (sets in sample_labels'
    layout)."""
    if not isinstance(bits, torch.Tensor) or bits.dtype != torch.int32:
        raise TypeError(f"bits must be an int32 tensor, got {getattr(bits, 'dtype', type(bits))}")
    W = (L + 31) // 32
    if bits.dim() != 3 or bits.shape[0] != B or bits.shape[1] < 1 or bits.shape[2] != W:
        raise ValueError(f"bits has shape {tuple(bits.shape)}, expected ({B}, n_sets >= 1, {W}) for {L} labels")
    if bits.device != device:
        raise RuntimeError(f"mpvae_b200: bits is on {bits.device}, expected {device}")


def check_max_flips(max_flips):
    """max_flips as an int (None: no bound, 2^31 - 1), refused below 0."""
    if max_flips is None:
        return 2 ** 31 - 1
    if int(max_flips) < 0:
        raise ValueError(f"max_flips must be >= 0 (None for no bound), got {max_flips}")
    return min(int(max_flips), 2 ** 31 - 1)


def mode_workspace_bytes(S, B, L):
    """Bytes of the mode entry points' own scratch block (about 8 S L bytes per row)."""
    return int(_lib.lib().mpvae_mode_workspace_bytes(S, B, L))


def probit_score_sets(fx_out, r32, bits, S, *, noise=None, noise_spec=None, flags=0):
    """(log_prob (B, C) fp64, ess (B, C) fp64) of the C label sets per row in `bits` ((B, C, ceil(L / 32)) int32,
    sample_labels' layout) under the S-sample mixture probit_predict averages, on its noise
    (mpvae_probit_score_sets).  `noise` / `noise_spec` / `flags` as for probit_predict; inference only."""
    fx_out, r32, noise, dims = _predict_inputs("probit_score_sets", fx_out, r32, S, noise, noise_spec)
    S, B, L, Z = dims
    check_set_bits(bits, B, L, fx_out.device)
    bits = bits.contiguous()
    C_ = bits.shape[1]
    return tuple(_run_predict("mpvae_probit_score_sets", fx_out, r32, noise, noise_spec, flags, dims, _ptr(bits), C_,
                              Out((B, C_), torch.float64), Out((B, C_), torch.float64),
                              Scratch(mode_workspace_bytes(S, B, L)), prob=False))


def probit_predict_mode(fx_out, r32, S, max_flips=None, *, noise=None, noise_spec=None, flags=0):
    """(sets (B, L) bool, log_prob (B,) fp64, ess (B,) fp64, size (B,) int32, flips (B,) int32): per row the label set
    that maximises the S-sample mixture's probability, by candidates and steepest single-flip ascent
    (mpvae_probit_predict_mode).  `noise` / `noise_spec` / `flags` as for probit_predict; inference only."""
    max_flips = check_max_flips(max_flips)
    fx_out, r32, noise, dims = _predict_inputs("probit_predict_mode", fx_out, r32, S, noise, noise_spec)
    S, B, L, Z = dims
    sets, log_prob, ess, size, flips = _run_predict(
        "mpvae_probit_predict_mode", fx_out, r32, noise, noise_spec, flags, dims, max_flips,
        Out((B, L), torch.uint8), Out((B,), torch.float64), Out((B,), torch.float64), Out((B,), torch.int32),
        Out((B,), torch.int32), Scratch(mode_workspace_bytes(S, B, L)), prob=False)
    return sets.view(torch.bool), log_prob, ess, size, flips


# ---- closed-form prediction (csrc/predictive.cu): the S -> infinity limit of probit_predict ----

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
    _poison(scale)
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
    _poison(rho)
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
    _poison(prob)
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
    _poison(scale, prob)
    lib = _lib.lib()

    def launch():
        stream = _stream(dev)
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
    _poison(out)
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
