"""Test-time inference path: the loop of the reference's test.py:45-77 (and fairsoft_evaluate.py:59-81).

`model.eval()`, `torch.no_grad()`, `args.mode = 'test'` so that S = args.n_test_sample (mpvae.py:158); only
`indiv_prob` (mean_s E_x, the prediction) is consumed downstream (test.py:72), but the reference computes -- and
this path returns -- all 8 outputs.  Rows are independent, so with G ranks each rank scores a contiguous slice
and the predictions are gathered (no exchange inside the path, SURVEY 8e)."""
from __future__ import annotations

import copy
from typing import Optional

import torch
import torch.distributed as dist

from .train import shard_rows


@torch.no_grad()
def predict_proba(model, feats: torch.Tensor, labels: Optional[torch.Tensor], args, batch_size: Optional[int] = None,
                  loss_fn=None, gather: bool = True, group=None, predict_fn=None):
    """Returns (indiv_prob (N, L), summed-loss dict).  `feats` / `labels` are device tensors for ALL N rows.

    `labels=None` scores rows that have no labels: each batch runs only the feature branch (`model.feat_forward`) and
    `mpvae.predict` (or `predict_fn`, same signature), and the loss dict is None.  With labels, `VAE.forward` draws the
    label branch's reparameterisation noise first, so under the same torch seed the feature branch -- and hence the
    predictions -- differ from the label-free call; on the same fx_out the two give the same bits."""
    if labels is None and predict_fn is None:
        from .mpvae import predict as predict_fn
    if labels is not None and loss_fn is None:
        from .mpvae import compute_loss as loss_fn
    args = copy.copy(args)
    args.mode = "test"
    was_training = model.training
    model.eval()
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    n = feats.shape[0]
    lo, hi = shard_rows(n, rank, world)
    bs = min(batch_size or getattr(args, "batch_size", 128), max(hi - lo, 1))       # test.py:41
    probs, sums = [], {"total_loss": 0.0, "nll_loss": 0.0, "c_loss": 0.0}
    n_batches = (hi - lo - 1) // bs + 1 if hi > lo else 0                            # test.py:43
    for i in range(n_batches):
        a, b = lo + bs * i, min(lo + bs * (i + 1), hi)
        x = feats[a:b]
        args.dp_global_batch, args.dp_row0 = n, a
        # one Philox offset for the whole pass: a row's noise is keyed by its GLOBAL row index (dp_row0 + local row), so
        # predictions do not depend on the world size or on how the rows are batched
        args.noise_offset = getattr(args, "noise_offset_base", 0)
        if labels is None:
            feat_out, _, _ = model.feat_forward(x)
            probs.append(predict_fn(feat_out, model.r_sqrt_sigma, args))
            continue
        y = labels[a:b].float()
        label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar = model(y, x)
        out = loss_fn(y, label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar, model.r_sqrt_sigma, args)
        probs.append(out[6])
        sums["total_loss"] = sums["total_loss"] + out[0] * (b - a)                   # test.py:67-70
        sums["nll_loss"] = sums["nll_loss"] + out[1] * (b - a)
        sums["c_loss"] = sums["c_loss"] + out[3] * (b - a)
    width = labels.shape[1] if labels is not None else model.r_sqrt_sigma.shape[0]
    if labels is None:
        sums = None
    local = torch.cat(probs, 0) if probs else feats.new_empty((0, width))
    if was_training:
        model.train()
    if world == 1 or not gather:
        return local, sums
    # gather the row slices (padded to the largest shard so one all_gather serves unequal shards)
    sizes = [h - l for l, h in (shard_rows(n, r, world) for r in range(world))]
    width = local.shape[1]
    padded = local.new_zeros((max(sizes), width))
    padded[:local.shape[0]] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([p[:k] for p, k in zip(parts, sizes)], 0), sums
