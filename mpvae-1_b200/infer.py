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


def _score_rows(model, feats: torch.Tensor, args, batch_size: Optional[int], gather: bool, group, width: int, score):
    """The test-time row loop: `model.eval()`, `args.mode = 'test'`, this rank's contiguous slice of the N rows in
    batches of `batch_size` (default args.batch_size, test.py:41-43), then the gather of the slices.  score(a, b, args)
    returns the (b - a, width) result of rows [a, b); it sees args.dp_global_batch = N, args.dp_row0 = a and the
    pass's one noise offset."""
    args = copy.copy(args)
    args.mode = "test"
    was_training = model.training
    model.eval()
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    n = feats.shape[0]
    lo, hi = shard_rows(n, rank, world)
    bs = min(batch_size or getattr(args, "batch_size", 128), max(hi - lo, 1))       # test.py:41
    out = []
    n_batches = (hi - lo - 1) // bs + 1 if hi > lo else 0                            # test.py:43
    for i in range(n_batches):
        a, b = lo + bs * i, min(lo + bs * (i + 1), hi)
        args.dp_global_batch, args.dp_row0 = n, a
        # one Philox offset for the whole pass: a row's noise is keyed by its GLOBAL row index (dp_row0 + local row), so
        # predictions do not depend on the world size or on how the rows are batched
        args.noise_offset = getattr(args, "noise_offset_base", 0)
        out.append(score(a, b, args))
    local = torch.cat(out, 0) if out else feats.new_empty((0, width))
    if was_training:
        model.train()
    if world == 1 or not gather:
        return local
    # gather the row slices (padded to the largest shard so one all_gather serves unequal shards)
    sizes = [h - l for l, h in (shard_rows(n, r, world) for r in range(world))]
    width = local.shape[1]
    padded = local.new_zeros((max(sizes), width))
    padded[:local.shape[0]] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([p[:k] for p, k in zip(parts, sizes)], 0)


@torch.no_grad()
def predict_proba(model, feats: torch.Tensor, labels: Optional[torch.Tensor], args, batch_size: Optional[int] = None,
                  loss_fn=None, gather: bool = True, group=None, predict_fn=None):
    """Returns (indiv_prob (N, L), summed-loss dict).  `feats` / `labels` are device tensors for ALL N rows.

    `labels=None` scores rows that have no labels: each batch runs only the feature branch (`model.feat_forward`) and
    `mpvae.predict` (or `predict_fn`, same signature, e.g. `mpvae.predict_exact`), and the loss dict is None.  With
    labels, `VAE.forward` draws the label branch's reparameterisation noise first, so under the same torch seed the
    feature branch -- and hence the predictions -- differ from the label-free call; on the same fx_out the two give the
    same bits."""
    if labels is None and predict_fn is None:
        from .mpvae import predict as predict_fn
    if labels is not None and loss_fn is None:
        from .mpvae import compute_loss as loss_fn
    sums = {"total_loss": 0.0, "nll_loss": 0.0, "c_loss": 0.0}

    def score(a, b, args):
        x = feats[a:b]
        if labels is None:
            feat_out, _, _ = model.feat_forward(x)
            return predict_fn(feat_out, model.r_sqrt_sigma, args)
        y = labels[a:b].float()
        label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar = model(y, x)
        out = loss_fn(y, label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar, model.r_sqrt_sigma, args)
        sums["total_loss"] = sums["total_loss"] + out[0] * (b - a)                   # test.py:67-70
        sums["nll_loss"] = sums["nll_loss"] + out[1] * (b - a)
        sums["c_loss"] = sums["c_loss"] + out[3] * (b - a)
        return out[6]

    width = labels.shape[1] if labels is not None else model.r_sqrt_sigma.shape[0]
    probs = _score_rows(model, feats, args, batch_size, gather, group, width, score)
    return probs, (sums if labels is not None else None)


@torch.no_grad()
def predict_pairs(model, feats: torch.Tensor, pairs, args, batch_size: Optional[int] = None, gather: bool = True,
                  group=None):
    """(N, P) P(y_i = 1, y_j = 1 | x) for each row of `feats` (device tensor, ALL N rows) and each (i, j) of the (P, 2)
    label pairs (`mpvae.all_pairs(L)`: every pair), in closed form (`mpvae.PairPredictor`, prepared once per call).
    Same row sharding, batching and gather as `predict_proba`; a pair (i, i) gives the column of
    `predict_proba(..., predict_fn=mpvae.predict_exact)` under the same torch seed.  fx_out is drawn by
    `model.feat_forward` (its latent sample); the probit noise is integrated out."""
    from .mpvae import PairPredictor
    predictor = PairPredictor(model.r_sqrt_sigma, pairs, args)
    width = torch.as_tensor(pairs).shape[0]
    return _score_rows(model, feats, args, batch_size, gather, group, width,
                       lambda a, b, _: predictor(model.feat_forward(feats[a:b])[0]))
