"""Data-parallel training step: the loop body of the reference's train.py:103-129 (and its fairness twin,
fairsoft_train.py:47-146) as one object, one process per GPU.

    zero_grad -> batch shard -> VAE.forward -> compute_loss -> [extra regulariser] -> backward
              -> all-reduce(flat fp32 bucket: g_R || every MLP gradient) -> clip_grad_norm_ -> Adam -> StepLR

Batch rows are the unit that shards (every loss term is a mean over rows, mpvae.py:147,122,190): rank r owns
rows [r*B/G, (r+1)*B/G) of the global batch, gradients are averaged, and every rank then applies the identical
clip + Adam update, so parameters stay replicated without a broadcast.  The one exchange per step is an NCCL
all-reduce over NVLink; the g_R segment is launched from an autograd hook as soon as the probit backward has
produced it, so it overlaps the MLP backward.  Noise is Philox keyed by the GLOBAL row index, which makes the
result independent of the world size (an external (S, B_global, Z) noise tensor is sliced instead).

`peer_all=True` replaces every NCCL call of the step by the library's own exchange over NVLink peer memory (the bucket
is allocated there and summed in place; the loss terms ride in its scalar slots), which is what lets GraphedTrainStep
capture the step on every rank.

The reference has no distributed code at all (SURVEY.md section 2); with world_size == 1 this object is exactly
its single-GPU step.
"""
from __future__ import annotations

import copy
from typing import Callable, NamedTuple, Optional

import torch
import torch.distributed as dist
import torch.nn as nn


class StepOutput(NamedTuple):
    total_loss: torch.Tensor
    nll_loss: torch.Tensor
    nll_loss_x: torch.Tensor
    c_loss: torch.Tensor
    c_loss_x: torch.Tensor
    kl_loss: torch.Tensor
    indiv_prob: torch.Tensor          # this rank's rows
    indiv_prob_label: torch.Tensor
    grad_norm: torch.Tensor
    stepped: bool


def shard_rows(n_rows: int, rank: int, world: int):
    """Contiguous, near-equal row shards: rank r gets [lo, hi).  (Equal shards when world | n_rows.)"""
    base, rem = divmod(n_rows, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class GradBucket:
    """One flat fp32 buffer holding [g_R | pad | all fp32 parameter gradients | pad | 8 scalar slots]; .grad of every fp32
    parameter is a view into it (autograd accumulates in place), so the all-reduce needs no gather / scatter copies.
    The segments start at multiples of four floats (16-byte accesses of the peer-memory exchange); the scalar slots
    carry the step's loss terms through the same exchange when the step runs without NCCL.  `alloc(numel)` supplies the
    storage (peer-mapped memory for `peer_all`), default torch.zeros."""

    N_SCALARS = 8

    def __init__(self, r_shadow: Optional[torch.Tensor], params, alloc: Optional[Callable] = None):
        self.params = [p for p in params if p.requires_grad and p.dtype == torch.float32]
        dev = (r_shadow if r_shadow is not None else self.params[0]).device
        self.r_numel = r_shadow.numel() if r_shadow is not None else 0
        self.mlp_off = -(-self.r_numel // 4) * 4
        n_mlp = sum(p.numel() for p in self.params)
        self.grads_end = self.mlp_off + n_mlp
        self.scal_off = -(-self.grads_end // 4) * 4
        total = self.scal_off + self.N_SCALARS
        self.flat = alloc(total) if alloc is not None else torch.zeros(total, dtype=torch.float32, device=dev)
        assert self.flat.numel() == total and self.flat.dtype == torch.float32
        self.grads = self.flat[:self.grads_end]             # what the gradient norm is taken over (padding stays zero)
        self.scalars = self.flat[self.scal_off:]
        self.r_view = self.flat[:self.r_numel].view_as(r_shadow) if r_shadow is not None else None
        self.views = []
        off = self.mlp_off
        for p in self.params:
            self.views.append(self.flat[off:off + p.numel()].view_as(p))
            off += p.numel()

    def attach(self, r_shadow):
        self.flat.zero_()
        if r_shadow is not None:
            r_shadow.grad = self.r_view
        for p, v in zip(self.params, self.views):
            p.grad = v


class DataParallelStep:
    """`step(input_label, input_feat)` = one training step on the GLOBAL batch, this rank computing its shard."""

    def __init__(self, model: nn.Module, optimizer, scheduler, args, *, clip_norm: float = 100.0,
                 skip_nonfinite: bool = False, group=None, loss_fn: Optional[Callable] = None,
                 regulariser: Optional[Callable] = None, distributed: bool = True, peer_g_r: bool = False,
                 peer_all: bool = False, row_objective: Optional[Callable] = None):
        if row_objective is not None and regulariser is not None:
            raise ValueError("DataParallelStep takes row_objective or regulariser, not both: fold the regulariser into "
                             "the row objective")
        self.model, self.optimizer, self.scheduler = model, optimizer, scheduler
        self.args = copy.copy(args)
        self.clip_norm = clip_norm                 # 100 in train.py:126, 10 in fairsoft_train.py:141
        self.skip_nonfinite = skip_nonfinite       # has_finite_grad guard of fairsoft_train.py:142
        self.group = group
        self.world = dist.get_world_size(group) if (distributed and dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        # Only the probit noise is keyed by the GLOBAL row (Philox), so the loss is independent of the world size given
        # the encoder outputs.  Dropout masks and the reparameterisation eps come from torch's generator, which every
        # rank seeds identically (needed for identical initial weights): without the offset below all ranks would draw
        # the SAME eps / masks for their different rows.  `decorrelate_rng()` moves this rank's generators to a
        # rank-specific stream; call it AFTER the model has been built.  (Those draws then still depend on the world
        # size: that is inherent to sharding torch's generator and is a documented limitation.)
        self._rng_decorrelated = False
        self._library_loss = loss_fn is None
        if loss_fn is None:
            from .mpvae import compute_loss as loss_fn
        self.loss_fn = loss_fn
        self.regulariser = regulariser             # callable(StepOutput-like 8-tuple, row slice) -> scalar tensor
        # callable(8-tuple of compute_loss(..., reduction='none'), row slice) -> (rows,) tensor phi: the step minimises
        # sum_b phi_b / B over the global batch (see step)
        self.row_objective = row_objective
        self.step_no = 0
        r = getattr(model, "r_sqrt_sigma", None)
        self.r_param = r if (r is not None and r.requires_grad) else None
        self.r_shadow = None
        if self.r_param is not None:
            # fp32 working copy of the fp64 Parameter (the reference casts per call, mpvae.py:165); its gradient
            # lives in the bucket, and is cast back to fp64 for the optimizer after the all-reduce
            self.r_shadow = self.r_param.detach().float().requires_grad_(True)
        others = [p for n, p in model.named_parameters() if p is not self.r_param]
        # peer_all=True: the whole bucket lives in peer-mapped memory and is summed over the ranks by the library's
        # exchange kernel (peer.PeerBucket) -- no NCCL call anywhere in the step, which is what GraphedTrainStep needs
        # at world_size > 1.  Set-up is collective: if it fails on any rank, every rank keeps the NCCL path.
        self.pbucket = None
        alloc = None
        if peer_all and self.world > 1 and next(model.parameters()).is_cuda:
            def alloc(numel):
                from .peer import PeerBucket
                try:
                    self.pbucket = PeerBucket(numel, next(model.parameters()).device, self.group)
                except RuntimeError as e:
                    if self.rank == 0:
                        print(f"[mpvae_b200] peer_all unavailable ({e}); NCCL all-reduce")
                    return torch.zeros(numel, dtype=torch.float32, device=next(model.parameters()).device)
                return self.pbucket.flat
        self.bucket = GradBucket(self.r_shadow, others, alloc)
        self._pending = []
        self._r_issued = False          # the g_R segment's all-reduce of this step has been issued
        # peer_g_r=True: g_R is summed over the ranks inside the probit backward, over NVLink peer memory (peer.py),
        # instead of the NCCL all-reduce of that bucket segment.  Off by default: measured on 2 and 4 B200 the
        # exchange itself is 5-15 % faster than NCCL's (both move the same bytes over NVLink), but inside the
        # backward it cannot overlap the MLP backward the way the asynchronous NCCL call issued from the hook does
        self._want_ring = peer_g_r and self.world > 1 and self.r_shadow is not None and self._library_loss
        self.ring = None
        self._ring_step = False
        self._shadow_fresh = False      # the fused optimizer wrote the fp32 shadow of R during the last step
        if self.world > 1 and self.r_shadow is not None:
            self.r_shadow.register_post_accumulate_grad_hook(self._reduce_r_early)

    def decorrelate_rng(self, base_seed: Optional[int] = None):
        """Give this rank its own dropout / reparameterisation random stream (see __init__)."""
        if self.world > 1 and not self._rng_decorrelated:
            seed = (torch.initial_seed() if base_seed is None else int(base_seed)) + 7919 * (self.rank + 1)
            torch.manual_seed(seed)
            self._rng_decorrelated = True

    # -- collectives --------------------------------------------------------------------------------------
    def _peer_ring(self, n_rows: int):
        """The ring, if this step can use it: every rank needs at least one row (an idle rank would not reach the
        backward and the others would wait for its tiles)."""
        if not self._want_ring or n_rows < self.world:
            return None
        if self.ring is None:
            from .peer import PeerRing
            L, Z = self.r_shadow.shape
            if not (self.r_shadow.is_cuda and L * Z >= (1 << 16)):
                self._want_ring = False           # tiny R (or the CPU tests): the NCCL / gloo all-reduce of the bucket
                return None
            self.ring = PeerRing(L, Z, self.r_shadow.device, self.group)
        return self.ring

    def _reduce_r_early(self, _):
        """Fires as soon as the probit backward has written g_R: overlap its all-reduce with the MLP backward."""
        if self._ring_step or self._r_issued or self.pbucket is not None:
            return                                # g_R arrived already summed (peer ring) / already on its way / peer bucket
        self._r_issued = True
        seg = self.bucket.flat[:self.bucket.r_numel]
        self._pending.append(dist.all_reduce(seg, group=self.group, async_op=True))

    def _finish_reduce(self, divide: bool = True):
        """Every rank issues the SAME collectives in the SAME order whatever its local data was: first the g_R segment
        (from the hook if the probit backward ran on this rank, else here -- an empty shard, a frozen forward),
        then the MLP gradients.  A rank whose sequence depended on its shard would hang NCCL."""
        if self.world == 1:
            return
        if self.pbucket is not None:
            # one in-place exchange over NVLink peer memory: MLP gradients + the scalar slots, and g_R too unless the
            # probit backward already delivered it summed
            first = self.bucket.mlp_off if (self._ring_step or not self.bucket.r_numel) else 0
            self.pbucket.allreduce(first)
            if divide:
                self.bucket.grads.div_(self.world)
            return
        if self.bucket.r_numel and not self._ring_step:
            self._reduce_r_early(None)            # no-op when the hook already issued it
        seg = self.bucket.flat[self.bucket.mlp_off:self.bucket.grads_end]
        if seg.numel():
            self._pending.append(dist.all_reduce(seg, group=self.group, async_op=True))
        for w in self._pending:
            w.wait()
        self._pending = []
        self._r_issued = False
        if divide:
            self.bucket.grads.div_(self.world)

    # -- the step -------------------------------------------------------------------------------------------
    def step(self, input_label: torch.Tensor, input_feat: torch.Tensor, noise: Optional[torch.Tensor] = None,
             r_override: Optional[torch.Tensor] = None, label_mask: Optional[torch.Tensor] = None,
             row_weight: Optional[torch.Tensor] = None, pos_weight: Optional[torch.Tensor] = None,
             neg_weight: Optional[torch.Tensor] = None) -> StepOutput:
        """`input_label` (B, L) and `input_feat` (B, F) are the GLOBAL batch (train.py:106-111); every rank slices
        its rows.  `noise`, if given, is the global (S, B, Z) tensor (validation mode).  `r_override` is the
        fresh non-trainable R of residue_sigma == 'random' (train.py:120-122).  `label_mask`, if given, is the global
        (B, L) mask of observed labels (`compute_loss`): each rank passes its rows' slice to the loss as
        `label_mask=`; without it the loss is called exactly as before, so custom loss functions keep working.
        `row_weight`, if given, is the global (B,) row weight (`compute_loss`), sliced and passed as `row_weight=` in the
        same way.  Each rank's terms are sum_b w_b t_b / (its rows) and the shard weighting below makes the global loss
        sum over all rows of w_b t_b / B, as in one process.  `pos_weight` / `neg_weight`, if given, are the (L,) label
        weights (`compute_loss`): they weigh labels, not rows, so every rank passes them whole, again only when given.

        With `row_objective=f` (constructor), the loss is called with `reduction='none'` and `f(out, slice(lo, hi))`
        returns the shard's (hi - lo,) per-row values phi_b (e.g. `out[0] * keep`, or a group-DRO mixture of out[2]).  The
        step minimises sum_b phi_b / B over the global batch: each rank backpropagates phi.sum() * world / B, and the
        gradient average divides by world.  A selection over the global batch (a quantile of all rows' losses) is f's
        business: it may all-gather the detached terms itself.  The returned scalars stay the batch means of the per-row
        terms, so logging is unchanged."""
        args = self.args
        n_rows = input_label.shape[0]
        lo, hi = shard_rows(n_rows, self.rank, self.world)
        y, x = input_label[lo:hi], input_feat[lo:hi]
        args.dp_global_batch, args.dp_row0 = n_rows, lo
        ring = self._peer_ring(n_rows)
        args.peer_ring = ring
        # the ring only acts in the dense regime with the library's own backward; mirror ProbitELBO's decision
        S_now = args.n_train_sample if getattr(args, "mode", "train") == "train" else args.n_test_sample
        self._ring_step = ring is not None and ring.applies(S_now, hi - lo, ring.L, ring.Z, int(getattr(args, "mpvae_flags", 0)))
        if getattr(args, "noise_offset_auto", True):
            args.noise_offset = self.step_no         # same Philox offset on every rank
        if self.r_shadow is not None and not self._shadow_fresh:
            with torch.no_grad():
                self.r_shadow.copy_(self.r_param)
        self.bucket.attach(self.r_shadow)             # optimizer.zero_grad() of train.py:103 (in place, one memset)
        self._r_issued = False

        if hi > lo or self.world == 1:
            label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar = self.model(y, x)
            r = r_override if r_override is not None else (self.r_shadow if self.r_shadow is not None
                                                            else self.model.r_sqrt_sigma)
            kw = {} if noise is None else {"noise": noise[:, lo:hi]}
            if label_mask is not None:
                kw["label_mask"] = label_mask[lo:hi]
            if row_weight is not None:
                kw["row_weight"] = row_weight[lo:hi]
            if pos_weight is not None:
                kw["pos_weight"] = pos_weight
            if neg_weight is not None:
                kw["neg_weight"] = neg_weight
            if self.row_objective is not None:
                kw["reduction"] = "none"
            out = self.loss_fn(y, label_out, label_mu, label_logvar, feat_out, feat_mu, feat_logvar, r, args, **kw)
            if self.row_objective is not None:
                phi = self.row_objective(out, slice(lo, hi))
                if not isinstance(phi, torch.Tensor) or phi.shape != (hi - lo,):
                    raise ValueError(f"row_objective must return a ({hi - lo},) tensor (one value per row of the shard), "
                                     f"got {getattr(phi, 'shape', type(phi))}")
                (phi.sum() * (self.world / max(n_rows, 1))).backward()
                out = tuple(t.detach().mean() for t in out[:6]) + tuple(out[6:])
            else:
                total = out[0]
                if self.regulariser is not None:
                    extra = self.regulariser(out, slice(lo, hi))
                    if extra is not None:
                        total = total + extra
                # every term is a mean over this rank's rows; weight by the shard size so unequal shards still average
                weight = (hi - lo) * self.world / max(n_rows, 1)
                (total * weight if weight != 1.0 else total).backward()
        else:
            # a ragged last batch with fewer rows than ranks leaves this rank without a row: it contributes zero
            # gradients (the bucket was just zeroed) and zero-weighted scalars, and still joins every collective below
            zero = self.bucket.flat.new_zeros(())
            empty = input_label.new_zeros((0, input_label.shape[1]), dtype=torch.float32)
            out = (zero,) * 6 + (empty, empty)
        from .optim import FusedAdam
        fused = isinstance(self.optimizer, FusedAdam) and not self.skip_nonfinite and self.bucket.flat.is_cuda
        if self.pbucket is not None and hi > lo:
            # the step's loss terms ride in the bucket's scalar slots through the same exchange (row-weighted sums)
            self.bucket.scalars[:6].copy_(torch.stack([t.detach().float() for t in out[:6]]) * ((hi - lo) / max(n_rows, 1)))
        self._finish_reduce(divide=not fused)
        stepped = True
        self._shadow_fresh = False
        if fused:
            # clip + Adam as three launches over the flat bucket (optim.py); the 1/world of the gradient average is
            # folded into the gradient multiplier, g_R is consumed as fp32, the fp32 shadow of R is refreshed in place
            f32 = {self.r_param: self.bucket.r_view} if self.r_param is not None else None
            shadows = {self.r_param: self.r_shadow} if self.r_param is not None else None
            self.optimizer.step(max_norm=self.clip_norm, grad_scale=1.0 / self.world, flat_grad=self.bucket.grads,
                                f32_grads=f32, f32_shadows=shadows)
            grad_norm = self.optimizer.grad_norm
            self._shadow_fresh = self.r_param is not None and self.r_param in self.optimizer.shadowed
            if self.scheduler is not None:
                self.scheduler.step()
        else:
            if self.r_param is not None:
                self.r_param.grad = self.bucket.r_view.double()
            params = [p for p in self.model.parameters() if p.grad is not None]
            grad_norm = nn.utils.clip_grad_norm_(params, self.clip_norm)
            if self.skip_nonfinite and not bool(torch.isfinite(grad_norm)):
                stepped = False
            if stepped:
                self.optimizer.step()
                if self.scheduler is not None:
                    self.scheduler.step()
        self.step_no += 1
        scal = [t.detach() for t in out[:6]]
        if self.pbucket is not None:
            scal = list(self.bucket.scalars[:6].clone().unbind(0))
        elif self.world > 1:
            packed = torch.stack([t.float() for t in scal]) * ((hi - lo) / max(n_rows, 1))
            dist.all_reduce(packed, group=self.group)
            scal = list(packed.unbind(0))
        return StepOutput(*scal, out[6].detach(), out[7].detach(), grad_norm, stepped)


def train_one_epoch(step: DataParallelStep, feats, labels, batch_size: int, order=None, skip_empty: bool = True,
                    masks=None, weights=None, pos_weight=None, neg_weight=None):
    """Epoch driver with the reference's batching (train.py:98-111): int(N/bs)+1 steps, ragged (possibly empty)
    last batch.  `feats` / `labels` are device tensors (kept resident: SURVEY 8f-N4); returns per-step outputs.
    `masks`, if given, is the (N, L) mask of observed labels (`compute_loss`), sliced by the same index as `labels`;
    `weights`, if given, the (N,) row weights (`compute_loss(..., row_weight=)`), sliced the same way;
    `pos_weight` / `neg_weight`, if given, the (L,) label weights (`compute_loss`), passed to every step as they are.
    `skip_empty=False` reproduces the reference literally when bs | N: it runs the step on the empty batch, whose
    losses are NaN means (train.py:102; compute_loss returns them) and whose NaN gradients then reach Adam."""
    n = feats.shape[0]
    if order is None:
        order = torch.arange(n, device=feats.device)
    outs = []
    for i in range(int(n / float(batch_size)) + 1):
        idx = order[i * batch_size:min(batch_size * (i + 1), n)]
        if idx.numel() == 0 and skip_empty:
            continue          # the reference computes NaN losses on the empty batch and steps on them
        kw = {}
        if masks is not None:
            kw["label_mask"] = masks[idx]
        if weights is not None:
            kw["row_weight"] = weights[idx]
        if pos_weight is not None:
            kw["pos_weight"] = pos_weight
        if neg_weight is not None:
            kw["neg_weight"] = neg_weight
        outs.append(step.step(labels[idx], feats[idx], **kw))
    return outs


class GraphedTrainStep:
    """The whole training step (train.py:103-129) captured ONCE per batch size as a CUDA graph and replayed.

    For the reference's small configurations (yeast, mirflickr: 14-81 labels, batch 128) the step is a few hundred
    tiny launches, so the GPU idles while Python dispatches them; replaying a captured graph removes that host work.
    What makes the step capturable:
      * inputs live in static device buffers (`step()` copies the batch in, then replays);
      * the Philox stream offset is a DEVICE counter the noise kernel reads and the graph increments, so every replay
        draws fresh noise (`mpvae_probit_params.noise_offset_dev`);
      * Adam runs with `capturable=True` and a tensor learning rate; StepLR keeps running on the host between
        replays and writes the new rate into that tensor;
      * gradients are views into the flat bucket (no per-step allocation).
    Not supported in graph mode: world_size > 1 (see __init__), `skip_nonfinite` (needs a host decision) and Python-side
    regularisers that branch on data.  Outputs are static tensors that the next replay overwrites.  A label mask, row
    weights and label weights (`step(..., label_mask=, row_weight=, pos_weight=, neg_weight=)`) go into static buffers
    as well; each combination of the ones given is a capture of its own."""

    def __init__(self, stepper: DataParallelStep, warmup: int = 3):
        if stepper.skip_nonfinite:
            raise ValueError("GraphedTrainStep cannot skip non-finite steps (host decision); use DataParallelStep")
        if stepper.world > 1 and stepper.pbucket is None:
            # Capturing NCCL all-reduces hangs on this stack (torch 2.11 / NCCL 2.28.9, 2 x B200): in round 1 with the
            # early all-reduce issued from the autograd hook thread, and again in round 2 with every collective issued
            # inline from the capturing thread on the capture stream (10 min until the test's timeout,
            # profiles/r02_graph_multi_gpu.md).  So under N ranks the graph step needs the NCCL-free exchange:
            # DataParallelStep(..., peer_all=True) keeps the gradient bucket in peer-mapped memory and sums it with the
            # library's own kernel, whose flag values come from a device counter during replay.
            raise NotImplementedError("GraphedTrainStep under torch.distributed needs DataParallelStep(peer_all=True) "
                                      "(NCCL collectives cannot be captured on this stack)")
        self.stepper = stepper
        self.warmup = warmup
        self.graphs = {}
        dev = next(stepper.model.parameters()).device
        self.device = dev
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)      # Philox offset, bumped inside the graph
        stepper.args.noise_offset_tensor = self.counter
        stepper.args.noise_offset_auto = False
        stepper.args.noise_offset = 0
        from .optim import FusedAdam
        for group in stepper.optimizer.param_groups:
            if "capturable" in group and not group["capturable"]:
                raise ValueError("construct the optimizer with capturable=True for graph capture")
            if isinstance(stepper.optimizer, FusedAdam) and not (isinstance(group["lr"], torch.Tensor) and group["lr"].is_cuda):
                # a Python float would be baked into the captured launch; StepLR writes into the tensor between replays
                raise ValueError("FusedAdam under graph capture needs lr as a CUDA tensor: lr=torch.tensor(1e-3, device=...)")

    # -- warm-up runs on a snapshot: the first step() must be exactly ONE update, like the reference loop ----------
    def _snapshot(self):
        from .optim import FusedAdam
        st, opt = self.stepper, self.stepper.optimizer
        if isinstance(opt, FusedAdam) and opt._segments is None:
            opt._build()                                                  # flat buffers first: p.data become views of them
        snap = {"params": [p.detach().clone() for p in st.model.parameters()],
                "r_shadow": None if st.r_shadow is None else st.r_shadow.detach().clone(),
                "step_no": st.step_no, "shadow_fresh": st._shadow_fresh, "counter": self.counter.clone(),
                "rng_cuda": torch.cuda.get_rng_state(self.device), "rng_cpu": torch.get_rng_state()}
        if isinstance(opt, FusedAdam):
            snap["fused"] = ([(seg.flat_m.clone(), seg.flat_v.clone()) for seg in opt._segments], opt._scal.clone())
        else:
            snap["opt"] = {p: {k: (v.clone() if torch.is_tensor(v) else v) for k, v in s.items()} for p, s in opt.state.items()}
        return snap

    @torch.no_grad()
    def _restore(self, snap):
        from .optim import FusedAdam
        st, opt = self.stepper, self.stepper.optimizer
        for p, saved in zip(st.model.parameters(), snap["params"]):
            p.data.copy_(saved)
        if snap["r_shadow"] is not None:
            st.r_shadow.copy_(snap["r_shadow"])
        st.step_no, st._shadow_fresh = snap["step_no"], snap["shadow_fresh"]
        self.counter.copy_(snap["counter"])
        torch.cuda.set_rng_state(snap["rng_cuda"], self.device)
        torch.set_rng_state(snap["rng_cpu"])
        if isinstance(opt, FusedAdam):
            for seg, (m, v) in zip(opt._segments, snap["fused"][0]):
                seg.flat_m.copy_(m); seg.flat_v.copy_(v)
            opt._scal.copy_(snap["fused"][1])
        else:
            # in place: the captured graph holds the addresses of the state tensors the warm-up created
            for p, s in opt.state.items():
                old = snap["opt"].get(p)
                for k, v in s.items():
                    if torch.is_tensor(v):
                        if old is not None and k in old:
                            v.copy_(old[k])
                        else:
                            v.zero_()                                     # state born during the warm-up: back to "fresh"

    def _capture(self, y, x, extra):
        static_y, static_x = y.clone(), x.clone()
        static_extra = {k: v.clone() for k, v in extra.items()}
        st = self.stepper
        if st.world > 1:
            st.pbucket.enable_graph_replay()
            if st._want_ring:
                ring = st._peer_ring(y.shape[0])
                if ring is not None:
                    ring.enable_graph_replay()
        snap = self._snapshot()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):                                  # also initialises optimizer state
                self._body(static_y, static_x, static_extra)
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = self._body(static_y, static_x, static_extra)
        self._restore(snap)                                               # parameters, moments, counters, RNG: as before
        return {"graph": graph, "y": static_y, "x": static_x, "extra": static_extra, "out": out}

    def _body(self, y, x, extra):
        st = self.stepper
        sched, st.scheduler = st.scheduler, None                          # the scheduler is stepped on the host
        try:
            out = st.step(y, x, **extra)
        finally:
            st.scheduler = sched
        self.counter.add_(1)
        return out

    def step(self, input_label: torch.Tensor, input_feat: torch.Tensor, row_weight: Optional[torch.Tensor] = None,
             label_mask: Optional[torch.Tensor] = None, pos_weight: Optional[torch.Tensor] = None,
             neg_weight: Optional[torch.Tensor] = None) -> StepOutput:
        from .probit import _check_label_mask, _check_label_weight, _check_row_weight
        B, L = input_label.shape
        extra = {}
        if label_mask is not None:
            extra["label_mask"] = _check_label_mask(label_mask, B, L, self.device)
        if row_weight is not None:
            extra["row_weight"] = _check_row_weight(row_weight, B, self.device)
        _check_label_weight(pos_weight, neg_weight, L, self.device)
        for name, w in (("pos_weight", pos_weight), ("neg_weight", neg_weight)):
            if w is not None:
                extra[name] = w.to(torch.float32)
        key = (tuple(input_label.shape), tuple(input_feat.shape), tuple(sorted(extra)))
        entry = self.graphs.get(key)
        if entry is None:
            entry = self.graphs[key] = self._capture(input_label, input_feat, extra)   # warm-up on a snapshot
        entry["y"].copy_(input_label)
        entry["x"].copy_(input_feat)
        for k, v in extra.items():
            entry["extra"][k].copy_(v)
        entry["graph"].replay()
        if self.stepper.scheduler is not None:
            self.stepper.scheduler.step()
        return entry["out"]


def pack_labels(y) -> torch.Tensor:
    """{0,1} label matrix (B, L) -> bits, (B, ceil(L/8)) uint8, label l in bit l % 8 of byte l // 8.  Labels are what the
    loader keeps on the HOST for the whole run (train.py:106-111 slices them per batch); as bits they cross PCIe at 1/32
    of the fp32 size and are packed once per data set, not per step."""
    import numpy as np
    a = y.cpu().numpy() if torch.is_tensor(y) else np.asarray(y)
    if not np.isin(a, (0, 1)).all():
        raise ValueError("pack_labels: the label matrix must hold only 0 and 1")
    return torch.from_numpy(np.packbits(a.astype(np.uint8), axis=1, bitorder="little"))


def unpack_labels(bits: torch.Tensor, n_labels: int) -> torch.Tensor:
    """Inverse of `pack_labels` on the tensor's device: (B, ceil(L/8)) uint8 -> (B, L) float32."""
    shifts = torch.arange(8, device=bits.device, dtype=torch.uint8)
    y = torch.bitwise_and(torch.bitwise_right_shift(bits.unsqueeze(-1), shifts), 1)
    return y.reshape(bits.shape[0], -1)[:, :n_labels].float()


class HostBatchPrefetcher:
    """Double-buffered host -> device staging of a step's inputs (SURVEY 8f-N4: train.py:106-111 does a blocking
    `torch.from_numpy(...).to(device)` per step).  Batches are copied from PINNED host tensors on a side stream into
    one of `depth` device slots while the previous step computes; `next()` makes the compute stream wait for the
    copy and hands out the slot, whose reuse in turn waits for that step's compute to finish."""

    def __init__(self, device, depth: int = 2):
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self.depth = depth
        self.slots = [None] * depth
        self.ready = [None] * depth        # copy finished (recorded on the side stream)
        self.free = [None] * depth         # compute finished with the slot (recorded on the compute stream)
        self.head = self.tail = 0          # next slot to fill / to hand out

    def push(self, host_batch: dict):
        """Start copying `host_batch` (name -> pinned CPU tensor).  At most `depth` batches may be in flight."""
        i = self.head % self.depth
        if self.slots[i] is None:
            self.slots[i] = {k: torch.empty(v.shape, dtype=v.dtype, device=self.device) for k, v in host_batch.items()}
        if self.free[i] is not None:
            self.stream.wait_event(self.free[i])
        with torch.cuda.stream(self.stream):
            for k, v in host_batch.items():
                self.slots[i][k].copy_(v, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self.ready[i] = ev
        self.head += 1

    def next(self) -> dict:
        """The oldest staged batch as device tensors; valid until `depth` more batches have been pushed."""
        assert self.tail < self.head, "nothing staged"
        i = self.tail % self.depth
        torch.cuda.current_stream(self.device).wait_event(self.ready[i])
        self.tail += 1
        self._last = i
        return self.slots[i]

    def release(self):
        """Call after the step that consumed the last `next()` has been enqueued: lets the slot be refilled."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self.free[self._last] = ev
