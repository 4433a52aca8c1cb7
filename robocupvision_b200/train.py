"""Fused train / eval steps: the reference's per-batch loop bodies as device-resident pipelines.

``TrainStep`` restates train.py:43-74 (zero_grad -> model(imgs) -> CrossEntropyLoss2d ->
+ decay*l1reg -> backward -> [pruned-grad mask] -> Adam.step -> argmax / correct pixels):
all parameters live in one flat fp32 arena (state_dict keys and nn.Parameter objects are
unchanged: each ``p.data`` becomes a view), gradients in a second arena, so the L1 sub-gradient,
the pruning mask and Adam are one kernel, and the data-parallel exchange is one or two NCCL
all-reduces of arena slices issued while backward is still running.  The whole step is
captured into a CUDA graph (no host syncs: the reference's three ``.item()`` reads per step
become device scalars the caller reads when it wants them).

``EvalStep`` restates train.py:114-153 (forward, loss, argmax, per-image confusion, IoU) with
no host round trips.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import dp, ops
from .engine import Plan


def _zeros(n, dtype, device) -> torch.Tensor:
    """Zero-filled state buffer: a stream-ordered memset on the GPU (no fill kernel); plain torch on the CPU, where only
    the host-side meters of the gloo tests live."""
    if torch.device(device).type == "cuda":
        return ops.zeros(n, dtype, device)
    return torch.zeros(n, dtype=dtype, device=device)


# diagnostic only (tools/ngpu_ab.sh): ranks run the data-parallel schedule WITHOUT exchanging gradients, which
# separates the cost of the lock-step from everything else that differs between one process and N
_SKIP_EXCHANGE = os.environ.get("RCV_B200_DP_SKIP_EXCHANGE", "") == "1"

_FUSED_HEAD = os.environ.get("RCV_B200_FUSED_HEAD", "1") != "0"

ARENA_ALIGN = 4  # floats: every parameter's slice starts on a 16-byte boundary (vector loads, TMA, no clones in ops._chk)


def flatten_parameters(model: nn.Module):
    """Move every parameter into one flat fp32 arena (order = model.parameters()); returns
    (arena, [(param, offset, numel)]).  Offsets are padded to multiples of ARENA_ALIGN floats; the padding stays
    zero under every optimiser of this module (zero gradient, sign(0) = 0, zero moments)."""
    params = list(model.parameters())
    dev = params[0].device
    offs, o = [], 0
    for p in params:
        offs.append(o)
        o += -(-p.numel() // ARENA_ALIGN) * ARENA_ALIGN
    arena = _zeros(o, torch.float32, dev)
    table = []
    for p, o in zip(params, offs):
        n = p.numel()
        arena[o:o + n].copy_(p.data.reshape(-1))
        p.data = arena[o:o + n].view(p.shape)
        table.append((p, o, n))
    return arena, table


def sync_bn_buffers(model: nn.Module, src: int = 0, group=None, average: bool = False) -> None:
    """Data-parallel training keeps BatchNorm running statistics rank-local (the reference has no SyncBN), so after
    training steps on different shards every rank holds slightly different eval-mode models.  Call this before a
    sharded validation pass and before writing a checkpoint: floating-point buffers are broadcast from rank `src`
    (or averaged over the group), integer buffers (num_batches_tracked) are broadcast.  No-op without a group."""
    dist = torch.distributed
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    ws = dist.get_world_size(group)
    for b in model.buffers():
        if average and b.is_floating_point():
            dist.all_reduce(b, group=group)
            b.div_(ws)
        else:
            dist.broadcast(b, src, group=group)
    plan = model.__dict__.get("_rcv_plan")
    if plan is not None:
        plan.epoch += 1  # folded-BatchNorm constants are cached per plan epoch


class TrainStep:
    def __init__(self, model: nn.Module, class_weights: Optional[Sequence[float]] = None, lr: float = 1e-3,
                 l1_decay: float = 1e-6, betas=(0.9, 0.999), eps: float = 1e-8,
                 masks: Optional[List[torch.Tensor]] = None, optimizer: str = "adam", momentum: float = 0.0,
                 weight_decay: float = 0.0, lr_mults: Optional[Sequence] = None,
                 process_group=None, use_graph: bool = True, overlap_comm: bool = True, n_buckets: int = 3,
                 force_comm_path: bool = False, reduce: Optional[str] = None,
                 fused_head: bool = _FUSED_HEAD, loss: str = "ce", dice_eps: float = 1e-7,
                 global_batch: bool = False):
        """masks: pruneModelNew-style list of bool tensors for the >1-D parameters, in parameter
        order (train.py:59-65); with masks the L1 term is dropped (train.py:53).
        optimizer: "adam" (train.py:357-363; torch defaults, no weight decay) or "sgd" (trainer.py:182-184:
        momentum, weight_decay, dampening 0; pass l1_decay=0 for the reference's SGD loop, which has no L1 term).
        lr_mults: [(module_or_param_list, multiplier)] for the reference's 10x group (train.py:357-363).
        n_buckets: data-parallel gradient buckets (cut at plan-node boundaries, dp.plan_buckets); each is
        all-reduced and its optimiser pass run on a side stream as soon as backward has passed its first node.
        force_comm_path: run the bucketed side-stream schedule even with one rank (tests).
        reduce: how the buckets are summed over ranks -- "peer": rcv_peer_allreduce, one kernel per bucket over the
        ranks' peer-mapped gradient arenas (peer.PeerExchange; the group is only used to exchange the IPC handles);
        "nccl": dist.all_reduce on the group.  Default: $RCV_B200_DP_REDUCE, else "peer" -- with dist.all_reduce taking
        over (with a warning, on every rank together) if the GPUs cannot map each other's memory.
        fused_head: run the classifier conv, the loss, the argmax and their backward as one kernel
        (ops.head_ce_train) where the plan ends in a bare 1x1 conv of 2..8 classes over 8 or 16 channels;
        otherwise (and with RCV_B200_FUSED_HEAD=0) the separate kernels run.
        loss: "ce" (CrossEntropyLoss2d, class_weights its weights) or "dice" (the reference's --useDice:
        DiceLoss(class_weights, dice_eps), the weights normalised to sum to the class count as DiceLoss does, all ones
        without class_weights).  Under "dice" the fused head is two kernels (ops.head_dice_fwd: the batch-wide sums
        and the correct count; ops.head_dice_train: the backward), the unfused head runs dice_fwd / dice_bwd on the
        logits.  The raw sums [intersection (C) | cardinality (C)] are kept in `dice_sums`, and the loss sums hold
        [dice loss, 1.0], so step(), loss_value() and step_async() read the Dice loss unchanged.  With N ranks the
        sums are rank-local and the gradients averaged: each rank's loss is the Dice loss of its own shard, the
        semantics DistributedDataParallel gives the reference's loop.
        The optimiser passes of the buckets run on the side stream with one rank too (overlap_comm): they overlap the
        encoder's backward (+0.5 % on the single-GPU step).
        global_batch: the N ranks, each holding B/N samples (the same shape on every rank), train ONE batch of B: what
        one process computes on all B samples, up to floating-point rounding -- BatchNorm batch statistics (summed
        over the ranks; the running variance's unbiased factor from the global count), BatchNorm backward, the CE
        normaliser sum(w[y]), the Dice sums, and the reported loss and correct count.  The small fp64 / int64 vectors
        are exchanged on the main stream in the middle of the step (rcv_peer_allreduce_f64 / _i64 over peer memory,
        dist.all_reduce under reduce="nccl"), and the gradients are summed over the ranks instead of averaged.
        Without it every rank's BatchNorm and loss see its own shard only (DistributedDataParallel's semantics).
        With one rank it changes nothing unless force_comm_path runs the exchanges (at world 1)."""
        if loss not in ("ce", "dice"):
            raise ValueError(f"TrainStep: loss must be 'ce' or 'dice', got {loss!r}")
        if optimizer not in ("adam", "sgd"):
            raise ValueError(f"TrainStep: optimizer must be 'adam' or 'sgd', got {optimizer!r}")
        if optimizer == "adam" and (weight_decay != 0.0 or momentum != 0.0):
            raise ValueError("TrainStep: optimizer='adam' is torch.optim.Adam with its defaults (train.py:357-363): "
                             "weight_decay and momentum must be 0 (they belong to optimizer='sgd')")
        asked = reduce or os.environ.get("RCV_B200_DP_REDUCE", "")
        if asked not in ("", "peer", "nccl"):
            raise ValueError(f"TrainStep: reduce must be 'peer' or 'nccl', got {asked!r}")
        self.model = model
        self.plan: Plan = model._get_plan()
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("TrainStep needs the model on a CUDA device (no CPU path)")
        self.dev = dev
        self.loss = loss
        self.dice_eps = float(dice_eps)
        if loss == "dice":
            if len(self.plan.outputs) != 1 or self.plan.nodes[self.plan.outputs[0] - 1].kind != "conv":
                raise ValueError("TrainStep(loss='dice'): the plan must end in one classifier conv")
            ncls = self.plan.nodes[self.plan.outputs[0] - 1].geom.cout
            w = torch.ones(ncls) if class_weights is None else torch.as_tensor(class_weights, dtype=torch.float32)
            if w.numel() != ncls:
                raise ValueError(f"TrainStep(loss='dice'): {w.numel()} class weights for {ncls} classes")
            class_weights = w / w.sum().item() * w.shape[0]  # DiceLoss.__init__
        self.class_w = None if class_weights is None else torch.as_tensor(
            class_weights, dtype=torch.float32).to(dev)
        # every small accumulator of a step in ONE buffer (one memset per step):
        # [l1 sum | CE loss sums (2) | correct pixels (int64 view) | BN batch statistics | BN backward sums]
        # loss="dice" appends [Dice sums (2C) | the unused loss sums of the correct-count pass of the unfused head (2)]
        # and keeps [dice loss, 1.0] where the CE loss sums are
        ns = self.plan.n_stats
        ndice = 2 * self.class_w.numel() + 2 if loss == "dice" else 0
        n_acc = 4 + 2 * ns + ndice
        self.arena, self.table = flatten_parameters(model)
        n = self.arena.numel()
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        force_comm_path = force_comm_path or os.environ.get("RCV_B200_FORCE_COMM_PATH", "") == "1"
        self.reduce = asked or "peer"
        self.peer = None
        self.grads = None
        if self.reduce == "peer" and (self.world > 1 or force_comm_path):
            from .peer import PeerExchange, PeerUnavailable
            try:
                # under global_batch the accumulators live in the peer-mapped block too, so the peers can read them
                self.peer = PeerExchange(n, dev, group=process_group, ndoubles=n_acc if global_batch else 0)
                self.grads = self.peer.grads
            except PeerUnavailable as e:  # raised on every rank or on none
                if asked == "peer":
                    raise
                import warnings
                warnings.warn(f"robocupvision_b200: peer-memory gradient exchange unavailable ({e}); "
                              "using dist.all_reduce", RuntimeWarning)
                self.reduce = "nccl"
        if self.world == 1 and self.peer is None:
            self.reduce = "none"
        # a global batch needs an exchange: none with one rank unless force_comm_path put the peer path in place
        self.global_batch = bool(global_batch) and self.reduce != "none"
        self._batch_reduce = _RankReduce(self) if self.global_batch else None
        self._shard_shape = None
        if self.grads is None:
            self.grads = _zeros(n, torch.float32, dev)
        if self.world > 1 and "RCV_PDL" not in os.environ:
            # programmatic dependent launch: measured -1.5 % with NCCL kernels inside the step's graph, neutral to
            # +0.8 % with the peer-memory exchange (2 x B200); single-process runs have it on from _lib.load()
            from . import _lib
            _lib.load().rcv_set_pdl(1 if self.peer is not None else 0)
        self.m = _zeros(n, torch.float32, dev)       # Adam exp_avg / SGD momentum buffer
        self.v = _zeros(n, torch.float32, dev) if optimizer == "adam" else None
        self.grad_views = {id(p): self.grads[o:o + k].view(p.shape) for p, o, k in self.table}
        self.offsets = {id(p): (o, k) for p, o, k in self.table}
        self.optimizer = optimizer
        self.betas, self.eps = betas, eps
        self.momentum, self.weight_decay = float(momentum), float(weight_decay)
        self.l1_decay = 0.0 if masks is not None else float(l1_decay)
        self.mask = None
        if masks is not None:
            self.mask = _zeros(n, torch.uint8, dev)
            i = 0
            for p, o, k in self.table:
                if p.dim() > 1:
                    self.mask[o:o + k] = masks[i].reshape(-1).to(dev).to(torch.uint8)
                    i += 1
        # lr groups: contiguous arena ranges (padding included) with a multiplier
        mult = torch.ones(len(self.table))
        if lr_mults:
            for group, mu in lr_mults:
                ps = list(group.parameters()) if isinstance(group, nn.Module) else list(group)
                ids = {id(p) for p in ps}
                for i, (p, _, _) in enumerate(self.table):
                    if id(p) in ids:
                        mult[i] = mu
        # Parameters no plan node owns (PB_FCN's unused patch-classification head) never receive a gradient: torch
        # leaves their .grad None and every optimiser skips them -- unless the L1 term (which sums over ALL
        # parameters, train.py:23-27) gives them one.  Without L1 they are left out of the optimiser ranges, so
        # SGD's weight decay does not touch them either.
        in_plan = {id(q) for q in self.plan.params}
        self.ranges = []  # (start, end, mult)
        ends = [o for _, o, _ in self.table[1:]] + [n]
        prev_end = None
        for (p, o, k), e, mu in zip(self.table, ends, mult.tolist()):
            if id(p) not in in_plan and self.l1_decay == 0.0:
                continue
            if self.ranges and self.ranges[-1][2] == mu and prev_end == o:
                self.ranges[-1] = (self.ranges[-1][0], e, mu)
            else:
                self.ranges.append((o, e, mu))
            prev_end = e
        self.base_lr = lr
        self._lr_host = torch.tensor([lr * r[2] for r in self.ranges], dtype=torch.float32).pin_memory()
        self.lr_dev = self._lr_host.to(dev)
        self.step_dev = _zeros(1, torch.int32, dev)
        self._accum = (self.peer.accum if self.global_batch and self.peer is not None
                       else _zeros(n_acc, torch.float64, dev))
        self._acc_l1, self._acc_ce = self._accum[0:1], self._accum[1:3]
        self._acc_corr = self._accum[3:4].view(torch.int64)
        self._acc_stats, self._acc_sums = self._accum[4:4 + ns], self._accum[4 + ns:4 + 2 * ns]
        self.dice_sums = self._accum[4 + 2 * ns:4 + 2 * ns + ndice - 2] if loss == "dice" else None
        self._acc_spare = self._accum[4 + 2 * ns + ndice - 2:] if loss == "dice" else None
        # distributed
        self.comm_path = overlap_comm or force_comm_path
        self.comm_stream = torch.cuda.Stream(device=dev) if self.comm_path else None
        # (first plan node, arena start, arena end), in the order backward completes them (arena tail first)
        self.buckets = dp.plan_buckets([[self.offsets[id(p)] for p in nd.params()] for nd in self.plan.nodes],
                                       [(o, k) for _, o, k in self.table], n, n_buckets) if self.comm_path else []
        if self.global_batch and self.peer is not None:
            from .peer import SMALL_SLOT
            if len(self.buckets) > SMALL_SLOT:
                raise ValueError(f"TrainStep(global_batch=True): at most {SMALL_SLOT} gradient buckets, "
                                 f"got {len(self.buckets)}")
        # the classifier head in one pass (ops.head_ce_train; two for Dice) where the plan ends in a bare 1x1 conv the
        # kernel covers
        self._head = self.plan.fusable_head() if fused_head else -1
        # outputs (device scalars)
        self.loss_sums = None
        self.l1_sum = None
        self.correct = None
        self.use_graph = use_graph
        self.graph = None
        self._graph_refs = []  # the plan's buffers self.graph bakes in (Plan.capture_refs): freed with the graph
        self.static_x = None
        self.static_y = None
        self.kernels_per_step = 0
        self._warm = 0
        self._pipe = None

    # ------------------------------------------------------------------ helpers
    def set_lr(self, lr: float):
        """Every group to lr * its multiplier (ReduceLROnPlateau-style schedulers, trainer.py:193)."""
        self.base_lr = lr
        self.set_group_lrs([lr * r[2] for r in self.ranges])

    def set_group_lrs(self, lrs: Sequence[float]):
        """One learning rate per arena range of `self.ranges` (= the reference's param groups, train.py:357-363),
        staged through pinned memory: the next replay of the step's graph reads them from the device."""
        if len(lrs) != len(self.ranges):
            raise ValueError(f"set_group_lrs: {len(self.ranges)} groups, got {len(lrs)} values")
        self._lr_host.copy_(torch.as_tensor(list(lrs), dtype=torch.float32))
        self.lr_dev.copy_(self._lr_host, non_blocking=True)

    def set_cosine_lr(self, epoch: int, t_max: int, eta_min: float = 0.0):
        """CosineAnnealingLR as train.py:364-365 / lr_scheduler.py apply it, stepped once per epoch: each group
        anneals from ITS OWN base rate (base_lr * multiplier) to the one shared eta_min:
        eta_min + (base_i - eta_min) * (1 + cos(pi * epoch / t_max)) / 2."""
        import math
        f = (1.0 + math.cos(math.pi * epoch / t_max)) / 2.0
        self.set_group_lrs([eta_min + (self.base_lr * r[2] - eta_min) * f for r in self.ranges])

    def _allreduce(self, a: int, b: int, slot: int = 0):
        """grads[a:b] <- sum over ranks, on the current stream."""
        if _SKIP_EXCHANGE:
            return
        if self.peer is not None:
            self.peer.allreduce(slot, a, b)
        elif self.world > 1 or self.pg is not None:
            torch.distributed.all_reduce(self.grads[a:b], group=self.pg)

    def _reduce_f64(self, t: torch.Tensor, scale: float = 1.0):
        """t (a float64 slice of the accumulator buffer) <- scale * sum over ranks, on the current stream."""
        if self.peer is not None:
            self.peer.allreduce_f64(t, scale)
        else:
            dist = torch.distributed
            dist.all_reduce(t, op=dist.ReduceOp.SUM if scale == 1.0 else dist.ReduceOp.AVG, group=self.pg)

    def _reduce_i64(self, t: torch.Tensor):
        """t (an int64 view of the accumulator buffer) <- sum over ranks, on the current stream."""
        if self.peer is not None:
            self.peer.allreduce_i64(t)
        else:
            torch.distributed.all_reduce(t, group=self.pg)

    def _optim_range(self, a: int, b: int, l1):
        """Optimiser pass over arena[a:b), split at the lr-group boundaries."""
        gscale = 1.0 if self.global_batch else 1.0 / self.world  # a global batch's gradient is the sum over ranks
        for i, (ra, rb, _) in enumerate(self.ranges):
            lo, hi = max(a, ra), min(b, rb)
            if lo >= hi:
                continue
            sl = slice(lo, hi)
            mk = None if self.mask is None else self.mask[sl]
            if self.optimizer == "adam":
                ops.adam_l1_step(self.arena[sl], self.grads[sl], self.m[sl], self.v[sl], lr=self.base_lr,
                                 beta1=self.betas[0], beta2=self.betas[1], eps=self.eps, step=0,
                                 l1_decay=self.l1_decay, grad_scale=gscale, mask=mk, l1_sum=l1,
                                 step_dev=self.step_dev, lr_dev=self.lr_dev[i:i + 1])
            else:
                # zero-initialised momentum buffer: mom*0 + g == torch's first-step `buf = g`, so no first-step flag
                ops.sgd_step(self.arena[sl], self.grads[sl], self.m[sl], lr=self.base_lr, momentum=self.momentum,
                             weight_decay=self.weight_decay, grad_scale=gscale, mask=mk, l1_decay=self.l1_decay,
                             l1_sum=l1, lr_dev=self.lr_dev[i:i + 1])

    # ------------------------------------------------------------------ the step
    def _step_impl(self, x, y):
        k0 = ops.launch_count()
        # two memsets (no kernels) for everything the step accumulates into: optimizer.zero_grad() (train.py:45)
        # and the scalar / per-channel sums
        ops.zero_(self.grads)
        ops.zero_(self._accum)
        l1 = self._acc_l1
        ops.counter_add(self.step_dev, 1)
        head = self._head
        seed = None
        gb = self._batch_reduce
        if head >= 0 and self.loss == "ce":
            # the normaliser of the weighted mean loss depends on the labels only: produced here, so that the head
            # needs ONE pass (classifier conv + loss + argmax + their backward, ops.head_ce_train)
            ops.ce_weight_sum(y, self.class_w, self._acc_ce[1:2], self.plan.nodes[head].geom.cout)
            if gb is not None:
                self._reduce_f64(self._acc_ce[1:2])  # the head divides by the global normaliser
        outs, saved = self.plan.forward(x, training=True, save=True, stats_arena=self._acc_stats,
                                        stop_before=head if head >= 0 else None, batch_reduce=gb)
        if head >= 0 and saved[2].get(self.plan.nodes[head].src) is not None:
            raise RuntimeError("TrainStep: the classifier reads a BatchNorm that was deferred to its consumer")
        sums, corr = self._acc_ce, self._acc_corr
        if self.loss == "dice":
            seed, gouts = self._dice_head(outs, saved, y)
        elif head >= 0:
            nd = self.plan.nodes[head]
            dfeat = ops.head_ce_train(saved[0][nd.src], nd.conv.weight.detach(),
                                      None if nd.conv.bias is None else nd.conv.bias.detach(), y, self.class_w, sums,
                                      corr, self.grad_views[id(nd.conv.weight)],
                                      None if nd.conv.bias is None else self.grad_views[id(nd.conv.bias)])
            seed, gouts = {nd.src: dfeat}, [None]
        else:
            logits = outs[0]
            sums, _, _, corr = ops.ce_fwd(logits, y, self.class_w, want_correct=True, sums=self._acc_ce,
                                          corr=self._acc_corr)
            if gb is not None:
                self._reduce_f64(self._acc_ce)  # ce_bwd divides by the global normaliser
            gouts = [ops.ce_bwd(logits, y, self.class_w, sums)]
        if self.comm_path:
            cur = torch.cuda.current_stream()
            pending = [(k,) + tuple(bk) for k, bk in enumerate(self.buckets)]

            def flush(upto):
                """All-reduce + optimiser pass, on the comm stream, of every bucket whose gradients are final once
                backward has passed node `upto` (their weights are read by no later backward kernel)."""
                while pending and pending[0][1] >= upto:
                    k, _, a, b = pending.pop(0)
                    self.comm_stream.wait_stream(cur)
                    if self.plan._wgrad_stream is not None:  # weight gradients are produced on the side stream
                        self.comm_stream.wait_stream(self.plan._wgrad_stream)
                    with torch.cuda.stream(self.comm_stream):
                        self._allreduce(a, b, slot=k)
                        self._optim_range(a, b, l1)
            self.plan.backward(saved, gouts, False, self.grad_views, node_done=flush, sums_arena=self._acc_sums,
                               seed=seed, batch_reduce=gb)
            flush(-1)
            cur.wait_stream(self.comm_stream)
        else:
            self.plan.backward(saved, gouts, False, self.grad_views, sums_arena=self._acc_sums, seed=seed,
                               batch_reduce=gb)
            if self.world > 1:
                self._allreduce(0, self.arena.numel())
            self._optim_range(0, self.arena.numel(), l1)
        if gb is not None:
            # the reported loss and correct count of the global batch (the other loss paths reduced theirs already)
            if self.loss == "ce" and head >= 0:
                self._reduce_f64(self._acc_ce[0:1])
            self._reduce_i64(self._acc_corr)
        self.kernels_per_step = ops.launch_count() - k0
        return sums, l1, corr

    def _dice_head(self, outs, saved, y):
        """The Dice loss, its gradient seed for Plan.backward and the correct count: (seed, gouts)."""
        eps, w = self.dice_eps, self.class_w
        if self._head >= 0:
            nd = self.plan.nodes[self._head]
            feat, wt = saved[0][nd.src], nd.conv.weight.detach()
            bias = None if nd.conv.bias is None else nd.conv.bias.detach()
            ops.head_dice_fwd(feat, wt, bias, y, self.dice_sums, self._acc_corr)
            if self._batch_reduce is not None:
                self._reduce_f64(self.dice_sums)
            dfeat = ops.head_dice_train(feat, wt, bias, y, w, self.dice_sums, eps, self._acc_ce,
                                        self.grad_views[id(nd.conv.weight)],
                                        None if nd.conv.bias is None else self.grad_views[id(nd.conv.bias)])
            return {nd.src: dfeat}, [None]
        logits = outs[0]
        ops.dice_fwd(logits, y, sums=self.dice_sums)
        if self._batch_reduce is not None:
            self._reduce_f64(self.dice_sums)
        ops.ce_fwd(logits, y, None, want_correct=True, sums=self._acc_spare, corr=self._acc_corr)
        ops.dice_loss(self.dice_sums, w, eps, self._acc_ce)
        return None, [ops.dice_bwd(logits, y, w, self.dice_sums, eps)]

    def step(self, x: torch.Tensor, y: torch.Tensor):
        """One training step on x [B,Cin,H,W] fp32, y [B,H,W] int64 (device tensors, or pinned
        host tensors which are copied H2D straight into the step's static input buffers).
        Returns (loss_sums float64[2], l1_sum float64[1], correct int64[1]) device tensors:
        CE loss = loss_sums[0]/loss_sums[1] (the Dice loss under loss="dice", loss_sums[1] = 1);
        total = CE + l1_decay*l1_sum."""
        self.model.train()
        self.plan.epoch += 1  # parameters / BN buffers change under raw kernels (also on graph replay)
        if self.global_batch and self.world > 1 and self._shard_shape != (tuple(x.shape), tuple(y.shape)):
            check_equal_shards(x, y, self.pg)  # once per input shape: before a capture, or eagerly
            self._shard_shape = (tuple(x.shape), tuple(y.shape))
        if not self.use_graph:
            x = x.to(self.dev, non_blocking=True)
            y = y.to(self.dev, non_blocking=True)
            self.loss_sums, self.l1_sum, self.correct = self._step_impl(x, y)
            self.plan.epoch += 1  # the optimiser wrote the weights after the step's panels were packed
            return self.loss_sums, self.l1_sum, self.correct
        if self.graph is None or self.static_x.shape != x.shape:
            self._capture(x, y)
        else:
            self.static_x.copy_(x, non_blocking=True)
            self.static_y.copy_(y, non_blocking=True)
            self.graph.replay()
        # the optimiser wrote the weights AFTER this step's tensor-core panels were packed: an eval-mode forward
        # that follows must not reuse them (packed-panel / folded-BN caches are keyed on the plan epoch)
        self.plan.epoch += 1
        return self.loss_sums, self.l1_sum, self.correct

    def step_async(self, x: torch.Tensor, y: torch.Tensor) -> "StepResult":
        """Pipelined form of step() for a loop fed from pinned host memory: this step's inputs go
        H2D on a copy stream into one of two staging buffers (overlapping the previous step, which
        is still running), the main stream waits for them, moves them into the graph's input
        buffers device-to-device and replays; the step's scalars (L1 sum, loss sums, correct count: the 32-byte head
        of the accumulator buffer) follow in ONE copy to pinned host memory.  Returns a handle whose wait() blocks until
        THIS step's scalars have landed -- call it one step late to keep the pipe full.
        (A second capture of the step over the staging buffers themselves would save the device-to-device copy,
        ~10 us; tried, and dropped after one unexplained failure of test_step_async_matches_step in three runs.)"""
        if self.graph is None or self.static_x.shape != x.shape or not self.use_graph or x.is_cuda:
            self.step(x, y)
            return StepResult.ready(self)
        self.model.train()
        self.plan.epoch += 1
        if self._pipe is None:
            self._pipe = _HostPipe(self.static_x, self.static_y, self.dev)
        pipe = self._pipe
        k = pipe.next_slot()
        cur = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(pipe.copy_stream):
            pipe.copy_stream.wait_event(pipe.free[k])      # the D2D that last read this slot is done
            pipe.sx[k].copy_(x, non_blocking=True)
            pipe.sy[k].copy_(y, non_blocking=True)
            pipe.loaded[k].record(pipe.copy_stream)
        cur.wait_event(pipe.loaded[k])
        self.static_x.copy_(pipe.sx[k], non_blocking=True)
        self.static_y.copy_(pipe.sy[k], non_blocking=True)
        pipe.free[k].record(cur)
        self.graph.replay()
        pipe.out[k].copy_(self._accum[:4], non_blocking=True)
        pipe.done[k].record(cur)
        self.plan.epoch += 1  # as in step(): the weights changed after the panels were packed
        return StepResult(pipe, k, self.l1_decay)

    def _state(self):
        return [t for t in (self.arena, self.m, self.v, self.step_dev) if t is not None] + list(self.model.buffers())

    def _capture(self, x, y):
        """First call for a shape: one eager warm-up step on a side stream (lazy CUDA module
        loading / attribute setting must not happen inside capture), state restored, the step
        captured, then replayed once -- so this call still performs exactly one step."""
        self.static_x = x.to(self.dev, copy=True)
        self.static_y = y.to(self.dev, copy=True)
        snap = [t.clone() for t in self._state()]
        cur = torch.cuda.current_stream()
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(cur)
        with torch.cuda.stream(s):
            self._step_impl(self.static_x, self.static_y)
        cur.wait_stream(s)
        torch.cuda.synchronize(self.dev)
        for t, t0 in zip(self._state(), snap):
            t.copy_(t0)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.loss_sums, self.l1_sum, self.correct = self._step_impl(self.static_x, self.static_y)
        self.graph = g
        self._graph_refs = self.plan.capture_refs()
        self._pipe = None  # the staging slots have the old shape
        g.replay()

    def broadcast_state(self, src: int = 0):
        """Make every rank start from rank `src`'s parameters and BatchNorm buffers."""
        if self.world > 1:
            for t in [self.arena] + [b for b in self.model.buffers() if b.is_floating_point()]:
                torch.distributed.broadcast(t, src, group=self.pg)

    def loss_value(self) -> float:
        """Host read (one sync) of the last step's total loss, as train.py:73 accumulates it."""
        num, den = self.loss_sums.tolist()
        if self.peer is not None:
            self.peer.check()
        return num / den + self.l1_decay * float(self.l1_sum)


class _RankReduce:
    """Plan.forward / Plan.backward's `batch_reduce` of a global-batch TrainStep: in-place sums and means over the
    ranks of float64 slices of the step's accumulator buffer, on the current stream."""

    def __init__(self, ts: TrainStep):
        self.world = ts.world
        self._ts = ts

    def sum(self, buf: torch.Tensor) -> None:
        self._ts._reduce_f64(buf)

    def mean(self, buf: torch.Tensor) -> None:
        self._ts._reduce_f64(buf, 1.0 / self.world)


def check_equal_shards(x: torch.Tensor, y: torch.Tensor, group=None) -> None:
    """A global batch divides by world * (this rank's count) and averages the BatchNorm backward sums, which is right
    only if every rank holds as many samples of the same size: compare the input shapes of all ranks (one
    all_gather_object; collective) and raise ValueError on every rank if they differ."""
    dist = torch.distributed
    mine = (tuple(x.shape), tuple(y.shape))
    every = [None] * dist.get_world_size(group)
    dist.all_gather_object(every, mine, group=group)
    if any(e != every[0] for e in every):
        raise ValueError(f"TrainStep(global_batch=True): every rank must hold the same shard shape, got "
                         f"(x, y) shapes {every}")


class _HostPipe:
    """Two staging slots (device inputs + pinned host outputs) and the events that order them."""

    def __init__(self, like_x, like_y, dev):
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.sx = [torch.empty_like(like_x) for _ in range(2)]
        self.sy = [torch.empty_like(like_y) for _ in range(2)]
        # [l1 sum | CE loss sums (2) | correct pixels (int64 bits)]: the head of TrainStep._accum
        self.out = [torch.empty(4, dtype=torch.float64).pin_memory() for _ in range(2)]
        self.out_f = self.out  # EvalStep.run_async: [loss | - | - | -] and the correct count beside it
        self.out_i = [torch.empty(1, dtype=torch.int64).pin_memory() for _ in range(2)]
        self.loaded = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.done = [torch.cuda.Event() for _ in range(2)]
        cur = torch.cuda.current_stream(dev)
        for e in self.free:
            e.record(cur)
        self.k = 1

    def next_slot(self) -> int:
        self.k ^= 1
        return self.k


class StepResult:
    """Host-side view of one pipelined step's scalars (TrainStep.step_async)."""

    def __init__(self, pipe, k, l1_decay):
        self.pipe, self.k, self.l1_decay, self._ts = pipe, k, l1_decay, None

    @staticmethod
    def ready(ts):
        """Result of a step that ran through step() (first call / device inputs): read now, the
        device scalars are overwritten by the next replay."""
        r = StepResult(None, 0, ts.l1_decay)
        num, den = ts.loss_sums.tolist()
        ce = num / den
        r._ts = (ce, ce + ts.l1_decay * float(ts.l1_sum), int(ts.correct))
        return r

    def wait(self):
        """-> (ce_loss, total_loss, correct) of that step, after its D2H copy has completed."""
        if self._ts is not None:
            return self._ts
        self.pipe.done[self.k].synchronize()
        f = self.pipe.out[self.k]
        ce = float(f[1]) / float(f[2])
        return ce, ce + self.l1_decay * float(f[0]), int(f.view(torch.int64)[3])


class EvalStep:
    """Validation batch (train.py:114-153): logits, weighted CE, argmax, correct-pixel count,
    per-image confusion and IoU sums -- no host syncs (the reference does 3+25*B `.item()`s)."""

    def __init__(self, model: nn.Module, class_weights=None, use_graph: bool = False):
        """use_graph: replay the batch from a CUDA graph (one capture per input shape and per state of
        the model's parameters / buffers).  The returned tensors are then the graph's static buffers:
        valid until the next call with the same shapes."""
        self.model = model
        dev = next(model.parameters()).device
        self.class_w = None if class_weights is None else torch.as_tensor(
            class_weights, dtype=torch.float32).to(dev)
        self._pipe = None
        self.use_graph = use_graph
        self._graphs = {}

    @torch.no_grad()
    def run_async(self, x_host, y_host):
        """Pipelined validation batch fed from pinned host memory: H2D on a copy stream into one of
        two staging slots (overlapping the previous batch's kernels), then __call__ on the slot."""
        dev = next(self.model.parameters()).device
        if self._pipe is None or self._pipe.sx[0].shape != x_host.shape:
            self._pipe = _HostPipe(torch.empty(x_host.shape, device=dev, dtype=x_host.dtype),
                                   torch.empty(y_host.shape, device=dev, dtype=y_host.dtype), dev)
        pipe = self._pipe
        k = pipe.next_slot()
        cur = torch.cuda.current_stream(dev)
        with torch.cuda.stream(pipe.copy_stream):
            pipe.copy_stream.wait_event(pipe.free[k])
            pipe.sx[k].copy_(x_host, non_blocking=True)
            pipe.sy[k].copy_(y_host, non_blocking=True)
            pipe.loaded[k].record(pipe.copy_stream)
        cur.wait_event(pipe.loaded[k])
        out = self(pipe.sx[k], pipe.sy[k])
        pipe.free[k].record(cur)
        pipe.out_f[k][:1].copy_(out["loss"].reshape(1), non_blocking=True)
        pipe.out_i[k].copy_(out["correct"], non_blocking=True)
        pipe.done[k].record(cur)
        out["host"] = (pipe, k)
        return out

    @staticmethod
    def wait_host(out):
        """-> (loss, correct) of a run_async batch once its D2H copy has completed."""
        pipe, k = out["host"]
        pipe.done[k].synchronize()
        return float(pipe.out_f[k][0]), int(pipe.out_i[k])

    @torch.no_grad()
    def _eager(self, x, y):
        was_training = self.model.training
        self.model.eval()
        try:
            logits = self.model(x)
        finally:
            self.model.train(was_training)
        sums, am, conf, corr = ops.ce_fwd(logits, y, self.class_w, want_argmax=True, want_conf=True,
                                          want_correct=True)
        iou, loss = ops.metric_tail(conf, sums)
        return {"logits": logits, "loss": loss, "argmax": am, "conf": conf, "correct": corr, "iou_sum": iou}

    def _state_key(self):
        """Anything a captured forward bakes in: folded BatchNorm constants and packed weight panels are
        cached per (tensor, version), so a graph is only valid while no parameter / buffer was written."""
        ts = list(self.model.parameters()) + list(self.model.buffers())
        plan = self.model._get_plan() if hasattr(self.model, "_get_plan") else None
        return (tuple((t.data_ptr(), t._version) for t in ts), plan.epoch if plan is not None else 0)

    @torch.no_grad()
    def __call__(self, x, y):
        if not self.use_graph:
            return self._eager(x, y)
        key = (tuple(x.shape), tuple(y.shape))
        ent = self._graphs.get(key)
        state = self._state_key()
        if ent is None or ent["state"] != state:
            sx, sy = torch.empty_like(x), torch.empty_like(y)
            sx.copy_(x)
            sy.copy_(y)
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):  # warm-up outside capture: lazy module loading, caches, packs
                self._eager(sx, sy)
            cur.wait_stream(side)
            torch.cuda.synchronize(x.device)
            g = torch.cuda.CUDAGraph()
            k0 = ops.launch_count()
            with torch.cuda.graph(g):
                out = self._eager(sx, sy)
            self.kernels_per_call = ops.launch_count() - k0  # rcv_* kernels one replay launches
            plan = self.model._get_plan() if hasattr(self.model, "_get_plan") else None
            # the plan's buffers the graph bakes in stay alive while the graph does, whatever sizes run in between
            refs = plan.capture_refs() if plan is not None else []
            ent = {"graph": g, "sx": sx, "sy": sy, "out": out, "state": self._state_key(), "refs": refs}
            self._graphs[key] = ent
        ent["sx"].copy_(x, non_blocking=True)
        ent["sy"].copy_(y, non_blocking=True)
        ent["graph"].replay()
        return dict(ent["out"])


def iou_sums(conf: torch.Tensor) -> torch.Tensor:
    """Sum over images of per-class IoU from per-image confusion [N,C,C] with the reference's
    union==0 -> 1 rule (train.py:148-153): union_c = row_c + col_c - conf[c,c]."""
    if conf.is_cuda:
        return ops.metric_tail(conf)[0]
    confd = conf.to(torch.float64)
    inter = torch.diagonal(confd, dim1=1, dim2=2)
    union = confd.sum(2) + confd.sum(1) - inter
    iou = torch.where(union == 0, torch.ones_like(inter), inter / union.clamp(min=1))
    return iou.sum(0)


class ValidationMeter:
    """Epoch sums of a validation pass and the reference's summary (train.py:104-178): every batch adds its
    per-image confusion counts, IoU sums, correct-pixel count and loss on the device (no host syncs; the reference
    does 3 + 25*B `.item()` reads per batch), and `summary()` reduces them over the data-parallel group once
    (one int64 and one float64 all-reduce: validation shards over independent images, SURVEY.md section 8e) and
    returns pixel accuracy, the column-normalised confusion matrix in percent, mean class accuracy, mean IoU and
    the model-selection score (meanClassAcc + meanIoU) / 2 exactly as train.py:157-164 computes them."""

    def __init__(self, num_classes: int, device, process_group=None):
        self.nc = num_classes
        self.pg = process_group
        # [conf (nc*nc) | correct | images | pixels | batches]
        self.ints = _zeros(num_classes * num_classes + 4, torch.int64, device)
        # [iou_sum (nc) | loss sum]
        self.flts = _zeros(num_classes + 1, torch.float64, device)

    @torch.no_grad()
    def update(self, out: dict, extra_loss=None) -> None:
        """`out` = EvalStep.__call__ result of one batch; extra_loss (device scalar or float) is added to the
        batch loss (train.py:121-124 adds the L1 term when not fine-tuning)."""
        conf = out["conf"]
        nc2 = self.nc * self.nc
        self.ints[:nc2] += conf.sum(0).reshape(-1)
        self.ints[nc2] += out["correct"].reshape(())
        self.ints[nc2 + 1] += conf.shape[0]
        self.ints[nc2 + 2] += out["argmax"].numel()
        self.ints[nc2 + 3] += 1
        self.flts[:self.nc] += out["iou_sum"]
        loss = out["loss"].to(torch.float64)
        if extra_loss is not None:
            loss = loss + extra_loss
        self.flts[self.nc] += loss.reshape(())

    def summary(self) -> dict:
        ints, flts = self.ints.clone(), self.flts.clone()
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            ws = torch.distributed.get_world_size(self.pg)
            if ws > 1:
                torch.distributed.all_reduce(ints, group=self.pg)
                torch.distributed.all_reduce(flts, group=self.pg)
        nc, nc2 = self.nc, self.nc * self.nc
        ints_h, flts_h = ints.cpu(), flts.cpu()  # the one host read of the pass
        conf = ints_h[:nc2].reshape(nc, nc).to(torch.float64)
        correct, imgs, pixels, batches = (int(v) for v in ints_h[nc2:nc2 + 4])
        lab_cnts = conf.sum(0)                                   # train.py:143 labCnts (per label = column sums)
        conf_pct = conf / (lab_cnts.view(1, -1) / 100.0)         # train.py:158-160
        mean_class_acc = float(torch.diagonal(conf_pct).sum()) / nc   # train.py:163-164
        mean_iou = float((flts_h[:nc] / max(imgs, 1)).sum()) / nc * 100  # train.py:162
        return {"pixel_acc": 100.0 * correct / max(pixels, 1),  # train.py:129 running_acc*outSize*100 / imgCnt
                "conf_pct": conf_pct, "conf": ints_h[:nc2].reshape(nc, nc), "mean_class_acc": mean_class_acc,
                "mean_iou": mean_iou, "score": (mean_class_acc + mean_iou) / 2, "images": imgs,
                "loss": float(flts_h[nc]) / max(batches, 1)}   # train.py:172 losstotal / len(valloader)
