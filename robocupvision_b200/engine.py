"""Execution plan for the encoder-decoder nets: a flat list of fused nodes built from the
``model.py``-compatible module tree, with a hand-scheduled forward and backward.

Each conv-type node is  conv [+bias] -> (ReLU, BatchNorm) in the block's order -> [+ skip]
and runs as:
  eval : 1 kernel  (implicit-GEMM conv with bias/ReLU/folded-BN/skip in the epilogue)
  train: conv (+bias, +ReLU for the `Conv` order, + per-channel sum / sum^2 in the epilogue)
         -> bn_finalize (tiny) -> bn_apply (scale/shift [+ReLU] [+skip])
  bwd  : bn_bwd_reduce -> bn_bwd_apply (-> dconv, dgamma, dbeta, dbias) -> dgrad (+ skip
         gradient summed in its epilogue) -> wgrad (split over pixels, RED atomics)
The autograd boundary is one ``torch.autograd.Function`` for the whole plan; parameter
gradients are views of one zero-filled flat buffer (or of the caller's arena).
"""
from __future__ import annotations

import warnings

from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import ops
from .ops import (EPI_AFFINE_RELU, EPI_NONE, EPI_RELU, EPI_RELU_AFFINE, MATH_AUTO, MATH_BF16, MATH_FP32, MATH_TF32,
                  PACK_DGRAD, PACK_FWD, ConvGeom)

# Math mode of the conv engine for every plan (rcv_math):
#   parity (default, = auto)  tcgen05 3xTF32 tensor-core tiles wherever the reduction is long enough, CUDA cores
#                             elsewhere: logits within 1e-4 of the fp32 reference (the mode every parity test runs)
#   tf32 / bf16               the FAST modes, reported separately: one kind::tf32 MMA per product / bf16 operands
#                             in the halo-staged kernel; their own tolerance tests (tests/test_gpu_fast_math.py)
#   fp32                      the CUDA-core engine everywhere (A/B comparisons, bisecting a numerical difference)
# RCV_B200_MATH sets the default; `model.set_math("bf16")` switches one model.
import os as _os

MATH_KEYS = {MATH_FP32: "fp32", MATH_AUTO: "parity", MATH_TF32: "tf32", MATH_BF16: "bf16"}
MATH_BY_NAME = {"fp32": MATH_FP32, "auto": MATH_AUTO, "parity": MATH_AUTO, "tf32": MATH_TF32, "bf16": MATH_BF16}
MATH_NAMES = {MATH_FP32: "fp32 FMA (CUDA cores)",
              MATH_AUTO: "tcgen05 kind::tf32 x3 (fp32-level accuracy), TMEM accumulators",
              MATH_TF32: "tcgen05 kind::tf32, one MMA per product (fast mode)",
              MATH_BF16: "tcgen05 kind::f16 with bf16 operands, fp32 accumulate (fast mode)"}
DEFAULT_MATH = MATH_BY_NAME[_os.environ.get("RCV_B200_MATH", "parity").lower()]
WGRAD_SIDE_STREAM = _os.environ.get("RCV_B200_WGRAD_STREAM", "1") != "0"
# Training forward: where every consumer of a BatchNorm block's output is a conv the halo-staged tensor-core
# kernel runs, the block's apply pass is skipped and the consumers normalise on load (rcv_conv_fwd_nl); the
# normalised tensor the consumers' weight gradients read is produced later, on the side stream.
BN_ON_LOAD = _os.environ.get("RCV_B200_BN_ON_LOAD", "1") != "0"
# ... and where the consumer's weight gradient runs on the tensor-core quad-gather kernel it can normalise on load
# too (rcv_conv_wgrad_nl): the BatchNorm output is then never written at all.  Off by default: measured slower
# (2.206 vs 2.150 ms per step, same box) -- the transform sits on the gather's critical path, while the materialising
# pass runs on the side stream in the shadow of the input gradients.
WGRAD_ON_LOAD = _os.environ.get("RCV_B200_WGRAD_ON_LOAD", "0") != "0"


class Node:
    __slots__ = ("kind", "src", "conv", "bn", "order", "skip", "skip_mode", "geom", "_fold_key",
                 "_fold_val", "skip_ch", "_pack", "_pack_key", "_tc", "_pack_bytes")

    def __init__(self, kind, src, conv=None, bn=None, order=EPI_NONE, skip=-1, skip_mode="add"):
        self.kind, self.src, self.conv, self.bn = kind, src, conv, bn
        self.order, self.skip, self.skip_mode = order, skip, skip_mode
        self.geom = ConvGeom.of(conv) if conv is not None else None
        self._fold_key = None
        self._fold_val = None
        self.skip_ch = 0
        self._pack = [None, None]      # persistent packed-weight buffers (fwd, dgrad)
        self._pack_key = [None, None]
        self._tc = {}                  # (direction, math) -> does this direction run on tensor cores
        self._pack_bytes = {}          # (direction, math, nhw) -> panel bytes

    def params(self) -> List[nn.Parameter]:
        out = []
        if self.conv is not None:
            out.append(self.conv.weight)
            if self.conv.bias is not None:
                out.append(self.conv.bias)
        if self.bn is not None:
            out += [self.bn.weight, self.bn.bias]
        return out

    def uses_tc(self, direction: int, math: int) -> bool:
        """Does this layer / direction run on the tensor-core engine (and so need a packed panel)."""
        if math == MATH_FP32 or self.kind != "conv":
            return False
        hit = self._tc.get((direction, math))
        if hit is None:
            hit = self._tc[(direction, math)] = ops.conv_uses_tensor_cores(self.geom, direction, math)
        return hit

    def pack_buffer(self, direction: int, math: int, nhw) -> torch.Tensor:
        """Persistent panel buffer (allocated once per device, math mode and panel size; a graph that captured a
        replaced buffer keeps it alive through Plan.capture_refs)."""
        w = self.conv.weight
        buf = self._pack[direction]
        nbytes = self._pack_bytes.get((direction, math, nhw))
        if nbytes is None:
            nbytes = self._pack_bytes[(direction, math, nhw)] = ops.conv_packed_bytes(self.geom, direction, math, nhw)
        if buf is None or buf.device != w.device or buf.numel() != nbytes:
            buf = torch.empty(nbytes, device=w.device, dtype=torch.uint8)
            self._pack[direction] = buf
            self._pack_key[direction] = None
        return buf

    def pack_key(self, epoch: int, math: int, nhw):
        w = self.conv.weight
        return (w.data_ptr(), w._version, epoch, math, nhw)

    def folded(self, epoch: int = 0):
        bn = self.bn
        ts = (bn.weight, bn.bias, bn.running_mean, bn.running_var)
        key = tuple((t.data_ptr(), t._version) for t in ts) + (epoch,)
        if key != self._fold_key:
            self._fold_val = ops.bn_fold(bn.weight.detach(), bn.bias.detach(), bn.running_mean,
                                         bn.running_var, bn.eps)
            self._fold_key = key
        return self._fold_val


class PlanBuilder:
    """acts[0] is the plan input; node t produces acts[t+1]."""

    def __init__(self):
        self.nodes: List[Node] = []

    def conv(self, src: int, conv: nn.Module, bn: Optional[nn.Module], order: int, skip: int = -1,
             skip_mode: str = "add", skip_ch: int = 0) -> int:
        if bn is None and order not in (EPI_NONE, EPI_RELU):
            raise ValueError("conv without BatchNorm takes EPI_NONE or EPI_RELU")
        if bn is not None and order not in (EPI_RELU_AFFINE, EPI_AFFINE_RELU):
            raise ValueError("conv with BatchNorm takes EPI_RELU_AFFINE or EPI_AFFINE_RELU")
        nd = Node("conv", src, conv, bn, order, skip, skip_mode)
        nd.skip_ch = skip_ch
        self.nodes.append(nd)
        return len(self.nodes)

    def pool(self, src: int) -> int:
        self.nodes.append(Node("pool", src))
        return len(self.nodes)


class Plan:
    def __init__(self, builder: PlanBuilder, outputs: Sequence[int]):
        self.nodes = builder.nodes
        self.outputs = list(outputs)
        self.params: List[nn.Parameter] = []
        seen = set()
        for nd in self.nodes:
            for p in nd.params():
                if id(p) not in seen:
                    seen.add(id(p))
                    self.params.append(p)
        self.math = DEFAULT_MATH
        self._wgrad_stream = None
        self._pack_tables = {}
        # bumped whenever parameters / BN buffers may have been written behind torch's back (raw
        # kernels of a training forward or of TrainStep): invalidates folded-BN and packed caches
        self.epoch = 0
        # consumers of every activation: (node index, "src" | "skip")
        self._consumers = {}
        for t, nd in enumerate(self.nodes):
            self._consumers.setdefault(nd.src, []).append((t, "src"))
            if nd.skip is not None and nd.skip >= 0:
                self._consumers.setdefault(nd.skip, []).append((t, "skip"))
        self._defer_cache = {}
        self._size_cache = {}
        self._workspace = None   # scratch of the tensor-core convs (ops.new_workspace), sized for the largest need seen
        self._ws_need = {}
        self.n_stats = 0
        self._sum_off = {}
        for t, nd in enumerate(self.nodes):
            if nd.bn is not None:
                self._sum_off[t] = self.n_stats
                self.n_stats += 2 * nd.geom.cout

    def _in_sizes(self, n: int, h: int, w: int):
        """(N, H, W) of every node's main input for a plan input of that size."""
        key = (n, h, w)
        hit = self._size_cache.get(key)
        if hit is None:
            hw = [(h, w)]
            for nd in self.nodes:
                ih, iw = hw[nd.src]
                hw.append((ih // 2, iw // 2) if nd.kind == "pool" else nd.geom.out_hw(ih, iw))
            hit = self._size_cache[key] = [(n, *hw[nd.src]) for nd in self.nodes]
        return hit

    def workspace(self, nhw, dev) -> Optional[torch.Tensor]:
        """The plan's conv scratch for a plan input of size nhw = (N, H, W): one buffer, shared by every tensor-core
        layer and direction (they run one after the other on the plan's main stream), zero-filled when allocated
        (the kernels leave it ready for the next launch).  None when no layer can use one."""
        key = (nhw, self.math)
        need = self._ws_need.get(key)
        if need is None:
            need = 0
            if self.math != MATH_FP32:
                for nd, (n, h, w) in zip(self.nodes, self._in_sizes(*nhw)):
                    if nd.kind == "conv":
                        for d in (PACK_FWD, PACK_DGRAD):
                            if nd.uses_tc(d, self.math):
                                need = max(need, ops.conv_workspace_bytes(nd.geom, n, h, w, d, self.math))
            self._ws_need[key] = need
        if need == 0:
            return None
        ws = self._workspace
        if ws is None or ws.device != dev or ws.numel() < need:
            ws = self._workspace = ops.new_workspace(need, dev)
        return ws

    def capture_refs(self) -> List[torch.Tensor]:
        """The device buffers a CUDA graph captured now can bake in: the conv workspace, every node's weight panels and
        the device table of every cached PackTable.  The plan replaces them when an input size needs a larger or a
        different buffer, so whoever keeps a graph keeps this list beside it: a replaced buffer is then freed only
        once no graph that uses it is left."""
        refs = [] if self._workspace is None else [self._workspace]
        refs += [b for nd in self.nodes for b in nd._pack if b is not None]
        refs += [tbl.table for tbl in self._pack_tables.values()]
        return refs

    def _ensure_packed(self, directions, fresh: bool, x_requires_grad: bool, nhw):
        """Weight panels of every tensor-core layer, re-packed in ONE launch when `fresh` (training:
        the weights change every step) or when any weight tensor / the plan epoch changed.  nhw: the plan input's
        (N, H, W) -- a panel's layout follows the kernel the layer runs on at its input size (bf16 panels of the
        fast mode, and any future size-dependent layout)."""
        sizes = self._in_sizes(*nhw)  # panel layouts follow the kernel each layer runs on at its input size
        jobs = [(nd, d, sz) for nd, sz in zip(self.nodes, sizes) if nd.kind == "conv" for d in directions
                if nd.uses_tc(d, self.math) and not (d == PACK_DGRAD and nd.src == 0 and not x_requires_grad)]
        if not jobs:
            return
        bufs = [nd.pack_buffer(d, self.math, sz) for nd, d, sz in jobs]
        if not fresh and all(nd._pack_key[d] == nd.pack_key(self.epoch, self.math, sz) for nd, d, sz in jobs):
            return
        tkey = tuple((nd.conv.weight.data_ptr(), b.data_ptr(), sz) for (nd, _, sz), b in zip(jobs, bufs))
        tbl = self._pack_tables.get((tuple(directions), self.math))
        if tbl is None or tbl.key != tkey:
            tbl = ops.PackTable([(nd.geom, d, nd.conv.weight.detach(), b) for (nd, d, _), b in zip(jobs, bufs)],
                                math=self.math, sizes=[sz for _, _, sz in jobs])
            tbl.key = tkey
            self._pack_tables[(tuple(directions), self.math)] = tbl
        tbl.run()
        for nd, d, sz in jobs:
            nd._pack_key[d] = nd.pack_key(self.epoch, self.math, sz)

    def _defer_bn_apply(self, t: int, n: int, h: int, w: int) -> bool:
        """Can node t's BatchNorm apply pass be left to its consumers (normalise-on-load)?  Its output must feed only
        conv nodes, as their main input, that the halo-staged tensor-core kernel runs at this size; it must not be
        a plan output and the node must not add a skip tensor after the BatchNorm."""
        key = (t, n, h, w)
        hit = self._defer_cache.get(key)
        if hit is None:
            nd = self.nodes[t]
            cons = self._consumers.get(t + 1, [])
            hit = (BN_ON_LOAD and self.math != MATH_FP32 and nd.skip < 0 and (t + 1) not in self.outputs and
                   len(cons) > 0 and
                   all(role == "src" and self.nodes[c].kind == "conv" and
                       ops.conv_normalises_on_load(self.nodes[c].geom, n, h, w, self.math) for c, role in cons))
            self._defer_cache[key] = hit
        return hit

    # ------------------------------------------------------------------ forward
    def fusable_head(self) -> int:
        """Index of the last node if it is a bare 1x1 stride-1 classifier conv (no BatchNorm, no ReLU, no skip) whose
        output is the plan's only output -- the head TrainStep can hand to ops.head_ce_train -- else -1."""
        if not self.nodes or self.outputs != [len(self.nodes)]:
            return -1
        nd = self.nodes[-1]
        if nd.kind != "conv" or nd.bn is not None or nd.order != EPI_NONE or nd.skip >= 0:
            return -1
        g = nd.geom
        if g.k != 1 or g.stride != 1 or g.pad != 0 or g.transposed or not ops.head_ce_supported(g.cin, g.cout):
            return -1
        if any(other.src == len(self.nodes) or other.skip == len(self.nodes) for other in self.nodes):
            return -1
        return len(self.nodes) - 1

    def forward(self, x: torch.Tensor, training: bool, save: bool, stats_arena: Optional[torch.Tensor] = None,
                stop_before: Optional[int] = None, batch_reduce=None):
        """-> (outputs, saved).  training selects batch statistics for BatchNorm nodes whose
        module is in training mode; save keeps what backward needs.  stats_arena: caller-zeroed float64[n_stats]
        for the batch statistics (TrainStep zeroes all of a step's accumulators with one memset).
        stop_before: run nodes [0, stop_before) only (TrainStep's fused head); outputs that were not produced are
        None, and backward() then starts from the `seed` gradients it is given.
        batch_reduce: BatchNorm over a batch split across ranks (TrainStep(global_batch=True)) -- an object with
        `world` and `sum(buf)` / `mean(buf)`, which replace a float64 slice by its sum / mean over the ranks in place
        on the current stream.  Every train-mode BatchNorm's statistics are summed between its conv and its finalize,
        which then divides by the global count (this rank's N*H*W times world; every rank holds as many samples)."""
        x = ops._chk(x, name="input")
        if x.dim() != 4:
            raise ValueError(f"expected NCHW input, got shape {tuple(x.shape)}")
        dev = x.device
        acts: List[torch.Tensor] = [x]
        lazy: Dict[int, tuple] = {}  # activation index -> (scale, shift, relu): acts[i] holds the tensor BEFORE that affine
        saved: List[Optional[tuple]] = [None] * len(self.nodes)
        soff = 0
        if training:
            self.epoch += 1
        nhw = (x.shape[0], x.shape[2], x.shape[3])
        self._ensure_packed((PACK_FWD, PACK_DGRAD) if save else (PACK_FWD,), training, x.requires_grad, nhw)
        ws = self.workspace(nhw, dev)
        for t, nd in enumerate(self.nodes):
            if stop_before is not None and t >= stop_before:
                break
            src = acts[nd.src]
            if nd.kind == "pool":
                y, _, code = ops.maxpool2x2_fwd(src, want_idx=False, want_code=save)
                saved[t] = (code,)
                acts.append(y)
                continue
            g, conv, bn = nd.geom, nd.conv, nd.bn
            w = conv.weight.detach()
            b = conv.bias.detach() if conv.bias is not None else None
            skip = acts[nd.skip] if (nd.skip >= 0 and nd.skip_mode == "add") else None
            # partial skip (LabelProp, model.py:565: x[:, 0:8] += top): the train-mode BatchNorm apply pass adds it to
            # the first channels itself, and so does the narrow-layer engine's epilogue in eval mode
            partial_fused = False
            if nd.skip >= 0 and nd.skip_mode == "partial":
                if bn is not None and training and bn.training:
                    partial_fused = not self._defer_bn_apply(t, src.shape[0], *g.out_hw(src.shape[2], src.shape[3]))
                else:
                    partial_fused = ops.conv_takes_partial_residual(g, src.shape[0], src.shape[2], src.shape[3], self.math)
                if partial_fused:
                    skip = acts[nd.skip]
            wp = nd._pack[PACK_FWD] if nd.uses_tc(PACK_FWD, self.math) else None
            ina = lazy.get(nd.src)  # the producer's BatchNorm, applied on load
            if bn is None:
                y = ops.conv_fwd(g, src, w, b, epilogue=nd.order, math=self.math, wpacked=wp, in_affine=ina,
                                 workspace=ws)
                saved[t] = (y if nd.order == EPI_RELU else None,)
            elif training and bn.training:
                if stats_arena is None:
                    stats_arena = ops.zeros(self.n_stats, torch.float64, dev)
                stats = stats_arena[soff:soff + 2 * g.cout]
                soff += 2 * g.cout
                z = ops.conv_fwd(g, src, w, b, epilogue=EPI_RELU if nd.order == EPI_RELU_AFFINE else EPI_NONE,
                                 stats=stats, math=self.math, wpacked=wp, in_affine=ina, workspace=ws)
                count = z.numel() // g.cout
                if batch_reduce is not None:
                    batch_reduce.sum(stats)
                    count *= batch_reduce.world
                if bn.momentum is None:
                    momentum = 1.0 / float(int(bn.num_batches_tracked) + 1)
                else:
                    momentum = bn.momentum
                track = bn.track_running_stats and bn.running_mean is not None
                nbt = bn.num_batches_tracked if (track and bn.num_batches_tracked is not None) else None
                if self._defer_bn_apply(t, z.shape[0], z.shape[2], z.shape[3]):
                    scale, shift, mean, invstd = ops.bn_finalize(
                        stats, count, bn.weight.detach(), bn.bias.detach(), bn.running_mean if track else None,
                        bn.running_var if track else None, momentum, bn.eps, num_batches_tracked=nbt)
                    lazy[t + 1] = (scale, shift, nd.order == EPI_AFFINE_RELU)
                    y = z  # consumers read z through the affine
                else:
                    y, scale, shift, mean, invstd = ops.bn_finalize_apply(
                        z, stats, bn.weight.detach(), bn.bias.detach(),
                        bn.running_mean if track else None, bn.running_var if track else None, momentum, bn.eps,
                        relu=(nd.order == EPI_AFFINE_RELU), residual=skip, num_batches_tracked=nbt,
                        **({} if batch_reduce is None else {"count": count}))
                saved[t] = (z, scale, shift, mean, invstd)
            else:
                scale, shift = nd.folded(self.epoch)
                y = ops.conv_fwd(g, src, w, b, epilogue=nd.order, scale=scale, shift=shift, residual=skip,
                                 math=self.math, wpacked=wp, in_affine=ina, workspace=ws)
            if nd.skip >= 0 and nd.skip_mode == "partial" and not partial_fused:
                y[:, :nd.skip_ch] += acts[nd.skip]
            elif nd.skip >= 0 and nd.skip_mode == "cat":
                y = ops.concat_channels(y, acts[nd.skip])
            acts.append(y)
        outs = [acts[i] if i < len(acts) else None for i in self.outputs]
        return outs, ((acts, saved, lazy) if save else None)

    # ------------------------------------------------------------------ backward
    def backward(self, saved_all, gouts: Sequence[Optional[torch.Tensor]], x_needs_grad: bool,
                 grad_views: Optional[Dict[int, torch.Tensor]] = None, node_done=None,
                 sums_arena: Optional[torch.Tensor] = None, seed: Optional[Dict[int, torch.Tensor]] = None,
                 batch_reduce=None):
        """-> (dx or None, {id(param): grad}).  grad_views, if given, maps id(param) to zero-filled
        tensors that receive the gradients (the train step's flat arena).  node_done(t) is called
        once node t's parameter gradients are final (nodes are visited last to first).  sums_arena: caller-zeroed
        float64[n_stats] for the BatchNorm-backward sums.  seed: {activation index: gradient} for a forward that
        stopped early (forward(stop_before=...)): the nodes that did not run are skipped, node_done still sees them.
        batch_reduce: as for forward(); every BatchNorm backward then runs as its two passes with the channel sums
        averaged over the ranks between them.  The apply pass divides by this rank's N*H*W, so the averaged sums give
        the global means; the dgamma / dbeta it adds are the averages, which the sum all-reduce of the gradients
        turns back into the global sums."""
        acts, saved, lazy = saved_all
        lazy_done: Dict[int, torch.Tensor] = {}  # BatchNorm outputs materialised for a weight gradient, per activation
        dev = acts[0].device
        if grad_views is None:
            total = sum(p.numel() for p in self.params)
            flat = ops.zeros(total, torch.float32, dev)
            grad_views, o = {}, 0
            for p in self.params:
                grad_views[id(p)] = flat[o:o + p.numel()].view(p.shape)
                o += p.numel()
        grads: List[Optional[torch.Tensor]] = [None] * len(acts)

        def add_to(i, g):
            grads[i] = g if grads[i] is None else grads[i] + g

        for oi, g in zip(self.outputs, gouts):
            if g is not None:
                add_to(oi, g)
        for i, g in (seed or {}).items():
            add_to(i, g)
        if sums_arena is None:
            sums_arena = ops.zeros(max(self.n_stats, 1), torch.float64, dev)
        # Weight gradients run on a side stream: dgrad(t) and wgrad(t) only share their input, so the
        # wgrad CTAs fill the SMs a dgrad's partial last wave leaves idle (150 tiles on 148 SMs at
        # 15x20) and overlap the next node's BatchNorm backward.  Tensors the side stream reads are
        # kept alive until the streams join, so the caching allocator cannot hand them out early.
        side = None
        if WGRAD_SIDE_STREAM:
            cur = torch.cuda.current_stream(dev)
            if self._wgrad_stream is None or self._wgrad_stream.device != dev:
                self._wgrad_stream = torch.cuda.Stream(device=dev)
            side = self._wgrad_stream
        keep: List[torch.Tensor] = []
        for t in range(len(self.nodes) - 1, -1, -1):
            if t + 1 < len(acts):  # (a node the forward pass stopped before has no activation and no gradient)
                self._backward_node(t, acts, saved, grads, grad_views, sums_arena, x_needs_grad, add_to, side, keep,
                                    lazy, lazy_done, batch_reduce)
            if node_done is not None:
                node_done(t)
        if side is not None:
            cur.wait_stream(side)
        keep.clear()
        return grads[0], grad_views

    def _backward_node(self, t, acts, saved, grads, grad_views, sums_arena, x_needs_grad, add_to, side=None,
                       keep=None, lazy=None, lazy_done=None, batch_reduce=None):
        nd = self.nodes[t]
        g = grads[t + 1]
        grads[t + 1] = None
        if nd.bn is not None:
            soff = self._sum_off[t]
            sums = sums_arena[soff:soff + 2 * nd.geom.cout]
        if g is None:
            return
        g = ops._chk(g, name="grad")
        src = acts[nd.src]
        in_hw = (src.shape[2], src.shape[3])
        if nd.kind == "pool":
            add_to(nd.src, ops.maxpool2x2_bwd(g, saved[t][0], in_hw))
            return
        geom, conv, bn = nd.geom, nd.conv, nd.bn
        if nd.skip >= 0:
            if nd.skip_mode == "add":
                add_to(nd.skip, g)
            elif nd.skip_mode == "partial":
                add_to(nd.skip, ops.channel_slice(g, 0, nd.skip_ch))
            else:  # cat
                add_to(nd.skip, ops.channel_slice(g, geom.cout, g.shape[1] - geom.cout))
                g = ops.channel_slice(g, 0, geom.cout)
        w = conv.weight.detach()
        has_bias = conv.bias is not None
        if bn is not None:
            if saved[t] is None or len(saved[t]) != 5:
                raise NotImplementedError(
                    "backward through an eval-mode BatchNorm block is not on the hot path "
                    "(call model.train() before the forward pass you differentiate)")
            z, scale, shift, mean, invstd = saved[t]
            dbias = grad_views[id(conv.bias)] if has_bias else None
            if batch_reduce is None:
                dconv, _, _, _ = ops.bn_bwd(nd.order, g, z, scale, shift, mean, invstd,
                                            dgamma=grad_views[id(bn.weight)], dbeta=grad_views[id(bn.bias)],
                                            dbias=dbias, sums=sums)
            else:
                ops.bn_bwd_reduce(nd.order, g, z, scale, shift, mean, invstd, sums)
                batch_reduce.mean(sums)
                dconv = ops.bn_bwd_apply(nd.order, g, z, scale, shift, mean, invstd, sums,
                                         dgamma=grad_views[id(bn.weight)], dbeta=grad_views[id(bn.bias)], dbias=dbias)
            wg_bias = None
        else:
            dconv = ops.relu_bwd(g, saved[t][0]) if nd.order == EPI_RELU else g
            wg_bias = grad_views[id(conv.bias)] if has_bias else None
        if nd.src != 0 or x_needs_grad:
            wp = nd._pack[PACK_DGRAD] if nd.uses_tc(PACK_DGRAD, self.math) else None
            x0 = acts[0]
            grads[nd.src] = ops.conv_dgrad(geom, dconv, w, in_hw, residual=grads[nd.src], math=self.math,
                                           wpacked=wp, workspace=self.workspace(
                                               (x0.shape[0], x0.shape[2], x0.shape[3]), x0.device))
        la = lazy.get(nd.src) if lazy else None
        if la is not None and WGRAD_ON_LOAD and ops.conv_wgrad_normalises_on_load(
                geom, src.shape[0], src.shape[2], src.shape[3], self.math):
            wg_affine, la = la, None  # the weight-gradient kernel applies the BatchNorm itself
        else:
            wg_affine = None

        def wgrad_src():
            """The tensor the weight gradient reads: for a normalise-on-load input, the producer's BatchNorm output,
            produced now (once per activation) on the stream the weight gradient runs on."""
            if la is None:
                return src
            y = lazy_done.get(nd.src)
            if y is None:
                y = ops.bn_apply(src, la[0], la[1], la[2])
                lazy_done[nd.src] = y
                if keep is not None:
                    keep.append(y)
            return y

        if side is None:
            ops.conv_wgrad(geom, wgrad_src(), dconv, dw=grad_views[id(conv.weight)], dbias=wg_bias, math=self.math,
                           in_affine=wg_affine)
        else:
            cur = torch.cuda.current_stream(src.device)
            side.wait_stream(cur)  # dconv (and every earlier write to the gradient arena) is ordered before
            keep.append(dconv)
            with torch.cuda.stream(side):
                ops.conv_wgrad(geom, wgrad_src(), dconv, dw=grad_views[id(conv.weight)], dbias=wg_bias,
                               math=self.math, in_affine=wg_affine)


class _PlanFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, plan: Plan, training: bool, need: bool, x: torch.Tensor, *params):
        # (grad mode is always off inside Function.forward, so `need` is decided by the caller)
        outs, saved = plan.forward(x, training, save=need and training)
        ctx.plan, ctx.saved, ctx.training = plan, saved, training
        ctx.x_needs_grad = x.requires_grad
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        if ctx.saved is None:
            raise NotImplementedError(
                "robocupvision_b200: backward needs a training-mode forward (model.train()); "
                "eval-mode forwards keep no activations")
        dx, gv = ctx.plan.backward(ctx.saved, gouts, ctx.x_needs_grad)
        ctx.saved = None
        return (None, None, None, dx, *[gv[id(p)] for p in ctx.plan.params])


def _alert_not_deterministic(what: str) -> None:
    """torch.use_deterministic_algorithms(True): raise RuntimeError naming `what`, or warn under warn_only=True, as
    torch's own nondeterministic ops do."""
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = (f"{what} does not have a deterministic implementation, but you set "
           "'torch.use_deterministic_algorithms(True)'. You can turn off determinism just for this operation, or use "
           "the 'warn_only=True' option.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(msg, UserWarning, stacklevel=3)
    else:
        raise RuntimeError(msg)


def run_plan(plan: Plan, x: torch.Tensor, training: bool) -> Tuple[torch.Tensor, ...]:
    if not x.is_cuda:
        raise RuntimeError(
            "robocupvision_b200 runs on CUDA (sm_100a) only: move the model and its input to the GPU. "
            "There is no CPU fallback; the CPU oracle under oracle/ is test infrastructure.")
    if x.dtype != torch.float32:
        raise TypeError(f"robocupvision_b200: fp32 input expected, got {x.dtype}")
    if training:
        # eval mode sums nothing across CTAs in floating point (the split reduction adds its shares in share order);
        # train mode adds the BatchNorm batch statistics, and its backward the weight / bias gradients and the
        # BatchNorm backward sums, with floating-point atomics
        _alert_not_deterministic(
            "robocupvision_b200 train-mode forward and backward (BatchNorm batch statistics, weight gradients, "
            "BatchNorm backward sums)")
    need = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in plan.params))
    return _PlanFn.apply(plan, training, need, x, *plan.params)
