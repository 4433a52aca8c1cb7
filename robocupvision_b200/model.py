"""Drop-in replacement for the hot-path classes of the reference ``model.py``.

Same class names, constructor signatures, sub-module names, parameter registration order and
``state_dict`` keys as /root/reference/model.py, so ``train.py``, ``trainer.py``, ``test.py``,
``tester.py``, ``detect.py`` and ``validLabelProp.py`` can ``from robocupvision_b200.model
import *`` instead of ``from model import *``.  Parameters still live in ordinary
``nn.Conv2d`` / ``nn.ConvTranspose2d`` / ``nn.BatchNorm2d`` holders (callers rely on
``isinstance(m, nn.Conv2d)``, ``reset_parameters()`` and ``weight.nonzero()``), but no torch
convolution / batch-norm / pooling kernel ever runs: every ``forward`` lowers the module tree
to an execution plan (engine.py) whose nodes are the sm_100a kernels of librcv_b200.so.

Block orders (reference file:line):
  Conv                   bn(relu(conv(x)+b))              model.py:105-116
  ConvPoolSimple         relu(bn(conv(x)))                model.py:166-176
  ConvPool               relu(bn(pool(relu(conv1(x)))))   model.py:126-142
  ConvPoolDouble         ... two dilated convs first      model.py:144-164
  upSampleTransposeConv  relu(bn(convT(x)+b))             model.py:178-194
  decoder skips          up(x) + skip (after the ReLU)    model.py:300-307, 505-509, 562-565
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .engine import Plan, PlanBuilder, run_plan
from .ops import EPI_AFFINE_RELU, EPI_NONE, EPI_RELU, EPI_RELU_AFFINE

__all__ = [
    "DiceLoss", "CrossEntropyLoss2d", "pruneModelNew", "pruneModel", "pruneModel2", "count_zero_weights",
    "getParamSize", "Pool", "PoolWithIndices", "MaxUnpool2x2", "UpsampleBilinear2x", "Conv", "ConvPool", "ConvPoolDouble", "ConvPoolSimple",
    "upSampleTransposeConv", "DownSampler", "DownSamplerThick", "Classifier", "PB_FCN", "FCN",
    "LevelDown", "UltClassifier", "ROBO_UNet", "LabelProp", "PB_FCN_2", "load_legacy_state_dict",
    "remap_legacy_keys", "torch", "nn",
]


# =============================================================================== plumbing
class _PlanModule(nn.Module):
    """nn.Module whose forward is a cached execution plan over its own sub-modules."""

    def _emit(self, b: PlanBuilder, src: int, **kw):
        raise NotImplementedError

    def _plan_outputs(self, b: PlanBuilder):
        return [self._emit(b, 0)]

    def _get_plan(self) -> Plan:
        plan = self.__dict__.get("_rcv_plan")
        if plan is None:
            b = PlanBuilder()
            outs = self._plan_outputs(b)
            plan = Plan(b, outs)
            self.__dict__["_rcv_plan"] = plan
        return plan

    def invalidate_plan(self):
        self.__dict__.pop("_rcv_plan", None)

    def set_math(self, mode: str):
        """Math mode of this model's tensor-core layers: "parity" (default: 3xTF32, logits within 1e-4 of fp32), the
        fast modes "tf32" / "bf16" (reported separately; see include/rcv_b200.h rcv_math), or "fp32" (CUDA cores)."""
        from .engine import MATH_BY_NAME
        plan = self._get_plan()
        plan.math = MATH_BY_NAME[mode.lower()]
        plan.epoch += 1
        plan._defer_cache.clear()
        return self

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k != "_rcv_plan":
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def forward(self, x):
        return run_plan(self._get_plan(), x, self.training)[0]


# =============================================================================== losses
_loss_scratches = {}


def _loss_scratch(op, logits):
    """Under torch.use_deterministic_algorithms(True): scratch for the fixed-order form of the loss reduction (its sums
    are then bitwise the same run after run on the same device).  Otherwise None: the atomic form.  The backward
    kernels of both losses are element-wise and need nothing.  One zero-filled scratch per (op, shape, device, stream),
    allocated on first use and kept: the kernels leave it ready for the next call, and calls on one stream are ordered,
    so a step in a loop allocates and fills nothing."""
    if not torch.are_deterministic_algorithms_enabled():
        return None
    n, c = logits.shape[0], logits.shape[1]
    hw = logits.numel() // (n * c)
    key = (op, n, c, hw, logits.device, torch.cuda.current_stream(logits.device).cuda_stream)
    scratch = _loss_scratches.get(key)
    if scratch is None:
        scratch = _loss_scratches[key] = ops.det_scratch(op, n, c, hw, logits.device)
    return scratch


class _WeightedCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, weight):
        sums, _, _, _ = ops.ce_fwd(logits, target, weight, scratch=_loss_scratch(ops.DET_CE_FWD, logits))
        ctx.save_for_backward(logits, target, sums)
        ctx.weight = weight
        return (sums[0] / sums[1]).to(torch.float32)

    @staticmethod
    def backward(ctx, gout):
        logits, target, sums = ctx.saved_tensors
        return ops.ce_bwd(logits, target, ctx.weight, sums, gscale=gout), None, None


class CrossEntropyLoss2d(nn.Module):
    """Class-weighted mean of -log softmax(x)[y] over all pixels (model.py:76-82):
    loss = sum_p w[y_p] * nll_p / sum_p w[y_p].  One fused kernel forward, one backward.  Under
    torch.use_deterministic_algorithms(True) the forward sums in fixed order (rcv_ce_fwd_det): the same logits give
    bitwise the same loss and gradient, run after run on one device."""

    def __init__(self, weight=None):
        super().__init__()
        self.register_buffer("weight", None if weight is None else torch.as_tensor(weight, dtype=torch.float32))

    def forward(self, inputs, targets):
        if not inputs.is_cuda:
            raise RuntimeError("robocupvision_b200.CrossEntropyLoss2d runs on CUDA only (no CPU fallback)")
        w = self.weight
        if w is not None and w.device != inputs.device:
            w = w.to(inputs.device)
            self.weight = w
        return _WeightedCE.apply(inputs, targets.long(), w)


class _Dice(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, weights, eps):
        sums = ops.dice_fwd(logits, target, scratch=_loss_scratch(ops.DET_DICE_FWD, logits))
        c = logits.shape[1]
        ctx.save_for_backward(logits, target, weights, sums)
        ctx.eps = eps
        dice = (2.0 * weights.double() * sums[:c] / (sums[c:] + eps)).mean()
        return (1.0 - dice).to(torch.float32)

    @staticmethod
    def backward(ctx, gout):
        logits, target, weights, sums = ctx.saved_tensors
        return ops.dice_bwd(logits, target, weights, sums, ctx.eps, gscale=gout), None, None, None


class DiceLoss(nn.Module):
    """Optional `--useDice` loss (model.py:5-43): 1 - mean_c(2 w_c I_c / (K_c + eps)) with the soft
    intersection I and cardinality K of softmax(logits) against the one-hot labels, w normalised to sum to C.
    CUDA logits, 2..8 classes: one fused kernel forward (rcv_dice_fwd) and one backward (rcv_dice_bwd); under
    torch.use_deterministic_algorithms(True) the forward sums in fixed order (rcv_dice_fwd_det).  The single-logit
    sigmoid form (model.py:25-32, never used by the drivers) stays plain tensor ops."""

    def __init__(self, weights, eps=1e-7):
        super().__init__()
        weights = torch.as_tensor(weights, dtype=torch.float32)
        self.weights = weights / weights.sum().item() * weights.shape[0]
        self.eps = eps

    def __call__(self, logits, true):
        c = logits.shape[1]
        lab = true.squeeze(1).long() if true.dim() == logits.dim() else true.long()
        if c == 1:
            pos = torch.sigmoid(logits)
            probas = torch.cat([pos, 1 - pos], dim=1)
            onehot = torch.stack([(lab == 1), (lab == 0)], dim=1).to(logits.dtype)
            dims = (0,) + tuple(range(2, logits.dim()))
            inter = (probas * onehot).sum(dims)
            card = (probas + onehot).sum(dims)
            w = self.weights.to(logits.device)
            return 1 - (2.0 * w * inter / (card + self.eps)).mean()
        if not logits.is_cuda:
            raise RuntimeError("robocupvision_b200.DiceLoss runs on CUDA only (no CPU fallback)")
        if self.weights.device != logits.device:
            self.weights = self.weights.to(logits.device)
        return _Dice.apply(logits, lab.contiguous(), self.weights, self.eps)


# =============================================================================== pruning helpers
def getParamSize(x):
    n = 1
    for s in x.size():
        n *= s
    return n


def pruneModelNew(params, ratio=0.01):
    """Magnitude pruning of every >1-D parameter below ratio*max|p| (model.py:45-57).
    Returns the list of boolean masks (in parameter order) later applied to the gradients."""
    masks = []
    for p in params:
        if p.dim() > 1:
            thresh = p.abs().max() * ratio
            small = p.abs() < thresh
            print("Pruned %f%% of the weights" % (float(small.sum()) / float((p != 0).sum()) * 100))
            p[small] = 0
            masks.append(p.abs() < thresh)
    return masks


def count_zero_weights(model):
    """Fraction of parameters below 1% of their tensor's max magnitude (model.py:59-66)."""
    small, total = 0, 0
    for p in model.parameters():
        small += (p.abs() < p.abs().max() * 0.01).sum().float()
        total += p.numel()
    return float(small / total)


def pruneModel(params, lower=73, upper=77):
    """Per-tensor threshold search so that lower..upper % of the weights fall below it
    (model.py:621-642)."""
    masks = []
    for p in params:
        if p.dim() > 1:
            p = p.data
            thresh = p.std()
            while True:
                pct = float((p.abs() < thresh).sum()) / float((p != 0).sum()) * 100
                if pct < lower:
                    thresh *= 1.025
                elif pct > upper:
                    thresh *= 0.975
                else:
                    break
            print("Pruned %f%% of the weights" % pct)
            p[p.abs() < thresh] = 0
            masks.append(p.abs() < thresh)
    return masks


def pruneModel2(params, ratio, lT, hT):
    """Zero the `ratio` smallest-magnitude entries of each >1-D parameter, with the size-dependent
    ratio adjustments of model.py:644-672."""
    masks = []
    for p in params:
        if p.dim() > 1:
            size = getParamSize(p)
            r = ratio
            if size < 100:
                r = 0
            elif size < lT:
                r = ratio * 0.8
            if size > hT:
                r = ratio * 1.05
            flat = p.reshape(-1)
            amount = int(flat.size(0) * r)
            if amount > 0:
                _, idx = torch.topk(flat.abs(), amount, dim=0, largest=False)
                flat[idx] = 0.0
            print("Pruned %d of %d weights (%.3f%%)" % (amount, flat.size(0), r))
            masks.append(flat.reshape(p.size()) == 0.0)
    return masks


# =============================================================================== blocks
class Pool(_PlanModule):
    """MaxPool2d(2,2) (model.py:92-103); `--UNet` only."""

    def __init__(self, ch, stride=2):
        super().__init__()
        self.ch = ch
        self.stride = stride
        self.pool = nn.MaxPool2d(stride, stride)

    def _emit(self, b, src, **kw):
        if self.stride != 2:
            raise NotImplementedError("Pool: only stride 2 is on the hot path")
        return b.pool(src)

    def getComp(self, W, H, pruned):
        return W * H * self.ch, W // self.stride, H // self.stride


class _PoolIdx(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        y, idx, code = ops.maxpool2x2_fwd(x, want_idx=True, want_code=True)
        ctx.save_for_backward(code)
        ctx.in_hw = tuple(x.shape[2:])
        ctx.mark_non_differentiable(idx)
        return y, idx

    @staticmethod
    def backward(ctx, dy, _didx):
        return ops.maxpool2x2_bwd(dy.contiguous(), ctx.saved_tensors[0], ctx.in_hw)


class _Unpool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, idx, skip):
        ctx.save_for_backward(idx)
        ctx.has_skip = skip is not None
        return ops.maxunpool2x2(y, idx=idx, skip=skip)

    @staticmethod
    def backward(ctx, dout):
        dout = dout.contiguous()
        return ops.maxunpool2x2_bwd(dout, idx=ctx.saved_tensors[0]), None, (dout if ctx.has_skip else None)


class _Bilinear2x(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, skip):
        ctx.has_skip = skip is not None
        return ops.upsample_bilinear2x(x, skip=skip)

    @staticmethod
    def backward(ctx, dout):
        dout = dout.contiguous()
        return ops.upsample_bilinear2x_bwd(dout), (dout if ctx.has_skip else None)


class PoolWithIndices(nn.Module):
    """nn.MaxPool2d(2, 2, return_indices=True): the pool half of the pool-index / unpool pair north_star names (the
    reference's own Pool, model.py:92-100, keeps the indices implicit).  -> (y, int64 indices)."""

    def forward(self, x):
        return _PoolIdx.apply(x)


class MaxUnpool2x2(nn.Module):
    """nn.MaxUnpool2d(2, 2) with an optional fused skip add (`up = unpool(x, idx) + skip`, the decoder pattern of
    model.py:505-509 with the transposed convolution swapped for an unpool)."""

    def forward(self, y, indices, skip=None):
        return _Unpool.apply(y, indices, skip)


class UpsampleBilinear2x(nn.Module):
    """F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False) with an optional fused skip add."""

    def forward(self, x, skip=None):
        return _Bilinear2x.apply(x, skip)


def _nnz_ratio(w, pruned):
    return float(w.nonzero().size(0)) / float(w.numel()) if pruned else 1


class Conv(_PlanModule):
    def __init__(self, inplanes, planes, size, stride=1):
        super().__init__()
        self.stride = stride
        self.size = size
        self.inch = inplanes
        self.ch = planes
        self.conv = nn.Conv2d(inplanes, planes, kernel_size=size, padding=size // 2, stride=stride)
        self.bn = nn.BatchNorm2d(planes)

    def _emit(self, b, src, **kw):
        return b.conv(src, self.conv, self.bn, EPI_RELU_AFFINE)

    def getComp(self, W, H, pruned):
        W, H = W // self.stride, H // self.stride
        r = _nnz_ratio(self.conv.weight, pruned)
        return self.size * self.size * W * H * self.inch * self.ch * 2 * r + W * H * self.ch * 4, W, H


class ConvPool(_PlanModule):
    def __init__(self, inplanes, planes):
        super().__init__()
        self.relu = nn.ReLU()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=3, dilation=2, padding=2, bias=False)
        self.pool = nn.Conv2d(planes, planes, kernel_size=3, padding=1, stride=2, bias=False)
        self.bn = nn.BatchNorm2d(planes)

    def _emit(self, b, src, **kw):
        t = b.conv(src, self.conv1, None, EPI_RELU)
        return b.conv(t, self.pool, self.bn, EPI_AFFINE_RELU)


class ConvPoolDouble(_PlanModule):
    def __init__(self, inplanes, planes):
        super().__init__()
        self.relu = nn.ReLU()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=3, dilation=2, padding=2, bias=False)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, dilation=2, padding=2, bias=False)
        self.pool = nn.Conv2d(planes, planes, kernel_size=3, padding=1, stride=2, bias=False)
        self.bn = nn.BatchNorm2d(planes)

    def _emit(self, b, src, **kw):
        t = b.conv(src, self.conv1, None, EPI_RELU)
        t = b.conv(t, self.conv2, None, EPI_RELU)
        return b.conv(t, self.pool, self.bn, EPI_AFFINE_RELU)


class ConvPoolSimple(_PlanModule):
    def __init__(self, inplanes, planes, size, stride, padding, dilation, bias):
        super().__init__()
        self.conv = nn.Conv2d(inplanes, planes, size, stride=stride, padding=padding, dilation=dilation,
                              bias=bias)
        self.bn = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU()

    def _emit(self, b, src, **kw):
        return b.conv(src, self.conv, self.bn, EPI_AFFINE_RELU)


class upSampleTransposeConv(_PlanModule):
    def __init__(self, inplanes, planes):
        super().__init__()
        self.stride = 2
        self.size = 3
        self.inch = inplanes
        self.ch = planes
        self.relu = nn.ReLU()
        self.conv = nn.ConvTranspose2d(inplanes, planes, kernel_size=3, padding=1, stride=2,
                                       output_padding=1, bias=True)
        self.bn = nn.BatchNorm2d(planes)

    def _emit(self, b, src, skip=-1, skip_mode="add", skip_ch=0, **kw):
        return b.conv(src, self.conv, self.bn, EPI_AFFINE_RELU, skip=skip, skip_mode=skip_mode,
                      skip_ch=skip_ch)

    def getComp(self, W, H, pruned):
        r = _nnz_ratio(self.conv.weight, pruned)
        return (self.size * self.size * W * H * self.inch * self.ch * 2 * r + W * H * self.ch * 4,
                W * self.stride, H * self.stride)


class DownSampler(_PlanModule):
    """PB-FCN encoder (model.py:201-232); forward returns (x4, x3, x2, x1, x0)."""

    def __init__(self, planes, noScale, channels=None):
        """channels (extension, default None = the reference's planes-derived widths): output channels of
        conv0..conv8 given explicitly -- the layout of channel-pruned checkpoints (PB_FCN_Channels)."""
        super().__init__()
        self.noScale = noScale
        p = planes
        c = [p // 4, p // 2, p, p * 2, p * 4, p * 4, p * 4, p * 4, p * 2] if channels is None else [int(v) for v in channels]
        if len(c) != 9:
            raise ValueError("DownSampler: channels must list the outputs of conv0..conv8")
        if channels is not None and noScale:
            raise ValueError("DownSampler: an explicit channel list describes the 160x120 encoder (noScale=False)")
        self.conv0 = ConvPoolSimple(3, c[0], 3, 1, 2, 2, False)
        self.conv1 = ConvPoolSimple(c[0], c[1], 3, 2, 1, 1, False)
        self.conv2 = ConvPool(c[1], c[2])
        self.conv_ext = ConvPool(c[2], c[2]) if noScale else None
        self.conv3 = ConvPool(c[2], c[3])
        self.conv4 = ConvPoolSimple(c[3], c[4], 3, 1, 2, 2, False)
        self.conv5 = ConvPoolSimple(c[4], c[5], 3, 1, 2, 2, False)
        self.conv6 = ConvPoolSimple(c[5], c[6], 3, 1, 2, 2, False)
        self.conv7 = ConvPoolSimple(c[6], c[7], 3, 1, 2, 2, False)
        self.conv8 = ConvPoolSimple(c[7], c[8], 3, 1, 2, 2, False)

    def _emit_all(self, b, src):
        x0 = self.conv0._emit(b, src)
        x1 = self.conv1._emit(b, x0)
        x2 = self.conv2._emit(b, x1)

        def belly(a):
            for m in (self.conv3, self.conv4, self.conv5, self.conv6, self.conv7, self.conv8):
                a = m._emit(b, a)
            return a

        if self.noScale:
            x3 = self.conv_ext._emit(b, x2)
            x4 = belly(x3)
        else:
            x3 = belly(x2)
            x4 = None
        return x4, x3, x2, x1, x0

    def _plan_outputs(self, b):
        self._outs = self._emit_all(b, 0)
        return [o for o in self._outs if o is not None]

    def forward(self, x):
        plan = self._get_plan()
        res = list(run_plan(plan, x, self.training))
        return tuple(None if o is None else res.pop(0) for o in self._outs)

    def __getitem__(self, item):
        return self.conv0 if item == 0 else nn.Module()


class DownSamplerThick(_PlanModule):
    def __init__(self, planes):
        super().__init__()
        h = planes // 2
        self.conv0 = ConvPoolSimple(3, h, 3, 1, 2, 2, False)
        self.conv0_1 = ConvPoolSimple(h, h, 3, 1, 2, 2, False)
        self.conv1 = ConvPoolSimple(h, h, 3, 2, 1, 1, False)
        self.conv2 = ConvPoolDouble(h, planes)
        self.conv3 = ConvPoolDouble(planes, planes * 2)
        self.conv4 = ConvPoolSimple(planes * 2, planes * 4, 3, 1, 2, 2, False)
        self.conv5 = ConvPoolSimple(planes * 4, planes * 2, 3, 1, 2, 2, False)

    def _emit_all(self, b, src):
        x0 = self.conv0_1._emit(b, self.conv0._emit(b, src))
        x1 = self.conv1._emit(b, x0)
        x2 = self.conv2._emit(b, x1)
        x3 = self.conv5._emit(b, self.conv4._emit(b, self.conv3._emit(b, x2)))
        return x3, x2, x1, x0

    def _plan_outputs(self, b):
        return list(self._emit_all(b, 0))

    def forward(self, x):
        return tuple(run_plan(self._get_plan(), x, self.training))


class Classifier(_PlanModule):
    def __init__(self, inplanes, num_classes, poolSize=0, kernelSize=1):
        super().__init__()
        self.classifier = nn.Conv2d(inplanes, num_classes, kernel_size=kernelSize, padding=kernelSize // 2)
        self.pool = None
        if poolSize > 1:
            self.pool = nn.MaxPool2d(poolSize)

    def _emit(self, b, src, **kw):
        if self.pool is not None:
            raise NotImplementedError(
                "Classifier with a pooling stage is the patch-classification head (classTrainer.py), "
                "which is outside the segmentation hot path")
        return b.conv(src, self.classifier, None, EPI_NONE)


class PB_FCN(_PlanModule):
    """The net all released pth/bestModelSeg*.pth belong to (model.py:269-309)."""

    def __init__(self, planes, num_classes, kernelSize, noScale, classify):
        super().__init__()
        self.noScale = noScale
        self.classify = classify
        self.img_shape = (240, 320) if self.noScale else (120, 160)
        mult = 2 if noScale else 1
        q = planes // 4
        self.FCN = DownSampler(planes, noScale)
        self.up1 = upSampleTransposeConv(planes * 2, planes)
        self.up2 = upSampleTransposeConv(planes, planes // 2 * mult)
        self.up3 = upSampleTransposeConv(planes // 2 * mult, q * mult)
        self.up4 = upSampleTransposeConv(planes // 2, q) if noScale else None
        self.classifier = Classifier(planes * 2, num_classes, poolSize=(2 if noScale else 4),
                                     kernelSize=kernelSize)
        self.segmenter = Classifier(q, num_classes, kernelSize=kernelSize)

    def _emit(self, b, src, **kw):
        if self.classify:
            raise NotImplementedError("PB_FCN(classify=True) is the patch-classification mode "
                                      "(outside the segmentation hot path)")
        f4, f3, f2, f1, f0 = self.FCN._emit_all(b, src)
        if self.noScale:
            x = self.up1._emit(b, f4, skip=f3)
            x = self.up2._emit(b, x, skip=f2)
            x = self.up3._emit(b, x, skip=f1)
            x = self.up4._emit(b, x, skip=f0)
        else:
            x = self.up1._emit(b, f3, skip=f2)
            x = self.up2._emit(b, x, skip=f1)
            x = self.up3._emit(b, x, skip=f0)
        return self.segmenter._emit(b, x)


class PB_FCN_Channels(PB_FCN):
    """PB_FCN at 160x120 (model.py:269-309) with every layer's width given explicitly: the layout of channel-pruned
    checkpoints, e.g. pth/bestModelSegFinetunedPruned_bu.pth (encoder 16-16-16-32-64-64-128-64-32, decoder 16-16-16,
    head 5x16), which no class of the reference's model.py can load.  Same blocks, same forward, same state_dict key
    names as PB_FCN(planes, C, k, False, 0) (the segmentation head is `segmenter`; legacy files call it `classifier`:
    load_legacy_state_dict); the unused patch-classification head is not built."""

    def __init__(self, enc, ups, num_classes=5, kernelSize=1):
        _PlanModule.__init__(self)
        enc, ups = [int(v) for v in enc], [int(v) for v in ups]
        if len(enc) != 9 or len(ups) != 3:
            raise ValueError("PB_FCN_Channels: enc lists conv0..conv8, ups lists up1..up3")
        if (ups[0], ups[1], ups[2]) != (enc[2], enc[1], enc[0]):
            raise ValueError(f"PB_FCN_Channels: decoder widths {ups} must equal the skip widths "
                             f"{[enc[2], enc[1], enc[0]]} (up_k(x) + f_k, model.py:303-305)")
        self.noScale, self.classify, self.img_shape = False, 0, (120, 160)
        self.enc, self.ups = tuple(enc), tuple(ups)
        self.FCN = DownSampler(0, False, channels=enc)
        self.up1 = upSampleTransposeConv(enc[8], ups[0])
        self.up2 = upSampleTransposeConv(ups[0], ups[1])
        self.up3 = upSampleTransposeConv(ups[1], ups[2])
        self.up4 = None
        self.segmenter = Classifier(ups[2], num_classes, kernelSize=kernelSize)

    @classmethod
    def from_state_dict(cls, state_dict):
        """Build the net a PB_FCN-family checkpoint describes (widths read off the weight shapes) and load it."""
        sd = state_dict
        enc = [sd[f"FCN.conv{i}.{'pool' if i in (2, 3) else 'conv'}.weight"].shape[0] for i in range(9)]
        ups = [sd[f"up{i}.conv.weight"].shape[1] for i in (1, 2, 3)]
        head = "segmenter.classifier.weight" if "segmenter.classifier.weight" in sd else "classifier.classifier.weight"
        m = cls(enc, ups, num_classes=sd[head].shape[0], kernelSize=sd[head].shape[2])
        load_legacy_state_dict(m, sd)
        return m


class FCN(_PlanModule):
    """Thicker variant of pth/bestModelSeg1*.pth (model.py:311-330)."""

    def __init__(self):
        super().__init__()
        planes = 32
        self.FCN = DownSamplerThick(32)
        self.up1 = upSampleTransposeConv(planes * 2, planes)
        self.up2 = upSampleTransposeConv(planes, planes // 2)
        self.up3 = upSampleTransposeConv(planes // 2, planes // 2)
        self.classifier = Classifier(planes // 2, 5, 1)

    def _emit(self, b, src, **kw):
        f3, f2, f1, f0 = self.FCN._emit_all(b, src)
        x = self.up1._emit(b, f3, skip=f2)
        x = self.up2._emit(b, x, skip=f1)
        x = self.up3._emit(b, x, skip=f0)
        return self.classifier._emit(b, x)


class LevelDown(_PlanModule):
    def __init__(self, inplanes, planes, levels, doPool, pool=False):
        super().__init__()
        self.layers = nn.Sequential()
        if pool:
            if doPool:
                self.layers.add_module("Pool", Pool(inplanes, 2))
                levels -= 1
            self.layers.add_module("Conv0", Conv(inplanes, planes, 3, stride=1))
        else:
            self.layers.add_module("Conv0", Conv(inplanes, planes, 3, stride=(2 if doPool else 1)))
        for i in range(levels - 1):
            self.layers.add_module("Conv%d" % (i + 1), Conv(planes, planes, 3))

    def _emit(self, b, src, **kw):
        for m in self.layers:
            src = m._emit(b, src)
        return src


class UltClassifier(_PlanModule):
    def __init__(self, inplanes, nClass, pool, dropout=0.5, size=1):
        super().__init__()
        self.layers = nn.Sequential()
        if pool:
            self.layers.add_module("Pool", nn.AdaptiveAvgPool2d(1))
            self.layers.add_module("DO", nn.Dropout2d(dropout))
        self.layers.add_module("Class", nn.Conv2d(inplanes, nClass, size, padding=size // 2))

    def _emit(self, b, src, **kw):
        if len(self.layers) != 1:
            raise NotImplementedError("UltClassifier(pool=True) is the classification head "
                                      "(outside the segmentation hot path)")
        return b.conv(src, self.layers.Class, None, EPI_NONE)


class ROBO_UNet(_PlanModule):
    """The paper's net (model.py:461-536)."""

    def __init__(self, noScale=False, planes=8, nClass=5, depth=4, levels=2, bellySize=5, bellyPlanes=128,
                 pool=False, v2=False, classSize=1):
        super().__init__()
        self.numClass = nClass
        self.planes = planes
        self.v2 = v2
        self.img_shape = (240, 320) if noScale else (120, 160)
        if noScale:
            depth += 1
        maxDepth = planes * pow(2, depth - 1)

        self.downPart = nn.ModuleList()
        self.downPart.add_module("Level0", LevelDown(3, planes, levels - 1, False, pool))
        for i in range(depth - 1):
            c = planes * pow(2, i)
            self.downPart.add_module("Level%d" % (i + 1), LevelDown(c, c * 2, levels, True, pool))

        self.PB = nn.Sequential()
        if bellySize > 0:
            self.PB.add_module("PB_1", LevelDown(maxDepth, bellyPlanes, bellySize - 1, False))
            self.PB.add_module("PB_2", LevelDown(bellyPlanes, maxDepth, 1, False))

        self.upPart = nn.ModuleList()
        for i in range(depth - 1):
            c = planes * pow(2, depth - 1 - i)
            o = c // 2
            if i > 0 and v2:
                c *= 2
            self.upPart.add_module("Up%d" % i, upSampleTransposeConv(c, o))

        self.segmenter = UltClassifier(planes * 2 if v2 else planes, nClass, False, size=classSize)

    def _emit(self, b, src, **kw):
        downs = [src]
        for level in self.downPart:
            downs.append(level._emit(b, downs[-1]))
        for level in self.PB:
            downs[-1] = level._emit(b, downs[-1])
        up = downs[-1]
        for i, layer in enumerate(self.upPart):
            up = layer._emit(b, up, skip=downs[-(i + 2)], skip_mode="cat" if self.v2 else "add")
        return self.segmenter._emit(b, up)

    def get_computations(self, pruned=False):
        """Analytic per-layer cost list, 2*MAC*(non-zero ratio) + 4/elem (model.py:513-536)."""
        H, W = self.img_shape
        comps = []
        for part in list(self.downPart) + list(self.PB):
            for m in part.layers:
                c, W, H = m.getComp(W, H, pruned)
                comps.append(c)
        for m in self.upPart:
            c, W, H = m.getComp(W, H, pruned)
            comps.append(c)
        comps.append(self.img_shape[0] * self.img_shape[1] * self.numClass * self.planes * 2)
        return comps


class LabelProp(_PlanModule):
    """Two-frame label propagation net (model.py:538-567).  The reference constructor passes an
    8th argument to ConvPoolSimple (a TypeError today) and its forward adds `top` in place into a
    ReLU output; this class is the constructible, autograd-safe equivalent with identical
    forward arithmetic and state_dict keys."""

    def __init__(self, numClass, numPlanes, dropout):
        super().__init__()
        p = numPlanes
        self.pre = ConvPoolSimple(8, p // 4, 3, 1, 1, 1, False)
        self.down1 = ConvPoolSimple(p // 4, p // 2, 3, 2, 1, 1, False)
        self.down2 = ConvPoolSimple(p // 2, p // 2, 3, 2, 1, 1, False)
        self.down3 = ConvPoolSimple(p // 2, p, 3, 2, 1, 1, False)
        self.conv1 = ConvPoolSimple(p, p * 2, 3, 1, 2, 2, False)
        self.conv2 = ConvPoolSimple(p * 2, p * 2, 3, 1, 2, 2, False)
        self.conv3 = ConvPoolSimple(p * 2, p, 3, 1, 2, 2, False)
        self.upConv1 = upSampleTransposeConv(p, p // 2)
        self.upConv2 = upSampleTransposeConv(p // 2, p // 2)
        self.upConv3 = upSampleTransposeConv(p // 2, p // 2)
        self.classifier = nn.Conv2d(p // 2, numClass, 1, padding=0)
        self._top_ch = p // 4

    def _emit(self, b, src, **kw):
        top = self.pre._emit(b, src)
        middle = self.down1._emit(b, top)
        bottom = self.down2._emit(b, middle)
        x = self.down3._emit(b, bottom)
        x = self.conv3._emit(b, self.conv2._emit(b, self.conv1._emit(b, x)))
        x = self.upConv1._emit(b, x, skip=bottom)
        x = self.upConv2._emit(b, x, skip=middle)
        if self.upConv3.ch == self._top_ch:
            x = self.upConv3._emit(b, x, skip=top)
        else:
            x = self.upConv3._emit(b, x, skip=top, skip_mode="partial", skip_ch=self._top_ch)
        return b.conv(x, self.classifier, None, EPI_NONE)


class PB_FCN_2(_PlanModule):
    """model.py:416-459: the ROBO_UNet trunk (one conv in Level0, strided LevelDowns, belly, transposed-conv decoder
    with additive skips) with a fixed option set and an extra image-classification head.  The segmentation branch
    (classify=False) runs on the plan; the classification branch (global average pool + dropout + 1x1 conv on the
    belly output, model.py:452-453) is outside the hot path and raises."""

    def __init__(self, classify, nClass=5, planes=8, depth=4, levels=2, bellySize=5, bellyPlanes=128):
        super().__init__()
        self.classify = classify
        self.img_shape = (120, 160)
        maxDepth = planes * pow(2, depth - 1)
        self.downPart = nn.ModuleList()
        self.downPart.add_module("Level0", LevelDown(3, planes, 1, False))
        for i in range(depth - 1):
            c = planes * pow(2, i)
            self.downPart.add_module("Level%d" % (i + 1), LevelDown(c, c * 2, levels, True))
        self.PB = nn.Sequential()
        self.PB.add_module("PB_1", LevelDown(maxDepth, bellyPlanes, bellySize - 1, False))
        self.PB.add_module("PB_2", LevelDown(bellyPlanes, maxDepth, 1, False))
        self.upPart = nn.ModuleList()
        for i in range(depth - 1):
            c = planes * pow(2, depth - 1 - i)
            self.upPart.add_module("Up%d" % i, upSampleTransposeConv(c, c // 2))
        self.classifier = UltClassifier(maxDepth, nClass, True)
        self.segmenter = UltClassifier(planes, nClass, False)

    def _emit(self, b, src, **kw):
        if self.classify:
            raise NotImplementedError("PB_FCN_2(classify=True) is the image-classification branch "
                                      "(outside the segmentation hot path this package accelerates)")
        downs = [src]
        for level in self.downPart:
            downs.append(level._emit(b, downs[-1]))
        for level in self.PB:
            downs[-1] = level._emit(b, downs[-1])
        up = downs[-1]
        for i, layer in enumerate(self.upPart):
            up = layer._emit(b, up, skip=downs[-(i + 2)])
        return self.segmenter._emit(b, up)


# =============================================================================== checkpoints
def remap_legacy_keys(state_dict):
    """Released pth/bestModelSeg*.pth were saved when PB_FCN's 1x1 segmentation head was the
    attribute `classifier`; today that head is `segmenter` and `classifier` is the (unused)
    patch-classification head (model.py:288-289).  Returns a copy with
    classifier.classifier.* renamed to segmenter.classifier.*."""
    out = {}
    for k, v in state_dict.items():
        if k.startswith("classifier.classifier."):
            out["segmenter." + k[len("classifier."):]] = v
        else:
            out[k] = v
    return out


def load_legacy_state_dict(model: nn.Module, state_dict, strict: bool = True):
    """Load a pre-0.4.1 checkpoint (no num_batches_tracked; PB_FCN legacy head name).
    Returns (missing, unexpected) like load_state_dict(strict=False); with strict=True anything
    missing other than num_batches_tracked / PB_FCN's unused classification head raises."""
    sd = dict(state_dict)
    if isinstance(model, PB_FCN) and "segmenter.classifier.weight" not in sd \
            and "classifier.classifier.weight" in sd \
            and tuple(sd["classifier.classifier.weight"].shape) == tuple(model.segmenter.classifier.weight.shape):
        sd = remap_legacy_keys(sd)
    res = model.load_state_dict(sd, strict=False)
    missing = [k for k in res.missing_keys if not k.endswith("num_batches_tracked")]
    if isinstance(model, PB_FCN):
        missing = [k for k in missing if not k.startswith("classifier.")]
    if strict and (missing or res.unexpected_keys):
        raise RuntimeError(f"load_legacy_state_dict: missing={missing} unexpected={res.unexpected_keys}")
    return missing, list(res.unexpected_keys)
