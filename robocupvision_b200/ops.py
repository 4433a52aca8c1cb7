"""Tensor-level wrappers over the C ABI (one function per rcv_* entry point).

PyTorch is plumbing here: it owns device memory (caching allocator) and the current
stream; every function below enqueues exactly the named librcv_b200 kernels on
``torch.cuda.current_stream()``.  Inputs must be CUDA tensors -- there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (DET_CE_FWD, DET_CE_WEIGHT_SUM, DET_DICE_FWD, DET_L1_SUM, ENGINE_DIRECT, ENGINE_NARROW, ENGINE_SIMT, ENGINE_UMMA, EPI_AFFINE, EPI_AFFINE_RELU, EPI_NONE,
                   EPI_RELU, EPI_RELU_AFFINE, MATH_AUTO, MATH_BF16, MATH_FP32, MATH_TF32, MATH_TF32X3, PACK_DGRAD,
                   PACK_FWD, ConvDesc)

__all__ = [
    "ConvGeom", "conv_fwd", "conv_dgrad", "conv_wgrad", "conv_pack", "conv_packed_bytes", "conv_workspace_bytes", "new_workspace", "conv_takes_partial_residual", "conv_uses_tensor_cores", "conv_engine", "conv_normalises_on_load", "PackTable", "bn_finalize_apply", "PACK_FWD", "PACK_DGRAD", "bn_finalize", "bn_fold", "bn_apply",
    "bn_bwd", "bn_bwd_reduce", "bn_bwd_apply", "relu_bwd", "channel_sum", "maxpool2x2_fwd", "maxpool2x2_bwd", "maxunpool2x2", "maxunpool2x2_bwd", "upsample_bilinear2x", "upsample_bilinear2x_bwd", "ce_fwd", "ce_bwd",
    "confusion", "metric_tail", "mask_label_lut", "mask_label_", "label_to_pred", "lp_assemble", "augment", "color_jitter_params", "dice_fwd", "dice_bwd", "dice_loss", "head_dice_fwd", "head_dice_train", "adam_l1_step", "sgd_step", "det_scratch_bytes", "det_scratch", "zero_", "zeros", "counter_add", "launch_count", "reset_launch_count",
    "EPI_NONE", "EPI_RELU", "EPI_RELU_AFFINE", "EPI_AFFINE_RELU", "EPI_AFFINE",
    "DET_CE_FWD", "DET_CE_WEIGHT_SUM", "DET_DICE_FWD", "DET_L1_SUM",
    "MATH_FP32", "MATH_TF32X3", "MATH_AUTO", "MATH_TF32", "MATH_BF16", "ENGINE_SIMT", "ENGINE_DIRECT", "ENGINE_UMMA", "ENGINE_NARROW",
]

_launches = 0  # kernels enqueued through this module (bench.py's gpu_launches)


def launch_count() -> int:
    return _launches


def reset_launch_count() -> None:
    global _launches
    _launches = 0


def _call(name: str, nkernels: int, *args) -> None:
    global _launches
    _launches += nkernels
    _lib.call(name, *args)


def _chk(t: torch.Tensor, dtype=torch.float32, name: str = "tensor") -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"robocupvision_b200: {name} must be a CUDA tensor "
                           "(there is no CPU path; the oracle lives in oracle/ for tests only)")
    if t.dtype != dtype:
        raise TypeError(f"robocupvision_b200: {name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone()
    return t


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class ConvGeom:
    """Geometry of one nn.Conv2d / nn.ConvTranspose2d on the hot path."""

    __slots__ = ("cin", "cout", "k", "stride", "pad", "dil", "transposed")

    def __init__(self, cin, cout, k=3, stride=1, pad=1, dil=1, transposed=False):
        self.cin, self.cout, self.k = int(cin), int(cout), int(k)
        self.stride, self.pad, self.dil = int(stride), int(pad), int(dil)
        self.transposed = bool(transposed)

    @staticmethod
    def of(m: torch.nn.Module) -> "ConvGeom":
        if isinstance(m, torch.nn.ConvTranspose2d):
            if not (m.kernel_size == (3, 3) and m.stride == (2, 2) and m.padding == (1, 1)
                    and m.output_padding == (1, 1) and m.dilation == (1, 1) and m.groups == 1):
                raise NotImplementedError(f"unsupported ConvTranspose2d geometry: {m}")
            return ConvGeom(m.in_channels, m.out_channels, 3, 2, 1, 1, True)
        if isinstance(m, torch.nn.Conv2d):
            k, s, p, d = m.kernel_size, m.stride, m.padding, m.dilation
            if not (k[0] == k[1] and s[0] == s[1] and p[0] == p[1] and d[0] == d[1] and m.groups == 1
                    and m.padding_mode == "zeros"):
                raise NotImplementedError(f"unsupported Conv2d geometry: {m}")
            return ConvGeom(m.in_channels, m.out_channels, k[0], s[0], p[0], d[0], False)
        raise TypeError(f"not a convolution module: {type(m)}")

    def out_hw(self, h: int, w: int) -> Tuple[int, int]:
        if self.transposed:
            return 2 * h, 2 * w
        e = self.dil * (self.k - 1) + 1
        return (h + 2 * self.pad - e) // self.stride + 1, (w + 2 * self.pad - e) // self.stride + 1

    def weight_shape(self):
        if self.transposed:
            return (self.cin, self.cout, 3, 3)
        return (self.cout, self.cin, self.k, self.k)

    def desc(self, n: int, h: int, w: int, epilogue: int = EPI_NONE, math: int = MATH_FP32) -> ConvDesc:
        return ConvDesc(n, self.cin, h, w, self.cout, self.k, self.stride, self.pad, self.dil,
                        1 if self.transposed else 0, epilogue, math)


# --------------------------------------------------------------------------- conv family
NOMINAL_NHW = (1, 16, 16)


def conv_packed_bytes(g: ConvGeom, direction: int, math: int = MATH_AUTO, nhw=NOMINAL_NHW) -> int:
    """Bytes of the layer's weight panel.  The panel layout follows the kernel the layer runs on AT THE INPUT SIZE
    `nhw` = (N, H, W): RCV_MATH_BF16 panels are bf16 for the layers the halo-staged kernel runs at that size (rows too
    long for the kernel's patch fall to the single-pass tf32 kernels and their fp32 panels).  Pass the real size; the
    nominal default is only good outside the bf16 mode."""
    d = g.desc(*nhw, EPI_NONE, math)
    n = _lib.load().rcv_conv_packed_bytes(C.byref(d), int(direction))
    if n == 0:
        raise _lib.RcvError("rcv_conv_packed_bytes", -1, _lib.load().rcv_last_error().decode())
    return int(n)


def conv_workspace_bytes(g: ConvGeom, n: int, h: int, w: int, direction: int = PACK_FWD, math: int = MATH_AUTO) -> int:
    """Bytes of scratch conv_fwd / conv_dgrad can use for this layer at this size (0: none); see `workspace`."""
    d = g.desc(n, h, w, EPI_NONE, math)
    return int(_lib.load().rcv_conv_workspace_bytes(C.byref(d), int(direction)))


def new_workspace(nbytes: int, device) -> torch.Tensor:
    """A zero-filled scratch buffer for the `workspace` argument of conv_fwd / conv_dgrad (rcv_conv_desc::workspace:
    zero-filled once by the caller, then owned by ONE stream of convolution launches at a time)."""
    return zeros(max(int(nbytes), 1024), torch.uint8, device)


def _with_ws(d: ConvDesc, workspace):
    if workspace is not None:
        d.workspace = workspace.data_ptr()
        d.workspace_bytes = workspace.numel() * workspace.element_size()
    return d


def conv_takes_partial_residual(g: ConvGeom, n: int, h: int, w: int, math: int = MATH_AUTO) -> bool:
    """Can conv_fwd add a residual that has fewer channels than the output (rcv_conv_desc::res_channels)?  Only the
    narrow-layer engine does."""
    return conv_engine(g, n, h, w, PACK_FWD, math) == ENGINE_NARROW


def conv_uses_tensor_cores(g: ConvGeom, direction: int, math: int = MATH_AUTO) -> bool:
    d = g.desc(1, 2, 2, EPI_NONE, math)
    return bool(_lib.load().rcv_conv_uses_tensor_cores(C.byref(d), int(direction)))


def conv_engine(g: ConvGeom, n: int, h: int, w: int, direction: int = PACK_FWD, math: int = MATH_AUTO) -> int:
    """rcv_engine the layer dispatches to at this size (ENGINE_SIMT / DIRECT / UMMA / NARROW)."""
    d = g.desc(n, h, w, EPI_NONE, math)
    e = _lib.load().rcv_conv_engine(C.byref(d), int(direction))
    if e < 0:
        raise _lib.RcvError("rcv_conv_engine", e, _lib.load().rcv_last_error().decode())
    return int(e)


def conv_pack(g: ConvGeom, w, direction: int, out=None, math: int = MATH_AUTO, nhw=NOMINAL_NHW):
    """Weight panel of the tensor-core engine for `w` in math mode `math` (one launch); `out` is reused when given.
    nhw: the input size the panel will be used at (see conv_packed_bytes)."""
    w = _chk(w, name="weight")
    if tuple(w.shape) != g.weight_shape():
        raise ValueError(f"conv_pack: w {tuple(w.shape)} does not match geometry")
    if out is None:
        out = torch.empty(conv_packed_bytes(g, direction, math, nhw), device=w.device, dtype=torch.uint8)
    d = g.desc(*nhw, EPI_NONE, math)
    _call("rcv_conv_pack", 1, C.byref(d), int(direction), _ptr(w), _ptr(out), _stream())
    return out


class PackTable:
    """Device-resident job table that re-packs the weight panels of many layers in one launch
    (rcv_conv_pack_table_*).  Valid while every weight / panel pointer it was built from is."""

    def __init__(self, jobs, math: int = MATH_AUTO, sizes=None):
        """jobs: list of (ConvGeom, direction, weight tensor, packed uint8 tensor); sizes: the (N, H, W) each panel is
        used at (see conv_packed_bytes), nominal when omitted."""
        n = len(jobs)
        lib = _lib.load()
        sizes = sizes or [NOMINAL_NHW] * n
        descs = (ConvDesc * n)(*[g.desc(*sz, EPI_NONE, math) for (g, _, _, _), sz in zip(jobs, sizes)])
        dirs = (C.c_int32 * n)(*[int(d) for _, d, _, _ in jobs])
        ws = (C.c_void_p * n)(*[w.data_ptr() for _, _, w, _ in jobs])
        ps = (C.c_void_p * n)(*[pk.data_ptr() for _, _, _, pk in jobs])
        nbytes = int(lib.rcv_conv_pack_table_bytes(n))
        host = torch.empty(nbytes, dtype=torch.uint8)
        total = C.c_int64(0)
        _lib.call("rcv_conv_pack_table_build", n, descs, dirs, ws, ps, C.c_void_p(host.data_ptr()), C.byref(total))
        self.n, self.total = n, int(total.value)
        self.key = tuple((w.data_ptr(), pk.data_ptr()) for _, _, w, pk in jobs)
        self.table = host.to(jobs[0][2].device)

    def run(self):
        _call("rcv_conv_pack_table_run", 1, _ptr(self.table), self.n, self.total, _stream())


def _res_channels(residual, c):
    """Channels of a residual tensor for the `res_channels` arguments: 0 = all; fewer = a partial skip (added to the
    first channels only, LabelProp model.py:565)."""
    if residual is None or residual.shape[1] == c:
        return 0
    if residual.shape[1] > c:
        raise ValueError("residual has more channels than the output")
    return int(residual.shape[1])


def bn_finalize_apply(z, stats, gamma, beta, running_mean, running_var, momentum, eps, relu, residual=None,
                      num_batches_tracked=None, count=None):
    """Train-mode BatchNorm forward in one launch -> (y, scale, shift, mean, invstd).  A residual with fewer channels
    than z is added to the first channels only.  count: elements per channel the statistics were summed over
    (rcv_bn_finalize_apply_count; statistics summed over the ranks of a global batch), default N*HW of z."""
    z = _chk(z, name="z")
    n, c = z.shape[0], z.shape[1]
    hw = z.numel() // (n * c)
    buf = torch.empty((4, c), device=z.device, dtype=torch.float32)
    y = torch.empty_like(z)
    if residual is not None:
        residual = _chk(residual, name="residual")
    head = ("rcv_bn_finalize_apply", 1, n, c, hw) if count is None else (
        "rcv_bn_finalize_apply_count", 1, n, c, hw, int(count))
    _call(*head, _ptr(stats), _ptr(gamma), _ptr(beta), _ptr(running_mean),
          _ptr(running_var), float(momentum), float(eps), _ptr(z), 1 if relu else 0, _ptr(residual),
          _res_channels(residual, c), _ptr(y),
          _ptr(buf[0]), _ptr(buf[1]), _ptr(buf[2]), _ptr(buf[3]), _ptr(num_batches_tracked), _stream())
    return y, buf[0], buf[1], buf[2], buf[3]


def _packed_for(g, w, wpacked, math, direction, nhw):
    if wpacked is None and math == MATH_TF32X3:
        wpacked = conv_pack(g, w, direction, math=math, nhw=nhw)
    return wpacked


def conv_normalises_on_load(g: ConvGeom, n: int, h: int, w: int, math: int = MATH_AUTO) -> bool:
    """Would conv_fwd(..., in_affine=...) be accepted for this layer at this size (halo-staged tensor-core kernel)."""
    d = g.desc(n, h, w, EPI_NONE, math)
    return bool(_lib.load().rcv_conv_normalises_on_load(C.byref(d)))


def conv_fwd(g: ConvGeom, x, w, bias=None, epilogue=EPI_NONE, scale=None, shift=None, residual=None,
             stats=None, math=MATH_FP32, out=None, wpacked=None, in_affine=None, workspace=None):
    x = _chk(x, name="x")
    w = _chk(w, name="weight")
    n, cin, h, wd = x.shape
    wpacked = _packed_for(g, w, wpacked, math, PACK_FWD, (n, h, wd))
    if cin != g.cin or tuple(w.shape) != g.weight_shape():
        raise ValueError(f"conv_fwd: x {tuple(x.shape)} / w {tuple(w.shape)} do not match geometry")
    ho, wo = g.out_hw(h, wd)
    y = out if out is not None else torch.empty((n, g.cout, ho, wo), device=x.device, dtype=torch.float32)
    if residual is not None:
        residual = _chk(residual, name="residual")
        # fewer channels than the output = a partial skip (first channels only; narrow-layer engine, see
        # conv_takes_partial_residual)
        if (residual.shape[0], *residual.shape[2:]) != (y.shape[0], *y.shape[2:]) or residual.shape[1] > y.shape[1]:
            raise ValueError(f"conv_fwd: residual {tuple(residual.shape)} does not fit output {tuple(y.shape)}")
    for t, nm in ((bias, "bias"), (scale, "scale"), (shift, "shift")):
        if t is not None and (t.numel() != g.cout or not t.is_cuda or t.dtype != torch.float32):
            raise ValueError(f"conv_fwd: bad {nm}")
    if stats is not None and (stats.dtype != torch.float64 or stats.numel() != 2 * g.cout):
        raise ValueError("conv_fwd: stats must be float64[2*Cout]")
    d = _with_ws(g.desc(n, h, wd, epilogue, math), workspace)
    d.res_channels = _res_channels(residual, g.cout)
    if in_affine is not None:
        # (in_scale, in_shift, relu): the BatchNorm of the block that produced x, applied on load (rcv_conv_fwd_nl)
        isc, ish, irelu = in_affine
        if isc.numel() != g.cin or ish.numel() != g.cin:
            raise ValueError("conv_fwd: in_affine must have Cin entries")
        _call("rcv_conv_fwd_nl", 1, C.byref(d), _ptr(x), _ptr(isc), _ptr(ish), 1 if irelu else 0, _ptr(w),
              _ptr(wpacked), _ptr(bias), _ptr(scale), _ptr(shift), _ptr(residual), _ptr(y), _ptr(stats), _stream())
        return y
    _call("rcv_conv_fwd", 1, C.byref(d), _ptr(x), _ptr(w), _ptr(wpacked), _ptr(bias), _ptr(scale), _ptr(shift),
          _ptr(residual), _ptr(y), _ptr(stats), _stream())
    return y


def conv_dgrad(g: ConvGeom, dy, w, in_hw: Tuple[int, int], residual=None, math=MATH_FP32, out=None,
               wpacked=None, workspace=None):
    """Input gradient; `residual` (shape of dx; may be `out`) is the gradient the same tensor
    receives from a second consumer and is added in the kernel epilogue."""
    dy = _chk(dy, name="dy")
    w = _chk(w, name="weight")
    n = dy.shape[0]
    h, wd = in_hw
    wpacked = _packed_for(g, w, wpacked, math, PACK_DGRAD, (n, h, wd))
    if tuple(dy.shape[1:]) != (g.cout, *g.out_hw(h, wd)):
        raise ValueError(f"conv_dgrad: dy {tuple(dy.shape)} does not match geometry for input {in_hw}")
    d = _with_ws(g.desc(n, h, wd, EPI_NONE, math), workspace)
    dx = out if out is not None else torch.empty((n, g.cin, h, wd), device=dy.device, dtype=torch.float32)
    if residual is not None:
        residual = _chk(residual, name="residual")
        if residual.shape != dx.shape:
            raise ValueError("conv_dgrad: residual shape mismatch")
    _call("rcv_conv_dgrad", 1, C.byref(d), _ptr(dy), _ptr(w), _ptr(wpacked), _ptr(residual), _ptr(dx), _stream())
    return dx


def conv_wgrad_normalises_on_load(g: ConvGeom, n: int, h: int, w: int, math: int = MATH_AUTO) -> bool:
    """Would conv_wgrad(..., in_affine=...) be accepted for this layer at this size (tensor-core quad gather)."""
    d = g.desc(n, h, w, EPI_NONE, math)
    return bool(_lib.load().rcv_conv_wgrad_normalises_on_load(C.byref(d)))


def conv_wgrad(g: ConvGeom, x, dy, dw=None, dbias=None, want_bias=False, math=MATH_FP32, in_affine=None):
    """Weight (and bias) gradient, accumulated into dw/dbias (zero-filled if not given).  in_affine = (scale, shift,
    relu): the gradient with respect to a conv of relu?(scale*x + shift) (rcv_conv_wgrad_nl)."""
    x = _chk(x, name="x")
    dy = _chk(dy, name="dy")
    n, _, h, wd = x.shape
    if dw is None:
        dw = zeros(g.weight_shape(), torch.float32, x.device)
    if dbias is None and want_bias:
        dbias = zeros(g.cout, torch.float32, x.device)
    d = g.desc(n, h, wd, EPI_NONE, math)
    if in_affine is not None:
        isc, ish, irelu = in_affine
        if isc.numel() != g.cin or ish.numel() != g.cin:
            raise ValueError("conv_wgrad: in_affine must have Cin entries")
        _call("rcv_conv_wgrad_nl", 1, C.byref(d), _ptr(x), _ptr(isc), _ptr(ish), 1 if irelu else 0, _ptr(dy),
              _ptr(dw), _ptr(dbias), _stream())
        return dw, dbias
    _call("rcv_conv_wgrad", 2 if (g.transposed and dbias is not None) else 1, C.byref(d), _ptr(x),
          _ptr(dy), _ptr(dw), _ptr(dbias), _stream())
    return dw, dbias


# --------------------------------------------------------------------------- batch norm
def bn_finalize(stats, count, gamma, beta, running_mean, running_var, momentum, eps, num_batches_tracked=None):
    c = stats.numel() // 2
    dev = stats.device
    buf = torch.empty((4, c), device=dev, dtype=torch.float32)
    scale, shift, mean, invstd = buf[0], buf[1], buf[2], buf[3]
    _call("rcv_bn_finalize", 1, c, int(count), _ptr(stats), _ptr(gamma), _ptr(beta), _ptr(running_mean),
          _ptr(running_var), float(momentum), float(eps), _ptr(scale), _ptr(shift), _ptr(mean),
          _ptr(invstd), _ptr(num_batches_tracked), _stream())
    return scale, shift, mean, invstd


def bn_fold(gamma, beta, mean, var, eps):
    c = mean.numel()
    buf = torch.empty((2, c), device=mean.device, dtype=torch.float32)
    _call("rcv_bn_fold", 1, c, _ptr(gamma), _ptr(beta), _ptr(mean), _ptr(var), float(eps), _ptr(buf[0]),
          _ptr(buf[1]), _stream())
    return buf[0], buf[1]


def bn_apply(z, scale, shift, relu: bool, residual=None, out=None):
    z = _chk(z, name="z")
    n, c = z.shape[0], z.shape[1]
    hw = z.numel() // (n * c)
    y = out if out is not None else torch.empty_like(z)
    if residual is not None:
        residual = _chk(residual, name="residual")
    _call("rcv_bn_apply", 1, n, c, hw, _ptr(z), _ptr(scale), _ptr(shift), 1 if relu else 0, _ptr(residual),
          _res_channels(residual, c), _ptr(y), _stream())
    return y


def bn_bwd(order: int, dy, z, scale, shift, mean, invstd, dgamma=None, dbeta=None, dbias=None,
           want_dbias: bool = False, sums=None):
    """-> (dconv, dgamma, dbeta, dbias|None).  Two passes: reduce, apply.  dgamma/dbeta/dbias are
    accumulated into when given (zero-filled buffers otherwise); sums is float64[2C] zeros."""
    dy = _chk(dy, name="dy")
    z = _chk(z, name="z")
    n, c = z.shape[0], z.shape[1]
    hw = z.numel() // (n * c)
    if sums is None:
        sums = zeros(2 * c, torch.float64, z.device)
    if dgamma is None or dbeta is None or (want_dbias and dbias is None):
        small = zeros((3, c), torch.float32, z.device)
        dgamma = small[0] if dgamma is None else dgamma
        dbeta = small[1] if dbeta is None else dbeta
        if want_dbias and dbias is None:
            dbias = small[2]
    dconv = torch.empty_like(z)
    st = _stream()
    # one cluster launch where the tensor suits it, else reduce + apply (the library decides; either way <= 2 kernels)
    fused = bool(_lib.load().rcv_bn_bwd_is_fused(n, c, hw)) and not ((dy.data_ptr() | z.data_ptr()) & 15)
    _call("rcv_bn_bwd", 1 if fused else 2, n, c, hw, order, _ptr(dy), _ptr(z), _ptr(scale), _ptr(shift), _ptr(mean),
          _ptr(invstd), _ptr(sums), _ptr(dconv), _ptr(dgamma), _ptr(dbeta), _ptr(dbias), st)
    return dconv, dgamma, dbeta, dbias


def bn_bwd_reduce(order: int, dy, z, scale, shift, mean, invstd, sums) -> None:
    """Pass 1 of the BatchNorm backward alone: sums[c] += sum(g), sums[C+c] += sum(g*xhat) (float64[2C], zeroed by the
    caller).  With bn_bwd_apply it is bn_bwd in two launches, with the sums in memory between them (a global batch
    averages them over the ranks there)."""
    dy = _chk(dy, name="dy")
    z = _chk(z, name="z")
    n, c = z.shape[0], z.shape[1]
    hw = z.numel() // (n * c)
    if sums.dtype != torch.float64 or sums.numel() != 2 * c:
        raise ValueError("bn_bwd_reduce: sums must be float64[2*C]")
    _call("rcv_bn_bwd_reduce", 1, n, c, hw, order, _ptr(dy), _ptr(z), _ptr(scale), _ptr(shift), _ptr(mean),
          _ptr(invstd), _ptr(sums), _stream())


def bn_bwd_apply(order: int, dy, z, scale, shift, mean, invstd, sums, dgamma=None, dbeta=None, dbias=None):
    """Pass 2 of the BatchNorm backward: -> dconv from the channel sums of bn_bwd_reduce (means = sums / (N*HW) of
    this z); dgamma += sums[C:], dbeta += sums[:C], dbias += sum(dconv) where given."""
    dy = _chk(dy, name="dy")
    z = _chk(z, name="z")
    n, c = z.shape[0], z.shape[1]
    hw = z.numel() // (n * c)
    if sums.dtype != torch.float64 or sums.numel() != 2 * c:
        raise ValueError("bn_bwd_apply: sums must be float64[2*C]")
    dconv = torch.empty_like(z)
    _call("rcv_bn_bwd_apply", 1, n, c, hw, order, _ptr(dy), _ptr(z), _ptr(scale), _ptr(shift), _ptr(mean),
          _ptr(invstd), _ptr(sums), _ptr(dconv), _ptr(dgamma), _ptr(dbeta), _ptr(dbias), _stream())
    return dconv


def relu_bwd(dy, y):
    dy = _chk(dy, name="dy")
    y = _chk(y, name="y")
    dx = torch.empty_like(dy)
    _call("rcv_relu_bwd", 1, dy.numel(), _ptr(dy), _ptr(y), _ptr(dx), _stream())
    return dx


def channel_sum(dy, out=None):
    dy = _chk(dy, name="dy")
    n, c = dy.shape[0], dy.shape[1]
    hw = dy.numel() // (n * c)
    if out is None:
        out = zeros(c, torch.float32, dy.device)
    _call("rcv_channel_sum", 1, n, c, hw, _ptr(dy), _ptr(out), _stream())
    return out


# --------------------------------------------------------------------------- pooling
def maxpool2x2_fwd(x, want_idx=False, want_code=True):
    x = _chk(x, name="x")
    n, c, h, w = x.shape
    y = torch.empty((n, c, h // 2, w // 2), device=x.device, dtype=torch.float32)
    idx = torch.empty(y.shape, device=x.device, dtype=torch.int64) if want_idx else None
    code = torch.empty(y.shape, device=x.device, dtype=torch.uint8) if want_code else None
    _call("rcv_maxpool2x2_fwd", 1, n, c, h, w, _ptr(x), _ptr(y), _ptr(idx), _ptr(code), _stream())
    return y, idx, code


def maxpool2x2_bwd(dy, code, in_hw):
    dy = _chk(dy, name="dy")
    n, c = dy.shape[0], dy.shape[1]
    h, w = in_hw
    dx = torch.empty((n, c, h, w), device=dy.device, dtype=torch.float32)
    _call("rcv_maxpool2x2_bwd", 1, n, c, h, w, _ptr(dy), _ptr(code), _ptr(dx), _stream())
    return dx


def maxunpool2x2(y, idx=None, code=None, skip=None):
    """F.max_unpool2d(y, idx, 2, 2) (+ skip) from the int64 indices or the uint8 window codes of maxpool2x2_fwd."""
    y = _chk(y, name="y")
    if idx is None and code is None:
        raise ValueError("maxunpool2x2: needs idx or code")
    n, c, ho, wo = y.shape
    out = torch.empty((n, c, 2 * ho, 2 * wo), device=y.device, dtype=torch.float32)
    if skip is not None:
        skip = _chk(skip, name="skip")
        if skip.shape != out.shape:
            raise ValueError("maxunpool2x2: skip shape mismatch")
    _call("rcv_maxunpool2x2_fwd", 1, n, c, 2 * ho, 2 * wo, _ptr(y), _ptr(idx), _ptr(code), _ptr(skip), _ptr(out), _stream())
    return out


def maxunpool2x2_bwd(dout, idx=None, code=None):
    dout = _chk(dout, name="dout")
    n, c, h, w = dout.shape
    dy = torch.empty((n, c, h // 2, w // 2), device=dout.device, dtype=torch.float32)
    _call("rcv_maxunpool2x2_bwd", 1, n, c, h, w, _ptr(dout), _ptr(idx), _ptr(code), _ptr(dy), _stream())
    return dy


def upsample_bilinear2x(x, skip=None):
    """F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False) (+ skip)."""
    x = _chk(x, name="x")
    n, c, h, w = x.shape
    out = torch.empty((n, c, 2 * h, 2 * w), device=x.device, dtype=torch.float32)
    if skip is not None:
        skip = _chk(skip, name="skip")
        if skip.shape != out.shape:
            raise ValueError("upsample_bilinear2x: skip shape mismatch")
    _call("rcv_upsample_bilinear2x_fwd", 1, n, c, h, w, _ptr(x), _ptr(skip), _ptr(out), _stream())
    return out


def upsample_bilinear2x_bwd(dout):
    dout = _chk(dout, name="dout")
    n, c, h2, w2 = dout.shape
    dx = torch.empty((n, c, h2 // 2, w2 // 2), device=dout.device, dtype=torch.float32)
    _call("rcv_upsample_bilinear2x_bwd", 1, n, c, h2 // 2, w2 // 2, _ptr(dout), _ptr(dx), _stream())
    return dx


def head_ce_supported(cin: int, classes: int) -> bool:
    """True if head_ce_train has a kernel for a `classes`-way 1x1 classifier over `cin` channels."""
    return bool(_lib.load().rcv_head_ce_supported(int(cin), int(classes)))


def ce_weight_sum(target, class_w, out, classes: int, scratch=None) -> None:
    """out[0] += sum over pixels of class_w[target] (the normaliser of the weighted mean loss; labels only).
    scratch: det_scratch(DET_CE_WEIGHT_SUM, ...) for the fixed-order sum (rcv_ce_weight_sum_det)."""
    target = _chk(target, torch.int64, "target")
    if scratch is None:
        _call("rcv_ce_weight_sum", 1, int(classes), target.numel(), _ptr(target), _ptr(class_w), _ptr(out), _stream())
    else:
        _call("rcv_ce_weight_sum_det", 1, int(classes), target.numel(), _ptr(target), _ptr(class_w), _ptr(out),
              *_scratch_args(scratch), _stream())


def head_ce_train(feat, weight, bias, target, class_w, sums, corr, dweight, dbias):
    """The classifier head of a training step in one pass (rcv_head_ce_train): -> dfeat.  sums: float64[2] with
    sums[1] already holding the weight sum (ce_weight_sum); sums[0], corr, dweight, dbias are accumulated into."""
    feat = _chk(feat, name="feat")
    target = _chk(target, torch.int64, "target")
    n, cin, h, w_ = feat.shape
    c = weight.shape[0]
    if weight.numel() != c * cin or tuple(target.shape) != (n, h, w_):
        raise ValueError(f"head_ce_train: feat {tuple(feat.shape)}, weight {tuple(weight.shape)}, target {tuple(target.shape)}")
    dfeat = torch.empty_like(feat)
    _call("rcv_head_ce_train", 1, n, cin, c, h * w_, _ptr(feat), _ptr(weight), _ptr(bias), _ptr(target), _ptr(class_w),
          None, _ptr(sums), _ptr(corr), _ptr(dfeat), _ptr(dweight), _ptr(dbias), _stream())
    return dfeat


def _head_shapes(fn, feat, weight, target):
    n, cin, h, w_ = feat.shape
    c = weight.shape[0]
    if weight.numel() != c * cin or tuple(target.shape) != (n, h, w_):
        raise ValueError(f"{fn}: feat {tuple(feat.shape)}, weight {tuple(weight.shape)}, target {tuple(target.shape)}")
    return n, cin, c, h * w_


def head_dice_fwd(feat, weight, bias, target, sums, corr) -> None:
    """Pass 1 of the Dice-loss classifier head (rcv_head_dice_fwd): sums float64[2C] += the soft intersection and
    cardinality of softmax(weight feat + bias) against the labels; corr int64[1] (or None) += correct pixels."""
    feat = _chk(feat, name="feat")
    target = _chk(target, torch.int64, "target")
    n, cin, c, hw = _head_shapes("head_dice_fwd", feat, weight, target)
    _call("rcv_head_dice_fwd", 1, n, cin, c, hw, _ptr(feat), _ptr(weight), _ptr(bias), _ptr(target), _ptr(sums),
          _ptr(corr), _stream())


def head_dice_train(feat, weight, bias, target, weights, sums, eps, loss, dweight, dbias, gscale=None):
    """Pass 2 of the Dice-loss classifier head (rcv_head_dice_train), after head_dice_fwd filled `sums`: -> dfeat.
    weights: the normalised Dice weights float32[C] (or None); loss: float64[2] (or None) <- [dice loss, 1.0];
    dweight, dbias are accumulated into."""
    feat = _chk(feat, name="feat")
    target = _chk(target, torch.int64, "target")
    n, cin, c, hw = _head_shapes("head_dice_train", feat, weight, target)
    if gscale is not None:
        gscale = _chk(gscale.reshape(1).to(torch.float32), name="gscale")
    dfeat = torch.empty_like(feat)
    _call("rcv_head_dice_train", 1, n, cin, c, hw, _ptr(feat), _ptr(weight), _ptr(bias), _ptr(target), _ptr(weights),
          _ptr(sums), float(eps), _ptr(gscale), _ptr(loss), _ptr(dfeat), _ptr(dweight), _ptr(dbias), _stream())
    return dfeat


def dice_loss(sums, weights, eps, loss) -> None:
    """loss float64[2] <- [1 - mean_c(2 w_c I_c / (K_c + eps)), 1.0] from dice_fwd's sums (rcv_dice_loss)."""
    _call("rcv_dice_loss", 1, sums.numel() // 2, _ptr(sums), _ptr(weights), float(eps), _ptr(loss), _stream())


def channel_slice(x, offset: int, count: int) -> torch.Tensor:
    """x[:, offset:offset+count] as a dense tensor (the gradient halves of a concatenated skip, the gradient of
    LabelProp's partial skip)."""
    x = _chk(x, name="x")
    n, c, h, w = x.shape
    out = torch.empty((n, count, h, w), device=x.device, dtype=torch.float32)
    _call("rcv_channel_copy", 1, n, h * w, count, _ptr(x), c, offset, _ptr(out), count, 0, _stream())
    return out


def concat_channels(a, b) -> torch.Tensor:
    """torch.cat([a, b], 1) (ROBO_UNet --v2, model.py:507)."""
    a, b = _chk(a, name="a"), _chk(b, name="b")
    if a.shape[0] != b.shape[0] or a.shape[2:] != b.shape[2:]:
        raise ValueError(f"concat_channels: {tuple(a.shape)} vs {tuple(b.shape)}")
    n, ca, h, w = a.shape
    cb = b.shape[1]
    out = torch.empty((n, ca + cb, h, w), device=a.device, dtype=torch.float32)
    _call("rcv_channel_copy", 1, n, h * w, ca, _ptr(a), ca, 0, _ptr(out), ca + cb, 0, _stream())
    _call("rcv_channel_copy", 1, n, h * w, cb, _ptr(b), cb, 0, _ptr(out), ca + cb, ca, _stream())
    return out


# --------------------------------------------------------------------------- loss / metrics
def ce_fwd(logits, target, class_w=None, want_argmax=False, want_conf=False, want_correct=False, sums=None,
           corr=None, scratch=None):
    """-> (loss_sums float64[2], argmax|None, conf int64[N,C,C]|None, correct int64[1]|None).  sums / corr:
    caller-zeroed accumulators to use instead of fresh ones.  scratch: det_scratch(DET_CE_FWD, ...) for loss sums in
    fixed order (rcv_ce_fwd_det)."""
    logits = _chk(logits, name="logits")
    target = _chk(target, torch.int64, "target")
    n, c = logits.shape[0], logits.shape[1]
    hw = logits.numel() // (n * c)
    if target.numel() != n * hw:
        raise ValueError(f"ce_fwd: target {tuple(target.shape)} does not match logits {tuple(logits.shape)}")
    dev = logits.device
    if sums is None:
        sums = zeros(2, torch.float64, dev)
    am = torch.empty((n, *logits.shape[2:]), device=dev, dtype=torch.int64) if want_argmax else None
    conf = zeros((n, c, c), torch.int64, dev) if want_conf else None
    if corr is None and want_correct:
        corr = zeros(1, torch.int64, dev)
    if class_w is not None:
        class_w = _chk(class_w, name="class_w")
        if class_w.numel() != c:
            raise ValueError("ce_fwd: class_w must have C entries")
    if scratch is None:
        _call("rcv_ce_fwd", 1, n, c, hw, _ptr(logits), _ptr(target), _ptr(class_w), _ptr(sums), _ptr(am),
              _ptr(conf), _ptr(corr), _stream())
    else:
        _call("rcv_ce_fwd_det", 1, n, c, hw, _ptr(logits), _ptr(target), _ptr(class_w), _ptr(sums), _ptr(am),
              _ptr(conf), _ptr(corr), *_scratch_args(scratch), _stream())
    return sums, am, conf, corr


def ce_bwd(logits, target, class_w, sums, gscale=None):
    logits = _chk(logits, name="logits")
    target = _chk(target, torch.int64, "target")
    n, c = logits.shape[0], logits.shape[1]
    hw = logits.numel() // (n * c)
    dl = torch.empty_like(logits)
    if gscale is not None:
        gscale = _chk(gscale.reshape(1).to(torch.float32), name="gscale")
    _call("rcv_ce_bwd", 1, n, c, hw, _ptr(logits), _ptr(target), _ptr(class_w), _ptr(sums), _ptr(gscale),
          _ptr(dl), _stream())
    return dl


def confusion(pred, target, num_classes: int):
    pred = _chk(pred, torch.int64, "pred")
    target = _chk(target, torch.int64, "target")
    n = pred.shape[0]
    hw = pred.numel() // n
    conf = zeros((n, num_classes, num_classes), torch.int64, pred.device)
    _call("rcv_confusion", 1, n, num_classes, hw, _ptr(pred), _ptr(target), _ptr(conf), _stream())
    return conf


def metric_tail(conf, loss_sums=None):
    """-> (iou_sum float64[C], loss float64[] | None) from per-image confusion counts int64[N,C,C] and the loss sums of
    ce_fwd: the validation loops' per-image IoU rule and the mean loss in one launch (rcv_metric_tail)."""
    conf = _chk(conf, torch.int64, "conf")
    n, c = conf.shape[0], conf.shape[1]
    out = torch.empty(c + 1, dtype=torch.float64, device=conf.device)
    _call("rcv_metric_tail", 1, n, c, _ptr(conf), _ptr(loss_sums), _ptr(out), _ptr(out[c:]) if loss_sums is not None else None,
          _stream())
    return out[:c], (out[c] if loss_sums is not None else None)


# --------------------------------------------------------------------------- input-side label ops
def mask_label_lut(nb: bool, nr: bool, ng: bool, nl: bool, num_classes: int = 5):
    """Lookup table of maskLabel (transform.py:26-49): the relabel applied to class ids 0..C-1."""
    lut = list(range(num_classes))
    b, r, g, l = 1, 2, 3, 4

    def drop(k, lut):
        return [0 if v == k else (v - 1 if v > k else v) for v in lut]
    if nb:
        lut = drop(b, lut); r, g, l = 1, 2, 3
    if nr:
        lut = drop(r, lut); g, l = 1, 2
    if ng:
        lut = drop(g, lut); l = 1
    if nl:
        lut = [0 if v == l else v for v in lut]
    return lut


def mask_label_(label, nb, nr, ng, nl, num_classes: int = 5):
    """In-place maskLabel on a CUDA int64 label tensor (one launch).  The tensor must be contiguous and 16-byte
    aligned: a strided or offset view would be relabelled in a temporary copy, not in place, so it is refused."""
    if label.is_cuda and (not label.is_contiguous() or label.data_ptr() % 16):
        raise ValueError("mask_label_: in-place relabel needs a contiguous, 16-byte aligned label tensor "
                         "(call .contiguous() first and use the returned tensor)")
    label = _chk(label, torch.int64, "label")
    lut = torch.tensor(mask_label_lut(nb, nr, ng, nl, num_classes), dtype=torch.int64, device=label.device)
    _call("rcv_label_lut", 1, label.numel(), _ptr(label), lut.numel(), _ptr(lut), _stream())
    return label


def label_to_pred(label, num_classes: int):
    """labelToPred (transform.py:172-183): int64 [B,H,W] -> float [B,C,H,W] of +-1."""
    label = _chk(label, torch.int64, "label")
    b, h, w = label.shape
    out = torch.empty((b, num_classes, h, w), device=label.device, dtype=torch.float32)
    _call("rcv_label_to_pred", 1, b, num_classes, h * w, _ptr(label), _ptr(out), _stream())
    return out


def lp_assemble(ya, yb, la, lb, num_classes: int = 5):
    """LabelProp batch assembly (labelPropTrain.py:178-193) for P frame pairs -> (inputs [2P,3+C,H,W],
    targets [2P,H,W])."""
    ya, yb = _chk(ya, name="ya"), _chk(yb, name="yb")
    la, lb = _chk(la, torch.int64, "la"), _chk(lb, torch.int64, "lb")
    p, h, w = ya.shape
    inputs = torch.empty((2 * p, 3 + num_classes, h, w), device=ya.device, dtype=torch.float32)
    targets = torch.empty((2 * p, h, w), device=ya.device, dtype=torch.int64)
    _call("rcv_lp_assemble", 1, p, num_classes, h * w, _ptr(ya), _ptr(yb), _ptr(la), _ptr(lb), _ptr(inputs),
          _ptr(targets), _stream())
    return inputs, targets


# --------------------------------------------------------------------------- optimiser tail
def color_jitter_params(flip, b_val, c_val, s_val, h_val, device):
    """Per-image parameter rows of rcv_augment from the scalars ColorJitter.__call__ draws
    (dataset.py:27-32): mtx = [[s cos h, -sin h], [sin h, s cos h]], as float32 like torch.FloatTensor."""
    import math
    rows = []
    for f, b, c, s_, h in zip(flip, b_val, c_val, s_val, h_val):
        rows.append([1.0 if f else 0.0, b, c, s_ * math.cos(h), -math.sin(h), math.sin(h), s_ * math.cos(h), 0.0])
    return torch.tensor(rows, dtype=torch.float32, device=device)


def augment(x, params, labels=None, mean=(0.5, 0.0, 0.0), std=(0.5, 0.5, 0.5)):
    """Normalize + horizontal flip + ColorJitter over a batch [N,3,H,W] (dataset.py:123-131); params from
    color_jitter_params.  -> (images, labels or None)."""
    x = _chk(x, name="images")
    n, c, h, w = x.shape
    if c != 3:
        raise ValueError("augment: 3-channel (YUV) images expected")
    params = _chk(params, name="params")
    if tuple(params.shape) != (n, 8):
        raise ValueError("augment: params must be [N, 8]")
    y = torch.empty_like(x)
    lo = None
    if labels is not None:
        labels = _chk(labels, torch.int64, "labels")
        lo = torch.empty_like(labels)
    m = (_lib._f32 * 3)(*[float(v) for v in mean])
    sd = (_lib._f32 * 3)(*[float(v) for v in std])
    _call("rcv_augment", 1, n, h, w, _ptr(x), _ptr(y), _ptr(labels), _ptr(lo), _ptr(params), m, sd, _stream())
    return y, lo


def dice_fwd(logits, target, scratch=None, sums=None):
    """-> float64[2C]: per-class soft intersection and cardinality of softmax(logits) vs the labels.  scratch:
    det_scratch(DET_DICE_FWD, ...) for the fixed-order sums (rcv_dice_fwd_det).  sums: a caller-zeroed float64[2C] to
    accumulate into instead of a fresh one."""
    logits = _chk(logits, name="logits")
    target = _chk(target, torch.int64, "target")
    n, c = logits.shape[0], logits.shape[1]
    hw = logits.numel() // (n * c)
    if sums is None:
        sums = zeros(2 * c, torch.float64, logits.device)
    if scratch is None:
        _call("rcv_dice_fwd", 1, n, c, hw, _ptr(logits), _ptr(target), _ptr(sums), _stream())
    else:
        _call("rcv_dice_fwd_det", 1, n, c, hw, _ptr(logits), _ptr(target), _ptr(sums), *_scratch_args(scratch),
              _stream())
    return sums


def dice_bwd(logits, target, weights, sums, eps, gscale=None):
    logits = _chk(logits, name="logits")
    n, c = logits.shape[0], logits.shape[1]
    hw = logits.numel() // (n * c)
    d = torch.empty_like(logits)
    if gscale is not None:
        gscale = gscale.to(torch.float32).reshape(1).contiguous()
    _call("rcv_dice_bwd", 1, n, c, hw, _ptr(logits), _ptr(target), _ptr(weights), _ptr(sums), float(eps),
          _ptr(gscale), _ptr(d), _stream())
    return d


def adam_l1_step(p, g, m, v, lr, beta1=0.9, beta2=0.999, eps=1e-8, step=1, l1_decay=0.0, grad_scale=1.0,
                 mask=None, l1_sum=None, step_dev=None, lr_dev=None, scratch=None):
    """scratch: det_scratch(DET_L1_SUM, ...) for l1_sum in fixed order (rcv_adam_l1_step_det)."""
    args = (p.numel(), _ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(mask), float(lr), float(beta1), float(beta2),
            float(eps), int(step), float(l1_decay), float(grad_scale), _ptr(l1_sum), _ptr(step_dev), _ptr(lr_dev))
    if scratch is None:
        _call("rcv_adam_l1_step", 1, *args, _stream())
    else:
        _call("rcv_adam_l1_step_det", 1, *args, *_scratch_args(scratch), _stream())


def sgd_step(p, g, buf, lr, momentum=0.0, weight_decay=0.0, grad_scale=1.0, mask=None, first_step=False,
             l1_decay=0.0, l1_sum=None, lr_dev=None, scratch=None):
    """scratch: det_scratch(DET_L1_SUM, ...) for l1_sum in fixed order (rcv_sgd_step_det)."""
    args = (p.numel(), _ptr(p), _ptr(g), _ptr(buf), _ptr(mask), float(lr), float(momentum), float(weight_decay),
            float(grad_scale), 1 if first_step else 0, float(l1_decay), _ptr(l1_sum), _ptr(lr_dev))
    if scratch is None:
        _call("rcv_sgd_step", 1, *args, _stream())
    else:
        _call("rcv_sgd_step_det", 1, *args, *_scratch_args(scratch), _stream())


# --------------------------------------------------------------------------- fixed-order reductions
def det_scratch_bytes(op: int, n: int, c: int, hw: int) -> int:
    """Bytes of scratch the fixed-order (_det) form of `op` (DET_CE_FWD, DET_CE_WEIGHT_SUM, DET_DICE_FWD,
    DET_L1_SUM) needs for N=n, C=c, HW=hw (see rcv_det_scratch_bytes for what each op reads).  Host only."""
    nb = _lib.load().rcv_det_scratch_bytes(int(op), int(n), int(c), int(hw))
    if nb == 0:
        raise ValueError(f"det_scratch_bytes: no fixed-order path for op {op} at N={n}, C={c}, HW={hw}")
    return nb


def det_scratch(op: int, n: int, c: int, hw: int, device) -> torch.Tensor:
    """Zero-filled scratch for the fixed-order form of `op` (see det_scratch_bytes).  The kernels leave it ready for
    the next call of the same op and size; one stream at a time."""
    return zeros(det_scratch_bytes(op, n, c, hw), torch.uint8, device)


def _scratch_args(scratch: torch.Tensor):
    if not scratch.is_cuda or scratch.dtype != torch.uint8 or not scratch.is_contiguous():
        raise RuntimeError("robocupvision_b200: scratch must be a contiguous CUDA uint8 tensor (det_scratch)")
    return _ptr(scratch), C.c_uint64(scratch.numel())


def zero_(t: torch.Tensor) -> torch.Tensor:
    """Stream-ordered zero fill without a kernel (a memset node under graph capture)."""
    if not t.is_cuda or not t.is_contiguous():
        raise RuntimeError("robocupvision_b200: zero_ needs a contiguous CUDA tensor")
    _lib.call("rcv_zero", _ptr(t), C.c_size_t(t.numel() * t.element_size()), _stream())
    return t


def zeros(shape, dtype, device) -> torch.Tensor:
    return zero_(torch.empty(shape, dtype=dtype, device=device))


def counter_add(counter, inc=1):
    _call("rcv_counter_add", 1, _ptr(counter), int(inc), _stream())
