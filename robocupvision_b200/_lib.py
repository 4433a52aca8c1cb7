"""ctypes binding of librcv_b200.so (include/rcv_b200.h).

This is the only place the shared library is loaded.  There is no fallback: if the
library is missing or fails to load, every op raises (``RcvLibraryError``) instead of
silently running something else.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "librcv_b200.so"


class RcvLibraryError(RuntimeError):
    pass


class RcvError(RuntimeError):
    """A librcv_b200 call returned a negative rcv_status."""

    def __init__(self, fn: str, code: int, msg: str):
        super().__init__(f"{fn} failed with rcv_status {code}: {msg}")
        self.code = code


# rcv_status
RCV_OK, RCV_ERR_BAD_ARG, RCV_ERR_UNSUPPORTED, RCV_ERR_CUDA, RCV_ERR_WORKSPACE = 0, -1, -2, -3, -4
# rcv_epilogue
EPI_NONE, EPI_RELU, EPI_RELU_AFFINE, EPI_AFFINE_RELU, EPI_AFFINE = 0, 1, 2, 3, 4
# rcv_math
MATH_FP32, MATH_TF32X3, MATH_AUTO, MATH_TF32, MATH_BF16 = 0, 1, 2, 3, 4
# rcv_det_op
DET_CE_FWD, DET_CE_WEIGHT_SUM, DET_DICE_FWD, DET_L1_SUM = 0, 1, 2, 3
# rcv_engine
ENGINE_SIMT, ENGINE_DIRECT, ENGINE_UMMA, ENGINE_NARROW = 0, 1, 2, 3


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "N", "Cin", "H", "W", "Cout", "ksize", "stride", "pad", "dil", "transposed", "epilogue", "math")] + [
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_uint64), ("res_channels", C.c_int32)]


_p = C.c_void_p
_i32, _i64, _f32 = C.c_int32, C.c_int64, C.c_float

# name -> argtypes (restype is always int unless listed in _RESTYPES)
SIGNATURES = {
    "rcv_version": [],
    "rcv_set_pdl": [C.c_int],
    "rcv_get_pdl": [],
    "rcv_last_error": [],
    "rcv_conv_out_hw": [C.POINTER(ConvDesc), C.POINTER(_i32), C.POINTER(_i32)],
    "rcv_conv_packed_bytes": [C.POINTER(ConvDesc), C.c_int],
    "rcv_conv_uses_tensor_cores": [C.POINTER(ConvDesc), C.c_int],
    "rcv_conv_workspace_bytes": [C.POINTER(ConvDesc), C.c_int],
    "rcv_conv_pack": [C.POINTER(ConvDesc), C.c_int, _p, _p, _p],
    "rcv_conv_engine": [C.POINTER(ConvDesc), C.c_int],
    "rcv_conv_pack_table_bytes": [_i32],
    "rcv_conv_pack_table_build": [_i32, C.POINTER(ConvDesc), C.POINTER(_i32), C.POINTER(_p), C.POINTER(_p), _p,
                                  C.POINTER(_i64)],
    "rcv_conv_pack_table_run": [_p, _i32, _i64, _p],
    "rcv_conv_fwd": [C.POINTER(ConvDesc), _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_conv_normalises_on_load": [C.POINTER(ConvDesc)],
    "rcv_conv_fwd_nl": [C.POINTER(ConvDesc), _p, _p, _p, C.c_int, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_conv_dgrad": [C.POINTER(ConvDesc), _p, _p, _p, _p, _p, _p],
    "rcv_conv_wgrad": [C.POINTER(ConvDesc), _p, _p, _p, _p, _p],
    "rcv_conv_wgrad_normalises_on_load": [C.POINTER(ConvDesc)],
    "rcv_conv_wgrad_nl": [C.POINTER(ConvDesc), _p, _p, _p, C.c_int, _p, _p, _p, _p],
    "rcv_bn_finalize": [_i32, _i64, _p, _p, _p, _p, _p, _f32, _f32, _p, _p, _p, _p, _p, _p],
    "rcv_bn_fold": [_i32, _p, _p, _p, _p, _f32, _p, _p, _p],
    "rcv_bn_apply": [_i32, _i32, _i64, _p, _p, _p, C.c_int, _p, _i32, _p, _p],
    "rcv_bn_finalize_apply": [_i32, _i32, _i64, _p, _p, _p, _p, _p, _f32, _f32, _p, C.c_int, _p, _i32, _p, _p, _p, _p,
                              _p, _p, _p],
    "rcv_bn_bwd_reduce": [_i32, _i32, _i64, C.c_int, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_bn_bwd_apply": [_i32, _i32, _i64, C.c_int, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_bn_bwd_is_fused": [_i32, _i32, _i64],
    "rcv_bn_bwd": [_i32, _i32, _i64, C.c_int, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_relu_bwd": [_i64, _p, _p, _p, _p],
    "rcv_channel_sum": [_i32, _i32, _i64, _p, _p, _p],
    "rcv_maxpool2x2_fwd": [_i32, _i32, _i32, _i32, _p, _p, _p, _p, _p],
    "rcv_maxpool2x2_bwd": [_i32, _i32, _i32, _i32, _p, _p, _p, _p],
    "rcv_maxunpool2x2_fwd": [_i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p],
    "rcv_maxunpool2x2_bwd": [_i32, _i32, _i32, _i32, _p, _p, _p, _p, _p],
    "rcv_upsample_bilinear2x_fwd": [_i32, _i32, _i32, _i32, _p, _p, _p, _p],
    "rcv_upsample_bilinear2x_bwd": [_i32, _i32, _i32, _i32, _p, _p, _p],
    "rcv_channel_copy": [_i64, _i64, _i32, _p, _i32, _i32, _p, _i32, _i32, _p],
    "rcv_head_ce_supported": [_i32, _i32],
    "rcv_ce_weight_sum": [_i32, _i64, _p, _p, _p, _p],
    "rcv_head_ce_train": [_i32, _i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_head_dice_fwd": [_i32, _i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p],
    "rcv_head_dice_train": [_i32, _i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _f32, _p, _p, _p, _p, _p, _p],
    "rcv_dice_loss": [_i32, _p, _p, _f32, _p, _p],
    "rcv_peer_flag_bytes": [],
    "rcv_peer_alloc": [C.c_uint64, C.POINTER(C.c_void_p), _p],
    "rcv_peer_open": [_p, C.POINTER(C.c_void_p)],
    "rcv_peer_close": [_p],
    "rcv_peer_free": [_p],
    "rcv_peer_allreduce": [_i32, _i32, _i32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i64, _i64, _p, _p],
    "rcv_ce_fwd": [_i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p, _p],
    "rcv_ce_bwd": [_i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p],
    "rcv_confusion": [_i32, _i32, _i64, _p, _p, _p, _p],
    "rcv_metric_tail": [_i32, _i32, _p, _p, _p, _p, _p],
    "rcv_label_lut": [_i64, _p, _i32, _p, _p],
    "rcv_label_to_pred": [_i64, _i32, _i64, _p, _p, _p],
    "rcv_lp_assemble": [_i64, _i32, _i64, _p, _p, _p, _p, _p, _p, _p],
    "rcv_augment": [_i32, _i32, _i32, _p, _p, _p, _p, _p, C.POINTER(_f32), C.POINTER(_f32), _p],
    "rcv_dice_fwd": [_i32, _i32, _i64, _p, _p, _p, _p],
    "rcv_dice_bwd": [_i32, _i32, _i64, _p, _p, _p, _p, _f32, _p, _p, _p],
    "rcv_adam_l1_step": [_i64, _p, _p, _p, _p, _p, _f32, _f32, _f32, _f32, _i32, _f32, _f32, _p, _p, _p, _p],
    "rcv_counter_add": [_p, _i32, _p],
    "rcv_sgd_step": [_i64, _p, _p, _p, _p, _f32, _f32, _f32, _f32, C.c_int, _f32, _p, _p, _p],
    "rcv_zero": [_p, C.c_size_t, _p],
    "rcv_det_scratch_bytes": [C.c_int, _i32, _i32, _i64],
    "rcv_ce_fwd_det": [_i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p, _p, C.c_uint64, _p],
    "rcv_ce_weight_sum_det": [_i32, _i64, _p, _p, _p, _p, C.c_uint64, _p],
    "rcv_dice_fwd_det": [_i32, _i32, _i64, _p, _p, _p, _p, C.c_uint64, _p],
    "rcv_adam_l1_step_det": [_i64, _p, _p, _p, _p, _p, _f32, _f32, _f32, _f32, _i32, _f32, _f32, _p, _p, _p, _p,
                             C.c_uint64, _p],
    "rcv_sgd_step_det": [_i64, _p, _p, _p, _p, _f32, _f32, _f32, _f32, C.c_int, _f32, _p, _p, _p, C.c_uint64, _p],
}
_RESTYPES = {"rcv_last_error": C.c_char_p, "rcv_conv_packed_bytes": C.c_size_t, "rcv_conv_workspace_bytes": C.c_size_t,
             "rcv_conv_pack_table_bytes": C.c_size_t, "rcv_peer_flag_bytes": C.c_uint64,
             "rcv_det_scratch_bytes": C.c_size_t}
PACK_FWD, PACK_DGRAD = 0, 1
ABI_VERSION = 5

_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the .so is absent and nvcc exists) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists() and build_if_missing and not os.environ.get("RCV_NO_BUILD"):
        try:
            from . import build as _build
            _build.build()
        except Exception as e:  # noqa: BLE001
            raise RcvLibraryError(
                f"librcv_b200.so is missing and could not be built ({e}); "
                "run `python -m robocupvision_b200.build`. There is no fallback path.") from e
    if not LIB_PATH.exists():
        raise RcvLibraryError(f"{LIB_PATH} not found; run `python -m robocupvision_b200.build`. "
                              "There is no fallback path.")
    try:
        lib = C.CDLL(str(LIB_PATH))
    except OSError as e:
        raise RcvLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    for name, argtypes in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise RcvLibraryError(f"{LIB_PATH} does not export {name}") from e
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    abi = lib.rcv_version()
    if abi != ABI_VERSION:
        raise RcvLibraryError(f"ABI version mismatch: library {abi}, binding {ABI_VERSION}")
    # Programmatic dependent launch: on for single-process runs (+0.9 % on the training step, every parity test
    # green in both modes); multi-process (NCCL kernels inside the step's graph) keeps plain stream order until
    # that combination has been measured.  RCV_PDL in the environment overrides.
    if "RCV_PDL" not in os.environ:
        try:
            world = int(os.environ.get("WORLD_SIZE", "1") or "1")
        except ValueError:
            world = 1
        lib.rcv_set_pdl(1 if world == 1 else 0)
    _lib = lib
    return lib


def call(name: str, *args) -> None:
    """Invoke an rcv_* entry point and raise RcvError on a negative status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RcvError(name, rc, lib.rcv_last_error().decode("utf-8", "replace"))
