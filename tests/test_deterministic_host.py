"""CPU suite for the fixed-order (_det) reductions: the scratch-size query answers without a GPU, follows the launch
geometry, and is 0 where an entry point refuses; the _det entry points refuse a missing or short scratch before any
launch; the train-mode module path refuses torch.use_deterministic_algorithms(True) as torch's own ops do."""
import ctypes as C
import warnings

import pytest
import torch


def _lib():
    from robocupvision_b200 import _lib
    return _lib, _lib.load()


def _slots_ce(n, hw):  # ce_fwd / dice_fwd grid: (chunks, N), chunks capped at ceil(148*8 / N)
    return min(max(-(-hw // 256), 1), max(-(-148 * 8 // n), 1)) * n


@pytest.mark.parametrize("n,c,hw", [(64, 5, 120 * 160), (8, 5, 480 * 640), (1, 2, 16), (65535, 8, 4)])
def test_scratch_bytes_follow_the_grid(n, c, hw):
    L, lib = _lib()
    pad = lambda b: 128 + (b + 127) // 128 * 128  # noqa: E731
    assert lib.rcv_det_scratch_bytes(L.DET_CE_FWD, n, c, hw) == pad(_slots_ce(n, hw) * 2 * 8)
    assert lib.rcv_det_scratch_bytes(L.DET_DICE_FWD, n, c, hw) == pad(_slots_ce(n, hw) * 2 * c * 8)
    count = n * hw
    assert lib.rcv_det_scratch_bytes(L.DET_CE_WEIGHT_SUM, n, c, hw) == pad(min(max(-(-count // 2048), 1), 592) * 8)
    assert lib.rcv_det_scratch_bytes(L.DET_L1_SUM, n, c, hw) == pad(min(max(-(-count // 256), 1), 1184) * 8)


def test_scratch_bytes_zero_where_refused():
    L, lib = _lib()
    assert lib.rcv_det_scratch_bytes(99, 4, 5, 100) == 0
    assert lib.rcv_det_scratch_bytes(L.DET_CE_FWD, 0, 5, 100) == 0
    assert lib.rcv_det_scratch_bytes(L.DET_CE_FWD, 65536, 5, 100) == 0
    assert lib.rcv_det_scratch_bytes(L.DET_DICE_FWD, 4, 1, 100) == 0
    assert lib.rcv_det_scratch_bytes(L.DET_DICE_FWD, 4, 9, 100) == 0
    assert lib.rcv_det_scratch_bytes(L.DET_L1_SUM, 1, 1, 0) == 0
    from robocupvision_b200 import ops
    with pytest.raises(ValueError, match="no fixed-order path"):
        ops.det_scratch_bytes(ops.DET_DICE_FWD, 4, 9, 100)
    assert ops.det_scratch_bytes(ops.DET_CE_FWD, 4, 5, 100) > 128


def test_det_entry_points_refuse_short_scratch():
    """The size check comes before any launch, so it runs without a device (pointers are never dereferenced)."""
    L, lib = _lib()
    fake = C.c_void_p(1 << 20)
    need = lib.rcv_det_scratch_bytes(L.DET_CE_FWD, 4, 5, 1000)
    assert lib.rcv_ce_fwd_det(4, 5, 1000, fake, fake, None, fake, None, None, None, None, 0, None) == L.RCV_ERR_WORKSPACE
    assert lib.rcv_ce_fwd_det(4, 5, 1000, fake, fake, None, fake, None, None, None, fake, need - 1,
                              None) == L.RCV_ERR_WORKSPACE
    assert b"needed" in lib.rcv_last_error()
    assert lib.rcv_ce_weight_sum_det(5, 4000, fake, None, fake, fake, 8, None) == L.RCV_ERR_WORKSPACE
    assert lib.rcv_dice_fwd_det(4, 5, 1000, fake, fake, fake, None, 0, None) == L.RCV_ERR_WORKSPACE
    assert lib.rcv_dice_fwd_det(4, 9, 1000, fake, fake, fake, fake, 1 << 20, None) == L.RCV_ERR_BAD_ARG
    assert lib.rcv_adam_l1_step_det(1000, fake, fake, fake, fake, None, 1e-3, 0.9, 0.999, 1e-8, 1, 0.0, 1.0, fake,
                                    None, None, None, 0, None) == L.RCV_ERR_WORKSPACE
    assert lib.rcv_sgd_step_det(1000, fake, fake, None, None, 1e-3, 0.0, 0.0, 1.0, 0, 0.0, fake, None, fake, 64,
                                None) == L.RCV_ERR_WORKSPACE
    assert lib.rcv_adam_l1_step_det(0, fake, fake, fake, fake, None, 1e-3, 0.9, 0.999, 1e-8, 1, 0.0, 1.0, None,
                                    None, None, None, 0, None) == L.RCV_ERR_BAD_ARG


def test_alert_follows_torch_deterministic_flags():
    from robocupvision_b200.engine import _alert_not_deterministic
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            _alert_not_deterministic("thing")
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="thing does not have a deterministic implementation"):
            _alert_not_deterministic("thing")
        torch.use_deterministic_algorithms(True, warn_only=True)
        with pytest.warns(UserWarning, match="thing does not have a deterministic implementation"):
            _alert_not_deterministic("thing")
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)
