"""Cost of the fixed-order (_det) reductions against the atomic forms, per call, at the sizes of a ROBO_UNet
training step (batch 64, 120x160, 5 classes; the Adam / SGD range is the net's whole parameter arena).

    python tools/det_reduction_cost.py [--reps 200] [--rounds 5]

Each entry point is timed with CUDA events over `reps` back-to-back calls on one stream, plain and fixed-order
alternating for `rounds` rounds; the best round of each is reported in microseconds per call, beside the card's name
and power limit."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def time_us(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("det_reduction_cost: needs a CUDA device")
    from robocupvision_b200 import ops
    from robocupvision_b200.model import ROBO_UNet
    dev = "cuda"
    n, c, h, w = 64, 5, 120, 160
    gen = torch.Generator().manual_seed(0)
    z = (torch.randn(n, c, h, w, generator=gen) * 3).to(dev)
    y = torch.randint(0, c, (n, h, w), generator=gen).to(dev)
    cw = (torch.rand(c, generator=gen) + 0.5).to(dev)
    npar = sum(p.numel() for p in ROBO_UNet().parameters())
    p = torch.randn(npar, generator=gen).to(dev)
    g = torch.randn(npar, generator=gen).to(dev)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    sums = ops.zeros(2 * c, torch.float64, dev)
    l1 = ops.zeros(1, torch.float64, dev)
    hw = h * w
    s_ce = ops.det_scratch(ops.DET_CE_FWD, n, c, hw, dev)
    s_ws = ops.det_scratch(ops.DET_CE_WEIGHT_SUM, n, c, hw, dev)
    s_dice = ops.det_scratch(ops.DET_DICE_FWD, n, c, hw, dev)
    s_l1 = ops.det_scratch(ops.DET_L1_SUM, 1, 1, npar, dev)
    cases = {
        "ce_fwd": lambda s: ops.ce_fwd(z, y, cw, sums=sums, scratch=s),
        "ce_weight_sum": lambda s: ops.ce_weight_sum(y, cw, sums, c, scratch=s),
        "dice_fwd": lambda s: ops.dice_fwd(z, y, scratch=s),
        "adam_l1_step": lambda s: ops.adam_l1_step(p, g, m, v, lr=1e-3, step=1, l1_decay=1e-6, l1_sum=l1, scratch=s),
        "sgd_step": lambda s: ops.sgd_step(p, g, m, lr=1e-3, momentum=0.9, l1_decay=1e-6, l1_sum=l1, scratch=s),
    }
    scratches = {"ce_fwd": s_ce, "ce_weight_sum": s_ws, "dice_fwd": s_dice, "adam_l1_step": s_l1, "sgd_step": s_l1}
    name, power = card()
    rows = {}
    for k, fn in cases.items():
        for s in (None, scratches[k]):  # warm-up: module load, first launch
            fn(s)
        torch.cuda.synchronize()
        plain, det = [], []
        for _ in range(a.rounds):
            plain.append(time_us(lambda: fn(None), a.reps))
            det.append(time_us(lambda: fn(scratches[k]), a.reps))
        rows[k] = {"plain_us": round(min(plain), 2), "det_us": round(min(det), 2),
                   "extra_us": round(min(det) - min(plain), 2)}
    print(json.dumps({"card": name, "power_limit": power, "batch": n, "hw": [h, w], "classes": c,
                      "params": npar, "reps": a.reps, "rounds": a.rounds, "per_call": rows}))


if __name__ == "__main__":
    main()
