"""Cost of a Dice-loss training step (TrainStep(loss="dice")) against the cross-entropy step, and the times of the two
Dice head kernels, at the benchmarked ROBO_UNet size (batch 64, 3x120x160, 5 classes, 8 channels into the head).

    python tools/dice_step_cost.py [--steps 50] [--rounds 7] [--reps 200]

Three graph-replayed steps are timed with CUDA events over `steps` back-to-back replays, alternating round by round:
loss="ce" (the default step), loss="dice" with the fused two-pass head and loss="dice" with the unfused head (conv ->
dice_fwd -> dice_bwd -> conv dgrad / wgrad); the median round of each is reported in ms per step.  The head kernels
rcv_head_dice_fwd and rcv_head_dice_train are timed alone over `reps` launches each (median of the rounds) and
reported with their algorithmic bytes over kernel time: pass 1 reads 4 Cin + 8 bytes per pixel (features, label),
pass 2 reads the same and writes 4 Cin (feature gradient).  Their working set (49 MB) fits in the 126 MB L2, so
back-to-back launches read it from there: the rates are L2-fed, as inside the step, where the decoder's last layer
has just written the features.  The card's name and power limit are printed beside the numbers."""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tests"))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def time_ms(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dice_step_cost: needs a CUDA device")
    import synth
    from robocupvision_b200 import ops
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import TrainStep
    dev = "cuda"
    n, h, w = 64, 120, 160
    x = synth.images(n, 3, h, w, seed=1).to(dev)
    y = synth.labels_learnable(x.cpu()).to(dev)
    configs = {"ce": dict(loss="ce"), "dice_fused": dict(loss="dice", fused_head=True),
               "dice_unfused": dict(loss="dice", fused_head=False)}
    steps = {}
    for k, kw in configs.items():
        torch.manual_seed(12345678)
        steps[k] = TrainStep(ROBO_UNet().to(dev), synth.CLASS_WEIGHTS, lr=1e-3, l1_decay=1e-6, use_graph=True, **kw)
        for _ in range(3):  # capture + warm replays
            steps[k].step(x, y)
    torch.cuda.synchronize()
    times = {k: [] for k in configs}
    for _ in range(a.rounds):
        for k, ts in steps.items():
            times[k].append(time_ms(lambda: ts.step(x, y), a.steps))
    step_rows = {k: {"ms_per_step": round(statistics.median(v), 4), "min_ms": round(min(v), 4),
                     "max_ms": round(max(v), 4), "kernels_per_step": steps[k].kernels_per_step,
                     "fused_head": steps[k]._head >= 0} for k, v in times.items()}
    del steps

    # the two head kernels alone, at the head of the same net: 5 classes over 8 channels
    c, cin = 5, 8
    gen = torch.Generator().manual_seed(0)
    feat = torch.randn(n, cin, h, w, generator=gen).to(dev)
    wt = (torch.randn(c, cin, generator=gen) * 0.3).to(dev)
    b = torch.zeros(c, device=dev)
    cw = torch.tensor(synth.CLASS_WEIGHTS)
    wn = (cw / cw.sum().item() * c).to(dev)
    sums = ops.zeros(2 * c, torch.float64, dev)
    corr = ops.zeros(1, torch.int64, dev)
    cell = ops.zeros(2, torch.float64, dev)
    dw, db = torch.zeros(c, cin, device=dev), torch.zeros(c, device=dev)
    dfeat = torch.empty_like(feat)
    kernels = {
        "head_dice_fwd": lambda: ops.head_dice_fwd(feat, wt, b, y, sums, corr),
        "head_dice_train": lambda: ops.head_dice_train(feat, wt, b, y, wn, sums, 1e-7, cell, dw, db),
    }
    px = n * h * w
    algo_bytes = {"head_dice_fwd": (4 * cin + 8) * px, "head_dice_train": (4 * cin + 8 + 4 * cin) * px}
    for fn in kernels.values():
        fn()
    torch.cuda.synchronize()
    kt = {k: [] for k in kernels}
    for _ in range(a.rounds):
        for k, fn in kernels.items():
            kt[k].append(time_ms(fn, a.reps))
    kernel_rows = {}
    for k, v in kt.items():
        us = statistics.median(v) * 1e3
        kernel_rows[k] = {"us": round(us, 2), "algorithmic_bytes": algo_bytes[k],
                          "algorithmic_TBps": round(algo_bytes[k] / (us * 1e-6) / 1e12, 3)}
    del dfeat
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power, "workload": "ROBO_UNet train step", "batch": n,
                      "hw": [h, w], "classes": c, "head_cin": cin, "steps": a.steps, "rounds": a.rounds,
                      "reps": a.reps, "step": step_rows, "kernels": kernel_rows}))


if __name__ == "__main__":
    main()
