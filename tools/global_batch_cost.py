"""Latency cost of TrainStep(global_batch=True) on ONE GPU: the global-batch step with force_comm_path=True (every
exchange kernel runs, at world 1 with local flags) against the plain step on the same communication path, for
ROBO_UNet at 3x120x160 and a few per-rank batch sizes.  With one rank the exchanges move no data between GPUs, so the
difference is a lower bound on what the option adds per step: the extra launches (one exchange per BatchNorm layer in
each direction, the loss normaliser, the end-of-step loss and correct count) and the BatchNorm backward layers that
leave the one-launch cluster kernel for two passes.  Multi-GPU strong scaling is not measured here.

    python tools/global_batch_cost.py [--batches 8 16 64] [--steps 50] [--rounds 7] [--reps 500]

Steps are graph-replayed and timed with CUDA events over `steps` back-to-back replays, the two variants alternating
round by round; the median round is reported.  rcv_peer_allreduce_f64 is also timed alone (world 1, 256 doubles:
the largest BatchNorm layer's statistics) over `reps` launches.  The card's name and power limit are printed beside
the numbers."""
import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tests"))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from dice_step_cost import card, time_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[8, 16, 64])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=500)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("global_batch_cost: needs a CUDA device")
    import synth
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import TrainStep
    dev = "cuda"
    h, w = 120, 160
    rows = {}
    for n in a.batches:
        x = synth.images(n, 3, h, w, seed=1).to(dev)
        y = synth.labels_learnable(x.cpu()).to(dev)
        steps = {}
        for k, gb in (("plain", False), ("global_batch", True)):
            torch.manual_seed(12345678)
            steps[k] = TrainStep(ROBO_UNet().to(dev), synth.CLASS_WEIGHTS, lr=1e-3, l1_decay=1e-6, use_graph=True,
                                 force_comm_path=True, global_batch=gb)
            for _ in range(3):  # capture + warm replays
                steps[k].step(x, y)
        torch.cuda.synchronize()
        times = {k: [] for k in steps}
        for _ in range(a.rounds):
            for k, ts in steps.items():
                times[k].append(time_ms(lambda: ts.step(x, y), a.steps))
        med = {k: statistics.median(v) for k, v in times.items()}
        rows[n] = {k: {"ms_per_step": round(med[k], 4), "min_ms": round(min(times[k]), 4),
                       "max_ms": round(max(times[k]), 4), "kernels_per_step": steps[k].kernels_per_step}
                   for k in steps}
        rows[n]["extra_us_per_step"] = round((med["global_batch"] - med["plain"]) * 1e3, 1)
        rows[n]["extra_percent"] = round(100.0 * (med["global_batch"] / med["plain"] - 1.0), 2)
        for ts in steps.values():
            ts.peer.check()
        del steps

    from robocupvision_b200.peer import PeerExchange
    px = PeerExchange(64, dev, ndoubles=256)
    t = px.accum
    for _ in range(10):
        px.allreduce_f64(t)
    torch.cuda.synchronize()
    us = statistics.median(time_ms(lambda: px.allreduce_f64(t), a.reps) for _ in range(a.rounds)) * 1e3
    px.check()
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power, "workload": "ROBO_UNet train step, one GPU",
                      "hw": [h, w], "steps": a.steps, "rounds": a.rounds, "by_batch": rows,
                      "peer_allreduce_f64_256_us": round(us, 2)}))


if __name__ == "__main__":
    main()
