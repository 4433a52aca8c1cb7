#!/usr/bin/env python
"""bench.py -- the hot path's throughput on B200, one JSON line on stdout (rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--batch B]
                    [--math parity|tf32|bf16] [--no-extras] [--no-cpu-baseline] [--no-graph] [--dump-outputs DIR]

Headline (default workload `train`): BASELINE.json configs[1] -- ROBO-UNet 160x120 TRAINING, batch 64 per GPU, synthetic
images/labels, 5 classes; a "step" is one full train step (forward, weighted CE, + L1 term, backward, Adam) over one
batch of synthetic frames.  value = frames/s over all ranks with inputs resident in HBM; e2e = the same through
robocupvision_b200.train.TrainStep.step_async with pinned-host inputs copied H2D and the loss read back D2H every
step.  The same line carries, under "extra", one record per remaining BASELINE config (inference 160x120 at batch 256
and batch 1, the pruned / VGA checkpoints, 640x480 training with trainer.py's SGD, --UNet and LabelProp training), each
with its own e2e, whole-step roofline and CPU baseline, and at --gpus N > 1 the data-parallel self-check `dp_check`.

--impl reference times the reference's own CPU implementation of the same step on the box's host cores: the
UNMODIFIED reference classes from baseline/_ref/model.py when that staged copy exists (__graft_entry__.build() stages
it from oracle.reference_dir() where that checkout of the original project exists; git-ignored), else the oracle port
(oracle/ref_train.py drives the same ATen CPU kernels the reference's model.py dispatches to).

--dump-outputs DIR writes, on rank 0, what the timed loop's last step returned as DIR/<name>.npy (see dump_outputs): a
training step's loss sums, L1 sum and correct-pixel count, an inference step's logits, loss, argmax, confusion,
correct count and IoU sums.  Inputs and initial weights are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import torch  # noqa: E402

import synth  # noqa: E402

# SURVEY.md section 8(d): algorithmic bytes / flops per frame (fp32 activations written once
# and read once per consumer; conv flops = 2*MAC), per workload.
WORKLOADS = {
    "train":       dict(net="ROBO_UNet", kw={}, cin=3, h=120, w=160, train=True, mflop=1489.3, mb=25.805, mb_step=19.30,
                        name="ROBO-UNet 160x120 training, batch 64/GPU, 5 classes (BASELINE configs[1])", batch=64),
    "infer":       dict(net="ROBO_UNet", kw={}, cin=3, h=120, w=160, train=False, mflop=496.4, mb=8.602, mb_step=2.758,
                        name="ROBO-UNet 160x120 inference", batch=256),
    "infer_pbfcn": dict(net="PB_FCN", kw=dict(noScale=False), cin=3, h=120, w=160, train=False, mflop=540.7, mb=9.370,
                        mb_step=2.746, name="PB_FCN 160x120 inference (the released pth/bestModelSeg*.pth net; "
                        "BASELINE configs[0] / configs[2])", batch=256, ckpt="bestModelSegFinetunedPruned"),
    "infer_vga":   dict(net="PB_FCN", kw=dict(noScale=True), cin=3, h=480, w=640, train=False, mflop=4005.9, mb=132.096,
                        mb_step=2.857, name="PB_FCN 640x480 inference (BASELINE configs[3])", batch=8,
                        ckpt="bestModelSegVGA"),
    "train_vga":   dict(net="PB_FCN", kw=dict(noScale=True), cin=3, h=480, w=640, train=True, mflop=12017.7, mb=396.3,
                        mb_step=20.0, name="PB_FCN 640x480 training, batch 8, SGD lr 0.1 momentum 0.5 wd 1e-3 "
                        "(trainer.py:113,182-184; BASELINE configs[3])", batch=8,
                        optim=dict(optimizer="sgd", lr=1e-1, momentum=0.5, weight_decay=1e-3, l1_decay=0.0)),
    "train_unet":  dict(net="ROBO_UNet", kw=dict(pool=True, levels=3, bellySize=0), cin=3, h=120, w=160, train=True,
                        mflop=494.0, mb=25.344, mb_step=2.76, name="U-Net (--UNet) 160x120 training, batch 64/GPU "
                        "(BASELINE configs[4])", batch=64),
    "train_lp":    dict(net="LabelProp", kw={}, cin=8, h=120, w=160, train=True, mflop=357.6, mb=23.040, mb_step=2.58,
                        name="LabelProp two-frame training, 16 samples = 8 frame pairs per GPU (BASELINE configs[4])",
                        batch=16),
}
# the extra records of a default run: (workload, batch, latency mode, checkpoint override, math mode override)
EXTRAS_1GPU = [("infer", 256, False, None, None), ("infer", 1, True, None, None),
               ("infer_pbfcn", 256, False, "bestModelSegFinetunedPruned", None), ("infer_pbfcn", 1, True, "bestModelSeg", None),
               ("infer_vga", 8, False, None, None), ("infer_vga", 1, True, None, None),
               ("train_vga", 8, False, None, None), ("train_unet", 64, False, None, None), ("train_lp", 16, False, None, None),
               # the FAST math modes, stated separately from the fp32-parity records above (their own dtype)
               ("train", 64, False, None, "bf16"), ("infer", 256, False, None, "bf16"), ("infer", 256, False, None, "tf32"),
               ("infer_pbfcn", 256, False, "bestModelSegFinetunedPruned", "bf16")]
EXTRAS_NGPU = [("train_unet", 64, False, None, None), ("train_lp", 16, False, None, None)]
ENGINE_NAMES = {0: "igemm (fp32 FFMA)", 1: "direct_conv (fp32 FFMA)",
                2: "umma_halo / umma_igemm (tcgen05, TMEM accumulators, halo-staged A operand for stride-1 3x3)",
                3: "narrow_conv (TMA halo staging + FFMA2)"}  # rcv_engine
METRIC = "robo_unet_160x120_train_frames_per_sec"
UNIT = "frames/s"
MATH_DTYPE = {"parity": "f32", "tf32": "tf32", "bf16": "bf16"}


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        p = json.loads(f.read_text())
        return dict(hbm=p["hbm_gbs"], tensor_burst=p["bf16_tflops"],
                    tensor_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self) -> int:
        """Rows read so far: summary(first=mark()) keeps the samples taken after this point."""
        return len(self.rows)

    def summary(self, first: int = 0, last: int = None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[first:last]:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()


def load_ckpt_state(name):
    """Released checkpoint as committed under tests/golden/ckpt (weights are data); None when absent."""
    f = ROOT / "tests" / "golden" / "ckpt" / (name + ".npz")
    if not f.exists():
        return None
    import numpy as np
    z = np.load(f)
    return {k: torch.from_numpy(z[k].copy()) for k in z.files}


def build_model(wl, device, ckpt=None):
    from robocupvision_b200 import model as M
    torch.manual_seed(12345678)  # train.py:332
    if wl["net"] == "ROBO_UNet":
        m = M.ROBO_UNet(**wl["kw"])
    elif wl["net"] == "PB_FCN":
        m = M.PB_FCN(32, 5, 1, wl["kw"]["noScale"], 0)
    else:
        m = M.LabelProp(5, 32, 0)
    used = None
    if ckpt:
        sd = load_ckpt_state(ckpt)
        if sd is not None:
            M.load_legacy_state_dict(m, sd)
            used = ckpt
    return m.to(device), used


def class_weights(wl):
    return synth.LP_CLASS_WEIGHTS if wl["net"] == "LabelProp" else synth.CLASS_WEIGHTS


# ------------------------------------------------------------------------------------------ the reference's CPU path
def _staged_reference():
    """The UNMODIFIED reference model.py, staged (git-ignored) under baseline/_ref by __graft_entry__.build()."""
    f = ROOT / "baseline" / "_ref" / "model.py"
    if not f.exists():
        return None
    import importlib.util
    spec = importlib.util.spec_from_file_location("rcv_reference_model", f)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _reference_step_fn(REFM, wl, ckpt, x, y):
    """train.py:43-74 / trainer.py:208-230 / tester.py:131-144 driven on the reference's own classes."""
    torch.manual_seed(12345678)
    if wl["net"] == "ROBO_UNet":
        m = REFM.ROBO_UNet(**wl["kw"])
    elif wl["net"] == "PB_FCN":
        m = REFM.PB_FCN(32, 5, 1, wl["kw"]["noScale"], 0)
    else:  # LabelProp: the shipped constructor passes a surplus 8th argument (SURVEY 8c ii); drop it
        orig = REFM.ConvPoolSimple.__init__
        REFM.ConvPoolSimple.__init__ = lambda self, i, p, s, st, pa, d, b, dropout=None: orig(self, i, p, s, st, pa, d, b)
        try:
            m = REFM.LabelProp(5, 32, 0)
        finally:
            REFM.ConvPoolSimple.__init__ = orig
    if ckpt:
        sd = load_ckpt_state(ckpt)
        if sd is not None:
            sd = {("segmenter." + k[len("classifier."):] if k.startswith("classifier.classifier.") else k): v
                  for k, v in sd.items()}
            m.load_state_dict(sd, strict=False)

    def fwd(inp):
        if wl["net"] != "LabelProp":
            return m(inp)
        top = m.pre(inp); middle = m.down1(top); bottom = m.down2(middle)  # model.py:556-567, line 565 out of place
        v = m.conv3(m.conv2(m.conv1(m.down3(bottom))))
        v = m.upConv2(m.upConv1(v) + bottom) + middle
        v = m.upConv3(v)
        return m.classifier(torch.cat([v[:, :8] + top, v[:, 8:]], 1))
    if not wl["train"]:
        m.eval()

        def step():
            with torch.no_grad():
                return fwd(x)
        return step
    crit = REFM.CrossEntropyLoss2d(torch.tensor(class_weights(wl)))
    o = wl.get("optim")
    if o:
        opt = torch.optim.SGD(m.parameters(), lr=o["lr"], momentum=o["momentum"], weight_decay=o["weight_decay"])
        decay = 0.0
    else:
        opt, decay = torch.optim.Adam(m.parameters(), lr=1e-3), 1e-6
    m.train()

    def step():
        opt.zero_grad()
        pred = fwd(x)
        loss = crit(pred, y)
        if decay:
            loss = loss + decay * sum(p.abs().sum() for p in m.parameters())
        loss.backward()
        opt.step()
        return float(loss), int((pred.argmax(1) == y).sum())
    return step


def _port_step_fn(wl, ckpt, x, y):
    from oracle import ref_model as R
    from oracle.ref_train import OracleTrainer
    from robocupvision_b200 import model as M  # module tree only (CPU init = the reference's init)
    m, _ = build_model(wl, "cpu", ckpt)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    if wl["net"] == "ROBO_UNet":
        kw = wl["kw"]
        okw = dict(pool=kw.get("pool", False), levels=kw.get("levels", 2), belly_size=kw.get("bellySize", 5))
        fwd = lambda s, xx, training: R.robo_unet_forward(s, xx, training=training, **okw)  # noqa: E731
    elif wl["net"] == "PB_FCN":
        ns = wl["kw"]["noScale"]
        fwd = lambda s, xx, training: R.pb_fcn_forward(s, xx, ns, training=training)  # noqa: E731
    else:
        fwd = lambda s, xx, training: R.labelprop_forward(s, xx, training=training)  # noqa: E731
    if not wl["train"]:
        def step():
            with torch.no_grad():
                return fwd(sd, x, False)
        return step
    o = wl.get("optim") or dict(optimizer="adam", lr=1e-3, l1_decay=1e-6)
    tr = OracleTrainer(sd, fwd, class_weights(wl), **o)
    return lambda: tr.step(x, y)


def cpu_reference(wl, batch, steps, warmup, ckpt=None, budget_s=None):
    """The reference's CPU path for this workload on all host threads -> (fps, ms/step, threads, kind, steps run).
    budget_s: stop after that many seconds of timed steps (bounded sample), at least one step."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    x = synth.images(batch, wl["cin"], wl["h"], wl["w"])
    y = synth.labels_random(batch, wl["h"], wl["w"])
    REFM = _staged_reference()
    if REFM is not None:
        fn, kind = _reference_step_fn(REFM, wl, ckpt, x, y), "reference"
    else:
        fn, kind = _port_step_fn(wl, ckpt, x, y), "port"
    for _ in range(warmup):
        fn()
    t0, n = time.perf_counter(), 0
    while n < steps:
        fn()
        n += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = (time.perf_counter() - t0) / n
    return batch / dt, dt * 1e3, threads, kind, n


DUMP_MAX_ELEMS = 1 << 20        # per array: larger outputs are stored as a fixed, seeded sample of this many elements
DUMP_MAX_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, arrays: dict) -> None:
    """arrays (name -> tensor) as out_dir/<name>.npy: floating point as float32 (float64 stays float64), integers as
    float64 (exact below 2**53).  An array of more than DUMP_MAX_ELEMS elements is flattened and sampled at indices
    drawn from a generator seeded with 0 (sorted), the same for every run of the same shape; smaller arrays keep
    their shape."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    host = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        t = t.cpu()
        host[name] = t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()
    total = sum(t.numel() * t.element_size() for t in host.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    for name, t in host.items():
        np.save(out_dir / f"{name}.npy", t.numpy())


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


class Job:
    """Per-process context: ranks, device, clock sampler."""

    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dev = None
        self.sampler = None
        self.flush_buf = None

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.world > 1:
            t = torch.tensor([v], device=self.dev, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            return float(t)
        return v

    def flush_l2(self):
        if self.flush_buf is None:
            self.flush_buf = torch.empty(64 * 1024 * 1024, device=self.dev)  # 256 MB > 126 MB L2
        self.flush_buf.zero_()


def run_workload(job: Job, key: str, batch: int, steps: int, warmup: int, headline: bool, latency: bool = False,
                 ckpt: str = None, cpu_budget_s: float = 3.0, math: str = None, dump_dir: str = None):
    """One workload on this job's ranks -> record (dict).  Also returns the model for the headline's kernel rooflines.
    dump_dir: write the last timed step's outputs there (dump_outputs)."""
    from robocupvision_b200 import _lib, ops
    from robocupvision_b200.train import EvalStep, TrainStep
    args, dev, world, rank = job.args, job.dev, job.world, job.rank
    wl = WORKLOADS[key]
    model, ckpt_used = build_model(wl, dev, ckpt or wl.get("ckpt"))
    if math:
        model.set_math(math)
    mode = math or args.math
    cw = class_weights(wl)
    nbatches = 8  # rotate distinct input batches; the per-step activation working set is >> L2 except at batch 1
    xs_host = [synth.images(batch, wl["cin"], wl["h"], wl["w"], seed=1234 + 17 * rank + i).pin_memory() for i in range(nbatches)]
    ys_host = [synth.labels_random(batch, wl["h"], wl["w"], seed=4321 + 17 * rank + i).pin_memory() for i in range(nbatches)]
    xs = [t.to(dev) for t in xs_host]
    ys = [t.to(dev) for t in ys_host]
    if wl["train"]:
        o = wl.get("optim") or dict(optimizer="adam", lr=1e-3, l1_decay=1e-6)
        ts = TrainStep(model, cw, use_graph=not args.no_graph, **o)
        ts.broadcast_state(0)
        step = lambda i: ts.step(xs[i % nbatches], ys[i % nbatches])  # noqa: E731
    else:
        ev = EvalStep(model, cw, use_graph=not args.no_graph)
        out = {}

        def step(i):
            out["r"] = ev(xs[i % nbatches], ys[i % nbatches])
    warmup = max(warmup, 3)
    for i in range(warmup):
        step(i)
    job.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    job.barrier()
    row0 = job.sampler.mark() if job.sampler else 0
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    job.barrier()
    ms_total = job.max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / steps
    if dump_dir is not None and rank == 0:
        # what TrainStep.step / EvalStep return, read before anything else runs the model again.  The weights a
        # training step leaves behind are not dumped: weight-gradient atomics and ReLU sign flips make them drift
        # between identical runs (DESIGN.md section 2), far more than the loss does
        if wl["train"]:
            res = {"loss_sums": ts.loss_sums, "l1_sum": ts.l1_sum, "correct": ts.correct}
        else:
            res = dict(out["r"])
        dump_outputs(dump_dir, res)
    extra_steps = 0
    if headline:
        # a timed region shorter than a few sampling periods: keep the same load running (untimed) until three
        # samples have been taken under it, and say so.  Every rank runs this loop (rank 0, which owns the poller,
        # decides; the decision travels through the all-reduce)
        per_round = max(8, int(200.0 / max(ms_step, 1e-3)))  # ~0.2 s of steps
        for _ in range(8):
            need = 1 if (job.sampler is not None and job.sampler.proc and job.sampler.mark() - row0 < 3) else 0
            need = int(job.max_over_ranks(float(need)))
            if not need:
                break
            for i in range(per_round):
                step(i)
            extra_steps += per_round
            job.barrier()
    row1 = job.sampler.mark() if job.sampler else 0
    value = batch * world / (ms_step * 1e-3)
    launches = (ts.kernels_per_step if wl["train"] else
                (ev.kernels_per_call if ev.use_graph else 0)) * steps

    # ---- e2e: pinned host inputs -> H2D -> step -> D2H of the loss, every step ----------------
    # The public pipelined API (TrainStep.step_async / EvalStep.run_async): step i's inputs are copied H2D on a copy
    # stream while step i-1 still computes, and every step's loss is copied D2H behind it and read by the host one
    # step later.  All copies happen inside the timed region, once per step.
    def e2e_loop(n):
        prev = None
        for i in range(n):
            if wl["train"]:
                h = ts.step_async(xs_host[i % nbatches], ys_host[i % nbatches])
                if prev is not None:
                    prev.wait()
            else:
                h = ev.run_async(xs_host[i % nbatches], ys_host[i % nbatches])
                if prev is not None:
                    EvalStep.wait_host(prev)
            prev = h
        return prev.wait() if wl["train"] else EvalStep.wait_host(prev)
    e2e_loop(4)
    job.barrier()
    t0 = time.perf_counter()
    e2e_loop(steps)
    job.barrier()
    e2e_ms = job.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)
    h2d = xs_host[0].numel() * 4 + ys_host[0].numel() * 8
    d2h = 32 if wl["train"] else 16

    pk = peaks()
    roof_step = {"bound": "hbm", "achieved": (wl["mb"] * batch + wl["mb_step"]) * 1e6 / (ms_step * 1e-3) / 1e9,
                 "peak": pk["hbm"], "unit": "GB/s", "peak_is": pk["source"],
                 "algorithmic_mb_per_frame": wl["mb"], "algorithmic_mb_per_step": wl["mb_step"],
                 "tflops": wl["mflop"] * batch * 1e6 / (ms_step * 1e-3) / 1e12}
    roof_step["frac"] = roof_step["achieved"] / roof_step["peak"]
    rec = {"workload": wl["name"], "key": key, "value": value, "unit": "samples/s" if key == "train_lp" else UNIT,
           "n_gpus": world, "batch_per_gpu": batch, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
           "dtype": MATH_DTYPE[mode], "math": mode,
           "weights": f"released checkpoint {ckpt_used}" if ckpt_used else "random init, seed 12345678",
           "e2e": {"value": batch * world / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
           "gpu_launches": int(launches), "roofline_whole_step": roof_step,
           "l2": "8 rotating input batches; per-step activation working set >> 126 MB L2" if batch * wl["mb"] > 252
                 else "8 rotating input batches; working set fits the 126 MB L2 (see latency_ms_l2_flushed)"}
    if wl["train"] and world > 1:
        # how the gradient buckets are summed: "peer" = rcv_peer_allreduce over NVLink peer memory, "nccl" = dist.all_reduce
        rec["dp_reduce"] = ts.reduce
        if ts.peer is not None:
            ts.peer.check()
    if latency:
        # per-frame latency, the reference's own inference metric (tester.py:142-144): each iteration timed alone with
        # CUDA events; once with the L2 flushed before every iteration (cold weights), once warm
        def timed(flush):
            ts_ms = []
            for i in range(max(10, min(steps, 50))):
                if flush:
                    job.flush_l2()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step(i)
                b.record()
                torch.cuda.synchronize()
                ts_ms.append(a.elapsed_time(b))
            ts_ms.sort()
            return ts_ms[len(ts_ms) // 2]
        rec["latency_ms_l2_flushed"] = timed(True) / batch
        rec["latency_ms_warm"] = timed(False) / batch
        t0 = time.perf_counter()
        n = 20
        for i in range(n):
            EvalStep.wait_host(ev.run_async(xs_host[i % nbatches], ys_host[i % nbatches]))
        rec["latency_ms_host_to_host"] = (time.perf_counter() - t0) * 1e3 / n / batch
    if math:
        rec["key"] = f"{key}_{math}"
        rec["note"] = "fast math mode, stated separately from the fp32-parity record of the same workload (tests/test_gpu_fast_math.py holds its tolerances)"
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not math:
        # bounded sample: at most 64 frames per CPU step, a few seconds of steps
        cb = min(batch, 64)
        fps, ms, threads, kind, n = cpu_reference(wl, cb, 12 if headline else 6, 1, ckpt or wl.get("ckpt"),
                                                  budget_s=None if headline else cpu_budget_s)
        rec["cpu_baseline"] = {"value": fps, "unit": rec["unit"], "cores": threads, "kind": kind, "ms_per_step": ms,
                               "sample": f"{n} steps of batch {cb} after 1 warm-up ("
                                         + ("the unmodified reference classes (baseline/_ref/model.py)" if kind == "reference"
                                            else "oracle port of the reference step") + f", torch {torch.__version__} CPU)"}
    if headline:
        rec["_clock_rows"] = (row0, row1, extra_steps)
    # release this workload's graphs / arenas before the next one
    return rec, model


def main():
    # stdout carries exactly one JSON line: everything else that writes to file descriptor 1 (NCCL's version
    # banner at NCCL_DEBUG=VERSION/WARN, library chatter) is sent to stderr for the whole run
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--math", default="parity", choices=list(MATH_DTYPE),
                    help="parity: fp32-level accuracy (3xTF32 tensor-core tiles); tf32 / bf16: the fast modes, reported "
                         "separately (their own tolerance tests)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--extra-steps", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference arm only times")
    if args.math != "parity":
        os.environ["RCV_B200_MATH"] = args.math
    wl = WORKLOADS[args.workload]
    batch = args.batch or wl["batch"]
    job = Job(args)
    rank, world = job.rank, job.world
    metric = METRIC if args.workload == "train" else f"{args.workload}_frames_per_sec"
    if args.math != "parity":
        metric += "_" + args.math

    if args.impl == "reference":
        if rank != 0:
            return 0
        # exactly --steps timed steps after --warmup untimed ones (a CPU step takes 0.2-2 s)
        steps, warm = args.steps, args.warmup
        cb = min(batch, 64)
        fps, ms, threads, kind, n = cpu_reference(wl, cb, steps, warm, wl.get("ckpt"))
        sample = (f"{n} steps of batch {cb} after {warm} warm-up ("
                  + ("the unmodified reference classes, baseline/_ref/model.py" if kind == "reference" else "oracle port")
                  + f", torch {torch.__version__} CPU)")
        line = {"impl": "reference", "metric": metric, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": n,
                "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl["name"], "batch_per_gpu": cb, "host_threads": threads},
                "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
                "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return 0

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: the product path has no CPU fallback")
    from robocupvision_b200 import _lib, dp
    lib = _lib.load()
    torch.cuda.set_device(job.local_rank)
    job.dev = dev = torch.device("cuda", job.local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=dev)
    # nvidia-smi needs a few hundred ms before its first row: start it ahead of the warm-up, keep the rows that
    # arrive from the start of the timed region on
    if rank == 0:  # one poller per job (rank 0's GPU): NVML queries are not free
        job.sampler = ClockSampler(job.local_rank)
        job.sampler.start()

    rec, model = run_workload(job, args.workload, batch, args.steps, args.warmup, headline=True,
                              dump_dir=args.dump_outputs)
    row0, row1, extra_steps = rec.pop("_clock_rows")
    clocks = job.sampler.summary(row0, row1) if job.sampler else {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    clocks["window"] = "timed region" if extra_steps == 0 else f"timed region + {extra_steps} untimed steps of the same load"
    pk = peaks()
    line = {"metric": metric, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": rec["warmup"], "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": MATH_DTYPE[args.math], "data": "synthetic",
            "config": {"workload": wl["name"], "batch_per_gpu": batch, "global_batch": batch * world,
                       "input": f"{wl['cin']}x{wl['h']}x{wl['w']}", "parallelism": f"dp{world}",
                       "math": args.math, "cuda_graph": bool(not args.no_graph),
                       "programmatic_dependent_launch": bool(lib.rcv_get_pdl()),
                       "l2": rec["l2"], "peaks": pk["source"]},
            "clocks": clocks, "e2e": rec["e2e"], "gpu_launches": rec["gpu_launches"],
            "roofline": dominant_kernel_roofline(model, wl, batch, dev, pk),
            "roofline_whole_step": rec["roofline_whole_step"],
            "roofline_hbm_layer": narrow_layer_roofline(model, wl, batch, dev, pk)}
    if "cpu_baseline" in rec:
        line["cpu_baseline"] = rec["cpu_baseline"]
    if "dp_reduce" in rec:
        line["config"]["gradient_exchange"] = {
            "peer": "rcv_peer_allreduce: one kernel per bucket over NVLink peer-mapped gradient arenas",
            "nccl": "dist.all_reduce (NCCL) per bucket"}[rec["dp_reduce"]]
    del model
    if world > 1 and wl["train"]:
        # numerical check of the N-rank product path (bucketed all-reduce + optimiser on the comm stream, inside a
        # CUDA graph) against serial N-shard gradient accumulation on one GPU
        from robocupvision_b200 import model as M
        ctor = {"ROBO_UNet": lambda: M.ROBO_UNet(**wl["kw"]), "PB_FCN": lambda: M.PB_FCN(32, 5, 1, wl["kw"].get("noScale", False), 0),
                "LabelProp": lambda: M.LabelProp(5, 32, 0)}[wl["net"]]
        try:
            line["dp_check"] = dp.self_check(ctor, class_weights(wl), 8, wl["cin"], wl["h"], wl["w"], steps=3,
                                             force_comm_path=False)
        except Exception as e:  # noqa: BLE001  (every rank raises or none: the check is symmetric)
            line["dp_check"] = {"ok": False, "error": repr(e)}
    if not args.no_extras and args.workload == "train":
        line["extra"] = []
        for key, b, lat, ck, mth in (EXTRAS_1GPU if world == 1 else EXTRAS_NGPU):
            if mth and args.math != "parity":
                continue
            torch.cuda.empty_cache()
            try:
                r, m = run_workload(job, key, b, args.extra_steps, 5, headline=False, latency=lat, ckpt=ck, math=mth)
                del m
            except Exception as e:  # noqa: BLE001
                r = {"workload": WORKLOADS[key]["name"], "key": key, "batch_per_gpu": b, "error": repr(e)}
            line["extra"].append(r)
    if job.sampler:
        job.sampler.stop()
    if rank == 0:
        emit(line)
    if world > 1:
        # NCCL communicators referenced by captured CUDA graphs can stall destroy_process_group()
        # at interpreter teardown (seen on 2xB200: line printed, ranks never exited).  All ranks
        # meet once more, drain their streams and leave without running the teardown.
        torch.distributed.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def _time_alone(fn, job_dev, n=13, skip=3):
    """Mean CUDA-event duration of fn() on the current stream, L2 flushed before every launch."""
    flush = torch.empty(64 * 1024 * 1024, device=job_dev)  # 256 MB > L2
    times = []
    for i in range(n):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= skip:
            times.append(e0.elapsed_time(e1))
    return sum(times) / len(times)


def _traffic(key):
    for name in ("r2_traffic.json", "r1_traffic.json"):
        f = ROOT / "profiles" / name
        if f.exists():
            ent = json.loads(f.read_text()).get(key)
            if ent:
                return ent
    return None


def dominant_kernel_roofline(model, wl, batch, dev, pk):
    """Time the kernel that dominates the step -- the implicit-GEMM conv on the widest layer --
    with CUDA events on the launching stream, on this workload's real tensors."""
    from robocupvision_b200 import engine, ops
    plan = model._get_plan()
    math = plan.math
    # widest conv node = most flops per launch
    best, best_fl = None, -1
    h, w = wl["h"], wl["w"]
    shapes = {0: (wl["cin"], h, w)}
    for t, nd in enumerate(plan.nodes):
        c, hh, ww = shapes[nd.src]
        if nd.kind == "pool":
            shapes[t + 1] = (c, hh // 2, ww // 2)
            continue
        ho, wo = nd.geom.out_hw(hh, ww)
        cout = nd.geom.cout * (2 if nd.skip_mode == "cat" and nd.skip >= 0 else 1)
        shapes[t + 1] = (cout, ho, wo)
        px = hh * ww if nd.geom.transposed else ho * wo
        fl = 2.0 * nd.geom.cin * nd.geom.cout * nd.geom.k ** 2 * px
        if fl > best_fl:
            best, best_fl, best_in = nd, fl, (c, hh, ww)
    g = best.geom
    x = torch.randn(batch, *best_in, device=dev)
    wt = best.conv.weight.detach()
    ho, wo = g.out_hw(best_in[1], best_in[2])
    y = torch.empty(batch, g.cout, ho, wo, device=dev)
    eng = ops.conv_engine(g, batch, best_in[1], best_in[2], ops.PACK_FWD, math)
    on_tc = eng == ops.ENGINE_UMMA
    wp = ops.conv_pack(g, wt, ops.PACK_FWD, math=math, nhw=(batch, best_in[1], best_in[2])) if on_tc else None
    ws = plan.workspace((batch, h, w), dev)  # the plan's conv scratch, as the step itself passes it
    ms = _time_alone(lambda: ops.conv_fwd(g, x, wt, None, epilogue=ops.EPI_RELU, out=y, math=math, wpacked=wp,
                                          workspace=ws), dev)
    flops = best_fl * batch
    bytes_alg = 4.0 * (x.numel() + y.numel() + wt.numel())
    intensity = flops / bytes_alg
    ridge = pk["tensor_sustained"] * 1e12 / (pk["hbm"] * 1e9)
    tfl = flops / (ms * 1e-3) / 1e12
    if intensity >= ridge * 0.5:
        # the burst figure: this kernel is timed alone.  The fp32-parity mode spends three TF32 MMAs per
        # product and TF32 runs at half the bf16 rate, so its ceiling is peak/6 (also reported).
        achieved, peak, unit, bound = tfl, pk["tensor_burst"], "TFLOP/s", "tensor"
    else:
        achieved, peak, unit, bound = bytes_alg / (ms * 1e-3) / 1e9, pk["hbm"], "GB/s", "hbm"
    mode = engine.MATH_NAMES.get(math, str(math))
    out = {"bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak, "traffic": None,
           "kernel": f"{ENGINE_NAMES.get(eng, str(eng))} conv fwd {g.cin}->{g.cout} "
                     f"k{g.k} s{g.stride} d{g.dil} @{best_in[1]}x{best_in[2]} batch {batch}",
           "us_per_launch": ms * 1e3, "flop_per_byte": intensity, "math": mode if on_tc else "fp32 FMA (CUDA cores)",
           "achieved_tflops": tfl, "achieved_gbs": bytes_alg / (ms * 1e-3) / 1e9,
           "peak_is": f"{pk['source']} bf16 dense (burst)", "algorithmic_bytes": bytes_alg}
    ent = _traffic(f"conv fwd {g.cin}->{g.cout} k{g.k} s{g.stride} d{g.dil} @{best_in[1]}x{best_in[2]} batch {batch}")
    if ent:
        out["traffic"], out["traffic_source"] = ent["bytes"], ent["source"]
    if on_tc:
        mmas = {"parity": 3.0, "tf32": 1.0, "bf16": 1.0}.get(engine.MATH_KEYS.get(math, "parity"), 3.0)
        rate = {"parity": 0.5, "tf32": 0.5, "bf16": 1.0}.get(engine.MATH_KEYS.get(math, "parity"), 0.5)
        out["mma_tflops_issued"] = mmas * tfl
        out["mode_ceiling_tflops"] = pk["tensor_burst"] * rate / mmas
        out["frac_of_mode_ceiling"] = tfl / out["mode_ceiling_tflops"]
    return out


def narrow_layer_roofline(model, wl, batch, dev, pk):
    """The HBM-shaped end of the net: the first conv node (3 or 8 input channels at full resolution) on the
    narrow-layer engine (TMA halo staging + FFMA2), timed alone with the L2 flushed, against measured HBM
    bandwidth.  Algorithmic bytes = input read once + output written once + weights (SURVEY.md 8d)."""
    from robocupvision_b200 import ops
    plan = model._get_plan()
    nd = next(n for n in plan.nodes if n.kind == "conv")
    g = nd.geom
    h, w = wl["h"], wl["w"]
    x = torch.randn(batch, g.cin, h, w, device=dev)
    wt = nd.conv.weight.detach()
    ho, wo = g.out_hw(h, w)
    y = torch.empty(batch, g.cout, ho, wo, device=dev)
    eng = ops.conv_engine(g, batch, h, w, ops.PACK_FWD, ops.MATH_AUTO)
    ms = _time_alone(lambda: ops.conv_fwd(g, x, wt, None, epilogue=ops.EPI_RELU, out=y, math=ops.MATH_AUTO), dev)
    bytes_alg = 4.0 * (x.numel() + y.numel() + wt.numel())
    flops = 2.0 * g.cin * g.cout * g.k ** 2 * ho * wo * batch
    gbs = bytes_alg / (ms * 1e-3) / 1e9
    out = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"], "traffic": None,
           "kernel": f"{ENGINE_NAMES.get(eng, str(eng))} conv fwd {g.cin}->{g.cout} k{g.k} s{g.stride} d{g.dil} @{h}x{w} batch {batch}",
           "us_per_launch": ms * 1e3, "algorithmic_bytes": bytes_alg, "flop_per_byte": flops / bytes_alg,
           "fp32_tflops": flops / (ms * 1e-3) / 1e12}
    ent = _traffic(f"conv fwd {g.cin}->{g.cout} k{g.k} s{g.stride} d{g.dil} @{h}x{w} batch {batch}")
    if ent:
        out["traffic"], out["traffic_source"] = ent["bytes"], ent["source"]
    return out


if __name__ == "__main__":
    sys.exit(main())
