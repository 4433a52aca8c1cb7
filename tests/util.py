"""Shared helpers for the parity tests."""
from __future__ import annotations

from pathlib import Path

import numpy as np
import torch

GOLDEN = Path(__file__).resolve().parent / "golden"
LOGIT_TOL = 1e-4


def max_err(a: torch.Tensor, b: torch.Tensor) -> float:
    return float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max())


def assert_close(name, got, ref, tol=1e-5, atol=0.0):
    """max |got-ref| <= tol * max(1, max|ref|) + atol  (SURVEY.md section 8c gate shape)."""
    got, ref = got.detach().cpu(), ref.detach().cpu()
    assert got.shape == ref.shape, f"{name}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    err = max_err(got, ref)
    scale = max(1.0, float(ref.abs().max())) if ref.numel() else 1.0
    assert err <= tol * scale + atol, f"{name}: max err {err:.3e} > {tol:.1e} * {scale:.3e}"
    return err


def check_eval_outputs(tag, out, ref, am_ref, y, loss_ref, num_classes=5):
    """Gates of one validation batch (an EvalStep result `out`) against reference logits `ref` (the oracle's), a
    reference label map `am_ref` and a reference loss: logits within LOGIT_TOL of the logit scale, argmax exact
    outside near-ties (reference top-2 margin below 1e-4), confusion, correct count and IoU sums exact against the
    kernel's own label map, loss within 1e-5 relative.  -> (max logit error, argmax flips)."""
    from oracle import ref_metrics
    logits = out["logits"].cpu()
    err = assert_close(f"{tag} logits", logits, ref, LOGIT_TOL)
    top2 = ref.topk(2, dim=1).values
    margin = top2[:, 0] - top2[:, 1]
    am = out["argmax"].cpu()
    diff = am != am_ref
    assert not bool((diff & (margin >= 1e-4)).any()), f"{tag}: argmax differs outside near-ties"
    conf_own = ref_metrics.confusion_per_image(am.numpy(), y.numpy(), num_classes)
    assert (out["conf"].cpu().numpy() == conf_own).all(), f"{tag}: confusion vs own label map"
    assert int(out["correct"]) == int((am == y).sum())
    assert np.allclose(out["iou_sum"].cpu().numpy(), ref_metrics.iou_sums(conf_own), rtol=0, atol=1e-12)
    loss = float(out["loss"])
    assert abs(loss - loss_ref) <= 1e-5 * max(1.0, abs(loss_ref)), f"{tag}: loss {loss} vs {loss_ref}"
    return err, int(diff.sum())


def tensors_held_by(owner) -> set:
    """ids of the tensors `owner` references: through attributes, containers, modules and the package's own objects
    (plans, nodes, pack tables), not through classes, functions or other modules' globals."""
    seen, held, todo = set(), set(), [owner]
    while todo:
        o = todo.pop()
        if id(o) in seen:
            continue
        seen.add(id(o))
        if isinstance(o, torch.Tensor):
            held.add(id(o))
        elif isinstance(o, dict):
            todo += list(o.values())
        elif isinstance(o, (list, tuple, set)):
            todo += list(o)
        elif isinstance(o, torch.nn.Module) or type(o).__module__.startswith("robocupvision_b200"):
            todo += list(getattr(o, "__dict__", {}).values())
            todo += [getattr(o, s, None) for s in getattr(type(o), "__slots__", ())]
    return held


def load_ckpt(name):
    z = np.load(GOLDEN / "ckpt" / (name + ".npz"))
    return {k: torch.from_numpy(z[k].copy()) for k in z.files}


def load_golden(name):
    z = np.load(GOLDEN / (name + ".npz"))
    return {k: z[k] for k in z.files}


def with_nbt(sd):
    """Add the num_batches_tracked entries pre-0.4.1 checkpoints lack."""
    out = dict(sd)
    for k in list(sd):
        if k.endswith("running_mean"):
            out.setdefault(k[: -len("running_mean")] + "num_batches_tracked", torch.zeros((), dtype=torch.long))
    return out
