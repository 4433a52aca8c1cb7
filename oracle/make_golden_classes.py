"""Generate what tests/test_oracle.py's two reference-class tests compare against:

  tests/golden/reference_classes.npz       outputs on one seeded 2x3x48x64 batch (every 3rd value): each
                                           ROBO_VARIANTS net (seed 3, in turn) in train and then eval mode, plus its
                                           BatchNorm buffers after the train-mode forward; randomly initialised PB_FCN
                                           (both noScale) and FCN in eval mode; CrossEntropyLoss2d on random logits
  tests/golden/reference_module_tree.json  for each tests/nets.py TREE_CASES entry built after seed 5: state_dict keys,
                                           shapes and the sha256 of every initial tensor, parameter order; and
                                           ROBO_UNet().get_computations()

    python -m oracle.make_golden_classes              from the original project's classes (oracle.reference_dir()),
                                                      after checking in the same process that the oracle and the
                                                      drop-in classes reproduce them bit for bit
    python -m oracle.make_golden_classes --from-port  from the drop-in classes and the oracle

The committed files were written with --from-port from an oracle (oracle/ref_model.py) and drop-in classes
(robocupvision_b200/model.py) identical to those that had passed that bit-for-bit comparison with the original.
Everything runs on one CPU thread (fixed accumulation order).
"""
from __future__ import annotations

import hashlib
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
OUT = ROOT / "tests" / "golden"
sys.path.insert(0, str(ROOT / "tests"))

import synth  # noqa: E402
from nets import ROBO_VARIANTS, TREE_CASES  # noqa: E402
from oracle import ref_model as R  # noqa: E402


def _sha(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().contiguous().numpy().tobytes()).hexdigest()


def _buffers(sd) -> np.ndarray:
    return np.concatenate([v.reshape(-1).double().numpy() for k, v in sd.items()
                           if k.endswith(("running_mean", "running_var", "num_batches_tracked"))])


def collect(classes, live: bool = False):
    """-> (arrays, tree) for `classes` (a module with the model.py classes).  Forward outputs are the oracle's, on
    state dicts of `classes`; live=True: `classes` is the original project and its own forwards must equal them."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        return _collect(classes, live)
    finally:
        torch.set_num_threads(threads)


def _collect(classes, live):
    from robocupvision_b200 import model as M
    arrays = {}
    torch.manual_seed(3)
    x = synth.images(2, 3, 48, 64, seed=8)
    with torch.no_grad():
        for tag, (kw, okw) in ROBO_VARIANTS.items():
            m = classes.ROBO_UNet(**kw)
            sd = {k: v.clone() for k, v in m.state_dict().items()}
            for mode in (True, False):
                y = R.robo_unet_forward(sd, x, training=mode, **okw)  # train mode updates sd's BatchNorm buffers
                if live:
                    m.train(mode)
                    assert torch.equal(m(x), y), (tag, mode)
                    assert all(torch.equal(v, sd[k]) for k, v in m.state_dict().items()), (tag, mode)
                arrays[f"{tag}_{'train' if mode else 'eval'}"] = y.reshape(-1)[::3].numpy().copy()
                if mode:
                    arrays[f"{tag}_buffers"] = _buffers(sd)
        for ns in (False, True):
            m = classes.PB_FCN(32, 5, 1, ns, 0).eval()
            y = R.pb_fcn_forward(m.state_dict(), x, ns)
            if live:
                assert torch.equal(m(x), y), ns
            arrays[f"pb_fcn_noscale{int(ns)}_eval"] = y.reshape(-1)[::3].numpy().copy()
        m = classes.FCN().eval()
        y = R.fcn_forward(m.state_dict(), x)
        if live:
            assert torch.equal(m(x), y)
        arrays["fcn_eval"] = y.reshape(-1)[::3].numpy().copy()
    labels = synth.labels_random(2, 48, 64)
    w = torch.tensor(synth.CLASS_WEIGHTS)
    lg = torch.randn(2, 5, 48, 64)
    loss = R.cross_entropy_2d(lg, labels, w)
    if live:
        assert torch.equal(classes.CrossEntropyLoss2d(w)(lg, labels), loss)
    arrays["cross_entropy_2d"] = np.array(float(loss))

    tree = {"cases": [], "computations": classes.ROBO_UNet().get_computations()}
    for name, args, kw in TREE_CASES:
        torch.manual_seed(5)
        m = getattr(classes, name)(*args, **kw)
        sd = m.state_dict()
        tree["cases"].append({"class": name, "args": list(args), "kwargs": kw, "keys": list(sd),
                              "shapes": [list(v.shape) for v in sd.values()], "sha256": [_sha(v) for v in sd.values()],
                              "params": [n for n, _ in m.named_parameters()]})
    if live:
        port = collect(M)[1]
        assert json.loads(json.dumps(port)) == json.loads(json.dumps(tree)), \
            "the drop-in module tree differs from the original's"
    return arrays, tree


def main():
    if "--from-port" in sys.argv:
        from robocupvision_b200 import model as classes
        live = False
    else:
        from oracle import reference_dir
        sys.path.insert(0, str(reference_dir()))
        import model as classes  # the original project's model.py
        live = True
    arrays, tree = collect(classes, live)
    np.savez_compressed(OUT / "reference_classes.npz", **arrays)
    (OUT / "reference_module_tree.json").write_text(json.dumps(tree, separators=(",", ":")) + "\n")
    print({k: v.shape for k, v in arrays.items()}, len(tree["cases"]), "module trees")


if __name__ == "__main__":
    main()
