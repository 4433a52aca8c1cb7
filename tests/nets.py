"""Builders shared by the model-level tests: the same net as (a) an oracle state dict on the
CPU and (b) the drop-in module, from released checkpoints or from the reference's seed."""
from __future__ import annotations

import torch

import synth
from oracle import ref_model as R
from util import load_ckpt, with_nbt

ROBO_VARIANTS = {
    "robo_default": (dict(), dict()),
    "robo_unet_pool": (dict(pool=True, levels=3, bellySize=0), dict(pool=True, levels=3, belly_size=0)),
    "robo_noscale": (dict(noScale=True), dict(no_scale=True)),
}

# (class name, args, kwargs) of the module trees pinned against the original project's classes
# (tests/golden/reference_module_tree.json, oracle/make_golden_classes.py)
TREE_CASES = ([("ROBO_UNet", (), kw) for kw, _ in ROBO_VARIANTS.values()]
              + [("ROBO_UNet", (), dict(v2=True, levels=1, bellySize=9, classSize=3, bellyPlanes=64))]
              + [("PB_FCN", (32, 5, 1, ns, 0), {}) for ns in (False, True)]
              + [("FCN", (), {}), ("DownSampler", (32, False), {})])


def robo_state(tag):
    """Seed 12345678 init (train.py:332-337) + three oracle training forwards so the running
    statistics are not the identity -- exactly what oracle/make_golden.py did with the reference."""
    from robocupvision_b200.model import ROBO_UNet
    kw, okw = ROBO_VARIANTS[tag]
    torch.manual_seed(12345678)
    m = ROBO_UNet(**kw)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    with torch.no_grad():
        for s in range(3):
            R.robo_unet_forward(sd, synth.images(4, 3, 48, 64, seed=77 + s), training=True, **okw)
    return sd, kw, okw


def pb_fcn_state(name):
    """Released PB_FCN checkpoint -> oracle state dict with the head under `segmenter`."""
    sd = load_ckpt(name)
    out = {}
    for k, v in sd.items():
        out[("segmenter." + k[len("classifier."):]) if k.startswith("classifier.classifier.") else k] = v
    return with_nbt(out), sd
