"""Host logic of the drop-in modules without a GPU: the execution plan each model family builds (node list, epilogue
orders, skip wiring, outputs), interpreted with ATen CPU ops (tests/plan_interp.py), against the CPU oracle on seeded
inputs -- eval mode and train mode (batch statistics + running-statistic updates)."""
import copy

import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import ref_model as R
from plan_interp import run_plan_cpu


def _warm(sd, fwd_train, cin=3):
    with torch.no_grad():
        for s in range(2):
            fwd_train(sd, synth.images(3, cin, 48, 64, seed=70 + s))
    return sd


def _cases():
    from robocupvision_b200 import model as M
    u = lambda **okw: (lambda sd, x, training=False: R.robo_unet_forward(sd, x, training=training, **okw))  # noqa: E731
    return {
        "robo_default": (lambda: M.ROBO_UNet(), u(), 3),
        "robo_unet_pool": (lambda: M.ROBO_UNet(pool=True, levels=3, bellySize=0), u(pool=True, levels=3, belly_size=0), 3),
        "robo_noscale": (lambda: M.ROBO_UNet(noScale=True), u(no_scale=True), 3),
        "robo_v2": (lambda: M.ROBO_UNet(v2=True, classSize=3), u(v2=True, class_size=3), 3),
        "robo_v2_shallow": (lambda: M.ROBO_UNet(v2=True, levels=1, bellySize=9, classSize=3, bellyPlanes=64, depth=3),
                            u(v2=True, levels=1, belly_size=9, class_size=3, depth=3), 3),
        "pb_fcn_2": (lambda: M.PB_FCN_2(False), u(), 3),
        "pb_fcn": (lambda: M.PB_FCN(32, 5, 1, False, 0),
                   lambda sd, x, training=False: R.pb_fcn_forward(sd, x, False, training), 3),
        "pb_fcn_vga": (lambda: M.PB_FCN(32, 5, 1, True, 0),
                       lambda sd, x, training=False: R.pb_fcn_forward(sd, x, True, training), 3),
        "pb_fcn_channels": (lambda: M.PB_FCN_Channels((16, 16, 16, 32, 64, 64, 128, 64, 32), (16, 16, 16)),
                            lambda sd, x, training=False: R.pb_fcn_forward(sd, x, False, training), 3),
        "fcn": (lambda: M.FCN(), lambda sd, x, training=False: R.fcn_forward(sd, x, training), 3),
        "labelprop": (lambda: M.LabelProp(5, 32, 0), lambda sd, x, training=False: R.labelprop_forward(sd, x, training), 8),
    }


@pytest.mark.parametrize("tag", list(_cases()))
def test_plan_wiring_matches_oracle(tag):
    make, oracle, cin = _cases()[tag]
    torch.manual_seed(12345678)
    m = make()
    sd = _warm({k: v.clone() for k, v in m.state_dict().items()}, lambda s, x: oracle(s, x, training=True), cin)
    m.load_state_dict(sd)
    plan = m._get_plan()
    x = synth.images(2, cin, 48, 64, seed=9)
    with torch.no_grad():
        m.eval()
        got = run_plan_cpu(plan, x, training=False)[0]
        ref = oracle(sd, x)
        assert got.shape == ref.shape
        assert float((got - ref).abs().max()) <= 1e-5 * max(1.0, float(ref.abs().max())), tag
        # train mode: batch statistics in the same places, running statistics updated identically
        m.train()
        sd_t = {k: v.clone() for k, v in sd.items()}
        got_t = run_plan_cpu(plan, x, training=True)[0]
        ref_t = oracle(sd_t, x, training=True)
        assert float((got_t - ref_t).abs().max()) <= 1e-5 * max(1.0, float(ref_t.abs().max())), tag
        for k, v in m.state_dict().items():
            if k.endswith("running_mean") or k.endswith("running_var"):
                assert torch.allclose(v, sd_t[k], rtol=1e-6, atol=1e-7), (tag, k)


def test_downsampler_plan_has_the_five_feature_maps():
    """DownSampler.forward returns (x4|None, x3, x2, x1, x0) (model.py:218-226): the plan's outputs in that order."""
    from robocupvision_b200 import model as M
    for no_scale in (False, True):
        torch.manual_seed(4)
        m = M.DownSampler(32, no_scale).eval()
        sd = {k: v.clone() for k, v in m.state_dict().items()}
        x = synth.images(2, 3, 48, 64, seed=3)
        with torch.no_grad():
            outs = run_plan_cpu(m._get_plan(), x)
            ref = [t for t in R.downsampler_forward(sd, x, no_scale, pfx="") if t is not None]
        assert len(outs) == len(ref)
        for a, b in zip(outs, ref):
            assert a.shape == b.shape and float((a - b).abs().max()) <= 1e-5 * max(1.0, float(b.abs().max()))


def test_deferred_batchnorm_schedule_is_conservative():
    """engine.Plan._defer_bn_apply (normalise-on-load): only blocks whose output feeds tensor-core stride-1 3x3 convs as
    their main input, is not a skip source and not a plan output."""
    from robocupvision_b200 import model as M, ops
    m = M.ROBO_UNet()
    plan = m._get_plan()
    shapes = {0: (64, 3, 120, 160)}
    deferred = []
    for t, nd in enumerate(plan.nodes):
        n, c, h, w = shapes[nd.src]
        if nd.kind == "pool":
            shapes[t + 1] = (n, c, h // 2, w // 2)
            continue
        ho, wo = nd.geom.out_hw(h, w)
        shapes[t + 1] = (n, nd.geom.cout, ho, wo)
        if nd.bn is not None and plan._defer_bn_apply(t, n, ho, wo):
            deferred.append(t)
    assert len(deferred) == 7
    skip_sources = {nd.skip for nd in plan.nodes if nd.kind == "conv" and nd.skip >= 0}
    for t in deferred:
        assert (t + 1) not in plan.outputs and (t + 1) not in skip_sources
        cons = [nd for nd in plan.nodes if nd.src == t + 1]
        assert cons and all(nd.kind == "conv" and nd.geom.k == 3 and nd.geom.stride == 1 and not nd.geom.transposed
                            and nd.geom.cin % 32 == 0 for nd in cons)
        n, c, h, w = shapes[t + 1]
        assert all(ops.conv_normalises_on_load(nd.geom, n, h, w, ops.MATH_AUTO) for nd in cons)


# ------------------------------------------------------------------ the real engine on CPU stand-ins for the kernels
@pytest.fixture
def cpu_engine(monkeypatch):
    """engine.Plan with its kernels replaced by ATen-CPU stand-ins (tests/fake_ops.py); single stream."""
    import fake_ops
    from robocupvision_b200 import engine
    monkeypatch.setattr(engine, "ops", fake_ops)
    monkeypatch.setattr(engine, "WGRAD_SIDE_STREAM", False)
    fake_ops.calls.clear()
    return engine, fake_ops


@pytest.mark.parametrize("wgrad_on_load", [False, True])
@pytest.mark.parametrize("tag", list(_cases()))
def test_engine_schedule_forward_backward_on_cpu(tag, wgrad_on_load, cpu_engine, monkeypatch):
    """Plan.forward(training) + Plan.backward -- the code the GPU runs, including the normalise-on-load schedule --
    against autograd over the oracle: logits, every parameter gradient, input gradient, running statistics."""
    engine, fake = cpu_engine
    monkeypatch.setattr(engine, "WGRAD_ON_LOAD", wgrad_on_load)
    make, oracle, cin = _cases()[tag]
    torch.manual_seed(12345678)
    m = make().train()
    sd = _warm({k: v.clone() for k, v in m.state_dict().items()}, lambda s, x: oracle(s, x, training=True), cin)
    m.load_state_dict(sd)
    # batch / size at which the tensor-core layers are eligible for normalise-on-load (host logic of the library)
    # (the five-level nets need H, W divisible by 32)
    h, w = (96, 128) if tag in ("robo_noscale", "pb_fcn_vga") else (120, 160)
    x = synth.images(8, cin, h, w, seed=11)
    y = synth.labels_learnable(x)

    def oracle_grads(dtype):
        """Autograd over the oracle in `dtype` -> (logits, d loss / d logits, state with .grad, d loss / d x)."""
        osd = R.leaf_state_dict({k: (v.clone().to(dtype) if v.is_floating_point() else v.clone()) for k, v in sd.items()})
        xr = x.detach().clone().to(dtype).requires_grad_(True)
        ref = oracle(osd, xr, training=True)
        # the gradient the training step feeds in: weighted cross entropy (train.py:52-56)
        lg = ref.detach().requires_grad_(True)
        R.cross_entropy_2d(lg, y, torch.tensor(synth.CLASS_WEIGHTS, dtype=dtype)).backward()
        ref.backward(lg.grad)
        return ref.detach(), lg.grad, osd, xr.grad

    ref, gout, osd, dx_ref = oracle_grads(torch.float32)
    _, _, osd64, dx64 = oracle_grads(torch.float64)

    plan = m._get_plan()
    with torch.no_grad():
        outs, saved = plan.forward(x, training=True, save=True)
        dx, gv = plan.backward(saved, [gout], x_needs_grad=True)
    assert float((outs[0] - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
    # Gate.  This test is about wiring (which tensor feeds which kernel, which gradient goes where): an error there is
    # O(1) on whole tensors.  Element-wise fp32 agreement is the GPU tests' business and is not attainable here at
    # full size: a ReLU that follows a BatchNorm flips on values within an ulp of zero (about one pixel per run at
    # 8 x 128 x 15 x 20 x 10 layers), which moves one output channel's gradient by a few per cent and everything
    # below it by ~1e-3 -- the fp32 oracle shows the same against the fp64 oracle.  So: relative L2 error per tensor
    # <= 1e-2 against the fp64 oracle, or within 4x the fp32 oracle's own deviation, whichever is larger.
    gmax = max(float(v.grad.abs().max()) for v in osd64.values() if v.grad is not None)
    # a conv bias feeding a train-mode BatchNorm directly (upSampleTransposeConv, model.py:191-193) has an exactly
    # zero true gradient: both sides hold rounding noise there
    from robocupvision_b200.model import upSampleTransposeConv
    noise = {f"{n}.conv.bias" for n, mod in m.named_modules() if isinstance(mod, upSampleTransposeConv)}

    def rel_l2(a, b):
        den = max(float(b.norm()), 1e-3 * gmax * b.numel() ** 0.5)
        return float((a.double() - b).norm()) / den

    for k, p in m.named_parameters():
        if osd64[k].grad is None or k in noise:
            continue
        g64 = osd64[k].grad
        err, floor = rel_l2(gv[id(p)], g64), rel_l2(osd[k].grad, g64)
        assert err <= max(1e-2, 4 * floor), f"{tag}: grad {k} rel L2 err {err:.3e} (fp32 oracle {floor:.3e})"
    assert rel_l2(dx, dx64) <= max(1e-2, 4 * rel_l2(dx_ref, dx64))
    for k, b in m.named_buffers():
        if b.is_floating_point():
            assert torch.allclose(b, osd[k], rtol=1e-5, atol=1e-6), (tag, k)
        else:
            assert int(b) == int(osd[k]), (tag, k)
    # the schedule: every deferred block is consumed on load, and materialised for a weight gradient only when that
    # gradient cannot normalise on load itself
    n_def = sum(plan._defer_cache.values())
    on_load = sum(1 for c in fake.calls if c == ("conv_fwd", True))
    assert (n_def > 0) == (on_load > 0)
    if tag == "robo_default":
        assert n_def == 7
    if wgrad_on_load:
        assert sum(1 for c in fake.calls if c == ("conv_wgrad", True)) == on_load
        assert sum(1 for c in fake.calls if c[0] == "bn_apply") == 0
    else:
        assert sum(1 for c in fake.calls if c == ("conv_wgrad", True)) == 0
        assert sum(1 for c in fake.calls if c[0] == "bn_apply") == n_def


def test_engine_eval_forward_on_cpu(cpu_engine):
    """Eval-mode plan (folded BatchNorm in the conv epilogue, no deferral) on the stand-ins == oracle."""
    engine, fake = cpu_engine
    for tag in ("robo_default", "robo_v2", "fcn", "pb_fcn_vga", "labelprop"):
        make, oracle, cin = _cases()[tag]
        torch.manual_seed(12345678)
        m = make()
        sd = _warm({k: v.clone() for k, v in m.state_dict().items()}, lambda s, x: oracle(s, x, training=True), cin)
        m.load_state_dict(sd)
        m.eval()
        x = synth.images(2, cin, 48, 64, seed=12)
        with torch.no_grad():
            outs, saved = m._get_plan().forward(x, training=False, save=False)
            ref = oracle(sd, x)
        assert saved is None and not any(c == ("conv_fwd", True) for c in fake.calls)
        assert float((outs[0] - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max())), tag


def _golden_eval_on_cpu(m, g, cin=3):
    """The module's plan, interpreted on the CPU, against the reference's golden logits / label maps."""
    import numpy as np
    i = 0
    while f"shape{i}" in g:
        n, c, h, w = (int(v) for v in g[f"shape{i}"])
        x = synth.images(n, c, h, w, seed=1234 + i)
        with torch.no_grad():
            logits = run_plan_cpu(m._get_plan(), x)[0]
        lf = logits.reshape(-1)
        sub = lf[::13] if lf.numel() > 50000 else lf
        gs = torch.from_numpy(g[f"logits_sub{i}"])
        assert float((sub - gs).abs().max()) <= 1e-4 * float(g[f"logits_absmax{i}"])
        am = logits.argmax(1)
        am_ref = torch.from_numpy(g[f"argmax{i}"].astype(np.int64))
        top2 = logits.topk(2, dim=1).values
        assert not bool(((am != am_ref) & ((top2[:, 0] - top2[:, 1]) >= 1e-4)).any())
        i += 1
    return i


def test_released_fcn_and_labelprop_checkpoints_through_the_plan():
    """pth/bestModelSeg1.pth (FCN, model.py:311-331) and pth/bestModelLPFinetunedPruned.pth (LabelProp) loaded into
    the drop-in classes: the plan reproduces the reference's golden outputs on the CPU."""
    from robocupvision_b200 import model as M
    from util import load_ckpt, load_golden
    m = M.FCN()
    M.load_legacy_state_dict(m, load_ckpt("bestModelSeg1"))
    assert _golden_eval_on_cpu(m.eval(), load_golden("bestModelSeg1_eval")) == 2
    lp = M.LabelProp(5, 32, 0)
    M.load_legacy_state_dict(lp, load_ckpt("bestModelLPFinetunedPruned"))
    assert _golden_eval_on_cpu(lp.eval(), load_golden("bestModelLPFinetunedPruned_eval")) == 2


@pytest.mark.parametrize("name", ["bestModelSeg", "bestModelSegFinetunedPruned", "bestModelSegFinetunedPruned_bu"])
def test_released_checkpoint_through_the_plan_matches_reference_golden(name):
    """Released PB_FCN-family checkpoints (incl. the channel-pruned `_bu` file no reference class loads) built with
    PB_FCN_Channels.from_state_dict: widths read off the shapes, legacy head name, no num_batches_tracked.  The
    module's plan, interpreted on the CPU, reproduces the REFERENCE's golden logits / label maps / confusion."""
    import numpy as np
    from robocupvision_b200 import model as M
    from util import load_ckpt, load_golden
    raw = load_ckpt(name)
    m = M.PB_FCN_Channels.from_state_dict(raw).eval()
    if name.endswith("_bu"):
        assert m.enc == (16, 16, 16, 32, 64, 64, 128, 64, 32) and m.ups == (16, 16, 16)
        assert sum(p.numel() for p in m.parameters()) == 252661
    else:  # the regular checkpoints describe PB_FCN(32, 5, 1, False, 0)
        ref = M.PB_FCN(32, 5, 1, False, 0)
        assert [tuple(p.shape) for p in m.parameters()] == \
               [tuple(p.shape) for n, p in ref.named_parameters() if not n.startswith("classifier.")]
    assert _golden_eval_on_cpu(m, load_golden(name + "_eval")) == 2


def test_every_released_checkpoint_layout_loads():
    """tests/golden/pth_manifest.json (oracle/make_pth_manifest.py: keys, shapes, dtypes of all 18 pth/*.pth of the
    reference): each file of the segmentation / label-propagation path loads strictly -- same keys in the same
    order, same shapes -- into the class it belongs to (SURVEY.md section 2 row 25); the three files of the
    patch-classification baselines are out of scope."""
    import json
    from robocupvision_b200 import model as M
    from util import GOLDEN
    man = json.loads((GOLDEN / "pth_manifest.json").read_text())
    assert len(man) == 18

    def owner(name):
        if name in ("bestClass", "bestModelHessL", "bestModelHessMC"):
            return None
        if name.endswith("_bu"):
            return "channels"
        if name.startswith("bestModelSegVGA"):
            return M.PB_FCN(32, 5, 1, True, 0)
        if name.startswith("bestModelSeg1"):
            return M.FCN()
        if name.startswith("bestModelSeg"):
            return M.PB_FCN(32, 5, 1, False, 0)
        if name.startswith("bestModelLP"):
            return M.LabelProp(5, 32, 0)
        return M.DownSampler(32, name == "bestModelVGA")

    loaded = 0
    for name, info in man.items():
        sd = {k: torch.full(shape, 0.5, dtype=getattr(torch, dt)) for k, shape, dt in info["entries"]}
        m = owner(name)
        if m is None:
            continue
        if m == "channels":
            m = M.PB_FCN_Channels.from_state_dict(sd)
        else:
            missing, unexpected = M.load_legacy_state_dict(m, sd)   # strict: raises on any mismatch
            assert missing == [] and unexpected == []
        # the same parameter set as the file (the legacy files list keys in their own order; load is by name)
        file_params = [k for k, _, _ in info["entries"] if not k.endswith(("running_mean", "running_var"))]
        file_params = [("segmenter." + k[len("classifier."):]) if k.startswith("classifier.classifier.") and
                       not isinstance(m, M.FCN) else k for k in file_params]
        own = [n for n, _ in m.named_parameters() if not (isinstance(m, M.PB_FCN) and n.startswith("classifier."))]
        assert sorted(own) == sorted(file_params), name
        assert all(float(p.detach().reshape(-1)[0]) == 0.5 for n, p in m.named_parameters()
                   if not (isinstance(m, M.PB_FCN) and n.startswith("classifier."))), name
        loaded += 1
    assert loaded == 15


def test_net_cfg_emitted_from_the_plan_matches_the_reference_files():
    """export.net_cfg (paramSave.py's companion file: the layer list an external engine reads next to weights.dat)
    emitted from the module's own plan == the reference's hand-written weights/net.cfg (PB_FCN 160x120),
    weightsVGA/net.cfg (PB_FCN 640x480) and weightsLP/net.cfg (LabelProp): same sections, keys, values, order, and the
    same text up to trailing blank lines (tests/golden/netcfg_manifest.json, oracle/make_pth_manifest.py)."""
    import hashlib
    import json
    from robocupvision_b200 import export as E, model as M
    from util import GOLDEN
    man = json.loads((GOLDEN / "netcfg_manifest.json").read_text())
    cases = {"weights": (M.PB_FCN(32, 5, 1, False, 0), {}),
             "weightsVGA": (M.PB_FCN(32, 5, 1, True, 0), dict(height=480, width=640)),
             "weightsLP": (M.LabelProp(5, 32, 0), {})}
    for name, (m, kw) in cases.items():
        text = E.net_cfg(m, **kw)
        got = [[sec, [[k, str(v)] for k, v in kvs]] for sec, kvs in E.net_cfg_sections(m, **kw)]
        assert got == man[name]["sections"], name
        assert [[s, [list(kv) for kv in kvs]] for s, kvs in E.parse_net_cfg(text)] == man[name]["sections"]
        assert hashlib.sha256(text.rstrip().encode()).hexdigest() == man[name]["sha256_rstrip"], name
    # the pair (net.cfg, weights.dat) is consistent: the values the layer list implies == the flatten's length
    lp = cases["weightsLP"][0]
    cin, n = 8, 0
    for sec, kvs in E.net_cfg_sections(lp):
        kv = dict(kvs)
        if sec in ("convolutional", "transposedconv"):
            bias = sec == "transposedconv" or "hasBias" not in kv
            n += kv["filters"] * cin * kv["size"] ** 2 + (kv["filters"] if bias else 0)
            cin = kv["filters"]
        elif sec == "batchnorm":
            n += 4 * cin
    assert n == int(json.loads((GOLDEN / "pth_manifest.json").read_text())["bestModelLPFinetunedPruned"]["params"])
    # nets the reference ships no cfg for: --UNet pools, --v2 routes, ROBO_UNet's conv -> ReLU -> BatchNorm order
    secs = [s for s, _ in E.net_cfg_sections(M.ROBO_UNet(pool=True, levels=3, bellySize=0))]
    assert secs.count("maxpool") == 3 and secs[-1] == "softmax"
    secs = E.net_cfg_sections(M.ROBO_UNet(v2=True, classSize=3))
    assert [s for s, _ in secs].count("route") == 3 and [s for s, _ in secs].count("shortcut") == 0
    d = E.net_cfg_sections(M.ROBO_UNet())
    assert d[1] == ("convolutional", [("filters", 8), ("size", 3), ("stride", 1), ("pad", 1), ("activation", "relu")])
    assert d[2] == ("batchnorm", [("activation", "linear")])


def test_engine_backward_side_stream_code_path_on_cpu(cpu_engine, monkeypatch):
    """The weight-gradient side-stream branch of Plan.backward (the default on the GPU) with torch.cuda's stream
    objects replaced by inert stand-ins: same gradients as the single-stream branch, every tensor the side stream
    reads is kept alive until the join, and the streams are joined exactly once."""
    import contextlib
    engine, fake = cpu_engine
    log = []

    class Stream:
        def __init__(self, device=None):
            self.device = device

        def wait_stream(self, other):
            log.append(("wait", self is main, other is main))

    main = Stream(torch.device("cpu"))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: main)
    monkeypatch.setattr(torch.cuda, "Stream", Stream)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    make, oracle, cin = _cases()["robo_default"]
    res = {}
    for side in (False, True):
        monkeypatch.setattr(engine, "WGRAD_SIDE_STREAM", side)
        torch.manual_seed(12345678)
        m = make().train()
        x = synth.images(8, cin, 120, 160, seed=11)
        gout = torch.randn(8, 5, 120, 160, generator=torch.Generator().manual_seed(4)) * 1e-3
        plan = m._get_plan()
        log.clear()
        with torch.no_grad():
            outs, saved = plan.forward(x, training=True, save=True)
            dx, gv = plan.backward(saved, [gout], x_needs_grad=True)
        res[side] = (dx, [gv[id(p)].clone() for p in m.parameters()], list(log))
    assert torch.equal(res[True][0], res[False][0])
    assert all(torch.equal(a, b) for a, b in zip(res[True][1], res[False][1]))
    assert res[False][2] == []
    waits = res[True][2]
    n_conv = sum(1 for nd in plan.nodes if nd.kind == "conv")
    assert waits.count(("wait", False, True)) == n_conv      # side waits for main before every weight gradient
    assert waits.count(("wait", True, False)) == 1 and waits[-1] == ("wait", True, False)   # one join, at the end


def test_graph_owner_keeps_the_plan_buffers_its_capture_baked_in(cpu_engine, monkeypatch):
    """EvalStep(use_graph=True) at batch 4, then 8, on the engine with size-dependent stand-ins for the workspace and
    panel sizes (every conv a tensor-core layer) and torch.cuda's graph and stream objects replaced by inert ones:
    the second size makes Plan.workspace return a larger buffer and replaces every panel and the pack table.  The
    tensors Plan.capture_refs returned before are then still referenced through the EvalStep, and freed once it is
    dropped."""
    import contextlib
    import gc
    import weakref

    from robocupvision_b200 import train
    from util import tensors_held_by
    engine, fake = cpu_engine

    class PackTable:
        def __init__(self, jobs, math=None, sizes=None):
            self.table = torch.zeros(64 * len(jobs), dtype=torch.uint8)

        def run(self):
            pass

    class Stream:
        def __init__(self, device=None):
            pass

        def wait_stream(self, other):
            pass

    class Graph:
        def replay(self):
            pass

    monkeypatch.setattr(fake, "conv_uses_tensor_cores", lambda g, direction, math=None: True)
    monkeypatch.setattr(fake, "conv_workspace_bytes", lambda g, n, h, w, direction=0, math=None: 4096 * n * h * w // 3072)
    monkeypatch.setattr(fake, "new_workspace", lambda nbytes, dev: torch.zeros(max(nbytes, 1024), dtype=torch.uint8))
    monkeypatch.setattr(fake, "conv_packed_bytes",
                        lambda g, direction, math=None, nhw=None: 4 * g.cin * g.cout * g.k * g.k + 256 * nhw[0])
    monkeypatch.setattr(fake, "PackTable", PackTable)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: Stream())
    monkeypatch.setattr(torch.cuda, "Stream", Stream)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "synchronize", lambda device=None: None)
    monkeypatch.setattr(torch.cuda, "CUDAGraph", Graph)
    monkeypatch.setattr(torch.cuda, "graph", lambda g: contextlib.nullcontext())
    monkeypatch.setattr(train.EvalStep, "_eager",
                        lambda self, x, y: {"logits": self.model._get_plan().forward(x, training=False, save=False)[0][0]})
    make, _, cin = _cases()["robo_default"]
    torch.manual_seed(12345678)
    m = make().eval()
    plan = m._get_plan()
    es = train.EvalStep(m, use_graph=True)
    with torch.no_grad():
        es(synth.images(4, cin, 48, 64, seed=1), synth.labels_random(4, 48, 64))
        ws4 = plan.workspace((4, 48, 64), torch.device("cpu"))
        refs = plan.capture_refs()
        assert any(t is ws4 for t in refs)
        assert len(refs) == 1 + sum(1 for nd in plan.nodes if nd.kind == "conv") + len(plan._pack_tables)
        es(synth.images(8, cin, 48, 64, seed=2), synth.labels_random(8, 48, 64))
        ws8 = plan.workspace((8, 48, 64), torch.device("cpu"))
    assert ws8 is not ws4 and ws8.numel() > ws4.numel()
    # every buffer of the first capture was replaced: the plan holds none of them, the EvalStep holds all of them
    assert not {id(t) for t in refs} & {id(t) for t in plan.capture_refs()}
    held = tensors_held_by(es)
    assert all(id(t) in held for t in refs), "the EvalStep must hold every buffer its graphs baked in"
    dead = [weakref.ref(t) for t in refs]
    del refs, ws4, es
    gc.collect()
    assert all(r() is None for r in dead), "dropping the graph's owner must free the buffers only its graph used"


@pytest.mark.parametrize("tag", ["robo_default", "labelprop"])
def test_fused_head_wiring_on_cpu(tag, cpu_engine):
    """TrainStep's fused classifier head: Plan.forward(stop_before=head) + ops.head_ce_train + Plan.backward(seed=...)
    give the gradients of the full plan fed with the cross-entropy gradient (same stand-in kernels on both sides)."""
    if tag not in _cases():
        pytest.skip(f"no case {tag}")
    engine, fake = cpu_engine
    make, oracle, cin = _cases()[tag]
    torch.manual_seed(12345678)
    m = make().train()
    plan = m._get_plan()
    head = plan.fusable_head()
    assert head == len(plan.nodes) - 1
    x = synth.images(2, cin, 24, 32, seed=5)
    y = synth.labels_learnable(x[:, :3])
    cw = torch.tensor(synth.CLASS_WEIGHTS)
    bufs = {k: v.clone() for k, v in m.state_dict().items()}
    with torch.no_grad():
        outs, saved = plan.forward(x, training=True, save=True)
        lg = outs[0].detach().clone().requires_grad_(True)
        with torch.enable_grad():
            loss = F.cross_entropy(lg, y, weight=cw)
            loss.backward()
        _, gv = plan.backward(saved, [lg.grad], x_needs_grad=False)
        ref = {id(p): gv[id(p)].clone() for p in plan.params}
        m.load_state_dict(bufs)  # the running statistics moved; same starting point for the second pass
        sums = torch.zeros(2, dtype=torch.float64)
        corr = torch.zeros(1, dtype=torch.int64)
        fake.ce_weight_sum(y, cw, sums[1:2], plan.nodes[head].geom.cout)
        outs2, saved2 = plan.forward(x, training=True, save=True, stop_before=head)
        assert outs2 == [None] and len(saved2[0]) == len(plan.nodes)
        nd = plan.nodes[head]
        total = sum(p.numel() for p in plan.params)
        flat = torch.zeros(total)
        views, o = {}, 0
        for p in plan.params:
            views[id(p)] = flat[o:o + p.numel()].view(p.shape)
            o += p.numel()
        dfeat = fake.head_ce_train(saved2[0][nd.src], nd.conv.weight.detach(), nd.conv.bias.detach(), y, cw, sums, corr,
                                   views[id(nd.conv.weight)], views[id(nd.conv.bias)])
        seen = []
        plan.backward(saved2, [None], False, views, node_done=seen.append, seed={nd.src: dfeat})
    assert seen == list(range(len(plan.nodes) - 1, -1, -1))
    assert abs(float(sums[0] / sums[1]) - float(loss)) <= 1e-6 * abs(float(loss))
    assert int(corr) == int((outs[0].argmax(1) == y).sum())
    for p in plan.params:
        a, b = views[id(p)], ref[id(p)]
        assert float((a - b).abs().max()) <= 1e-5 * max(1e-3, float(b.abs().max())), (tag, tuple(p.shape))
