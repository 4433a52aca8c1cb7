"""TrainStep(loss="dice") without a GPU: argument validation of the two-pass Dice head (rcv_head_dice_fwd /
rcv_head_dice_train) and of rcv_dice_loss, the refusal of an unknown loss, and the fused-Dice wiring through the real
Plan.forward(stop_before) / Plan.backward(seed) with ATen stand-ins of the two head passes, against autograd over the
oracle forward and the oracle's dice_loss."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import ref_model as R
from oracle.ref_transforms import dice_loss
from test_plan_host import _cases


def test_head_dice_validation_without_gpu():
    from robocupvision_b200 import _lib
    lib = _lib.load()
    BAD, UNS = _lib.RCV_ERR_BAD_ARG, _lib.RCV_ERR_UNSUPPORTED
    p = C.c_void_p(16)  # never dereferenced: every case below is refused before a launch
    assert lib.rcv_head_dice_fwd(4, 8, 5, 100, None, p, None, p, p, None, None) == BAD
    assert lib.rcv_head_dice_fwd(4, 8, 5, 100, p, p, None, p, None, None, None) == BAD
    assert lib.rcv_head_dice_fwd(0, 8, 5, 100, p, p, None, p, p, None, None) == BAD
    assert lib.rcv_head_dice_fwd(4, 8, 9, 100, p, p, None, p, p, None, None) == UNS
    assert b"9 classes over 8 channels" in lib.rcv_last_error()
    assert lib.rcv_head_dice_fwd(4, 32, 5, 100, p, p, None, p, p, None, None) == UNS
    args = lambda n, cin, c, feat, sums, dfeat, dw: (n, cin, c, 100, feat, p, None, p, None, sums, 1e-7, None, None,  # noqa: E731
                                                     dfeat, dw, None, None)
    assert lib.rcv_head_dice_train(*args(4, 8, 5, None, p, p, p)) == BAD
    assert lib.rcv_head_dice_train(*args(4, 8, 5, p, None, p, p)) == BAD
    assert lib.rcv_head_dice_train(*args(4, 8, 5, p, p, None, p)) == BAD
    assert lib.rcv_head_dice_train(*args(4, 8, 5, p, p, p, None)) == BAD
    assert lib.rcv_head_dice_train(*args(4, 8, 9, p, p, p, p)) == UNS
    assert b"9 classes over 8 channels" in lib.rcv_last_error()
    assert lib.rcv_head_dice_train(*args(4, 32, 5, p, p, p, p)) == UNS
    assert b"5 classes over 32 channels" in lib.rcv_last_error()
    assert lib.rcv_dice_loss(5, None, None, 1e-7, p, None) == BAD
    assert lib.rcv_dice_loss(5, p, None, 1e-7, None, None) == BAD
    assert lib.rcv_dice_loss(9, p, None, 1e-7, p, None) == UNS


def test_train_step_refuses_unknown_loss():
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import TrainStep
    with pytest.raises(ValueError, match="loss"):
        TrainStep(ROBO_UNet(), loss="bogus")


# ---- ATen stand-ins of the two head passes: the kernels' arithmetic, written out
def _head_logits(feat, weight, bias, target):
    c = weight.shape[0]
    z = F.conv2d(feat, weight.view(c, -1, 1, 1), bias)
    ok = ((target >= 0) & (target < c)).unsqueeze(1).to(z.dtype)
    oh = F.one_hot(target.clamp(0, c - 1), c).permute(0, 3, 1, 2).to(z.dtype) * ok
    return z, torch.softmax(z, 1), oh, ok


def fake_head_dice_fwd(feat, weight, bias, target, sums, corr):
    c = weight.shape[0]
    z, p, oh, ok = _head_logits(feat, weight, bias, target)
    sums[:c] += (p * oh).sum((0, 2, 3)).double()
    sums[c:] += ((p + oh) * ok).sum((0, 2, 3)).double()
    corr += (z.argmax(1) == target).sum()


def fake_head_dice_train(feat, weight, bias, target, weights, sums, eps, loss, dweight, dbias):
    c = weight.shape[0]
    _, p, oh, ok = _head_logits(feat, weight, bias, target)
    w = weights.double()
    inter, card = sums[:c], sums[c:] + float(torch.tensor(eps, dtype=torch.float32))
    a = (-2.0 * w / (c * card)).float().view(1, c, 1, 1)
    b = (2.0 * w * inter / (c * card * card)).float().view(1, c, 1, 1)
    g = b + a * oh
    dz = p * (g - (p * g).sum(1, keepdim=True)) * ok
    loss[0] = 1.0 - (2.0 * w * inter / card).mean()
    loss[1] = 1.0
    dweight += torch.einsum("nchw,nkhw->ck", dz, feat).reshape(dweight.shape)
    if dbias is not None:
        dbias += dz.sum((0, 2, 3))
    return torch.einsum("nchw,ck->nkhw", dz, weight.reshape(c, -1))


@pytest.fixture
def cpu_engine(monkeypatch):
    """engine.Plan with its kernels replaced by ATen-CPU stand-ins (tests/fake_ops.py); single stream."""
    import fake_ops
    from robocupvision_b200 import engine
    monkeypatch.setattr(engine, "ops", fake_ops)
    monkeypatch.setattr(engine, "WGRAD_SIDE_STREAM", False)
    fake_ops.calls.clear()
    return engine, fake_ops


@pytest.mark.parametrize("tag", ["robo_default", "labelprop"])
def test_fused_dice_head_wiring_on_cpu(tag, cpu_engine):
    """TrainStep(loss="dice")'s fused head: Plan.forward(stop_before=head) -> pass 1 (sums, correct count) -> pass 2
    (loss cell, dfeat, head weight gradients) -> Plan.backward(seed={src: dfeat}) give the Dice loss, every parameter
    gradient and the running statistics of autograd over the oracle forward + oracle dice_loss."""
    make, oracle, cin = _cases()[tag]
    torch.manual_seed(12345678)
    m = make().train()
    plan = m._get_plan()
    head = plan.fusable_head()
    assert head == len(plan.nodes) - 1
    x = synth.images(2, cin, 24, 32, seed=5)
    y = synth.labels_learnable(x[:, :3])
    cw = torch.tensor(synth.CLASS_WEIGHTS if tag == "robo_default" else synth.LP_CLASS_WEIGHTS)
    wn = cw / cw.sum().item() * cw.shape[0]  # DiceLoss.__init__, as TrainStep normalises them
    sd = {k: v.clone() for k, v in m.state_dict().items()}

    def oracle_run(dtype):
        osd = R.leaf_state_dict({k: (v.clone().to(dtype) if v.is_floating_point() else v.clone()) for k, v in sd.items()})
        logits = oracle(osd, x.to(dtype), training=True)
        loss = dice_loss(logits, y, cw.to(dtype))
        loss.backward()
        return float(loss.detach()), logits.detach(), osd

    loss32, logits32, osd32 = oracle_run(torch.float32)
    loss64, _, osd64 = oracle_run(torch.float64)
    with torch.no_grad():
        nd = plan.nodes[head]
        total = sum(p.numel() for p in plan.params)
        flat = torch.zeros(total)
        views, o = {}, 0
        for p in plan.params:
            views[id(p)] = flat[o:o + p.numel()].view(p.shape)
            o += p.numel()
        sums = torch.zeros(2 * nd.geom.cout, dtype=torch.float64)
        cell = torch.zeros(2, dtype=torch.float64)
        corr = torch.zeros(1, dtype=torch.int64)
        outs, saved = plan.forward(x, training=True, save=True, stop_before=head)
        assert outs == [None] and saved[2].get(nd.src) is None
        feat = saved[0][nd.src]
        fake_head_dice_fwd(feat, nd.conv.weight, nd.conv.bias, y, sums, corr)
        dfeat = fake_head_dice_train(feat, nd.conv.weight, nd.conv.bias, y, wn, sums, 1e-7, cell,
                                     views[id(nd.conv.weight)], views[id(nd.conv.bias)])
        seen = []
        plan.backward(saved, [None], False, views, node_done=seen.append, seed={nd.src: dfeat})
    assert seen == list(range(len(plan.nodes) - 1, -1, -1))
    assert float(cell[1]) == 1.0
    assert abs(float(cell[0]) - loss64) <= 1e-5 * abs(loss64), (float(cell[0]), loss64)
    assert int(corr) == int((logits32.argmax(1) == y).sum())
    gmax = max(float(v.grad.abs().max()) for v in osd64.values() if v.grad is not None)

    def rel_l2(a, b):
        return float((a.double() - b).norm()) / max(float(b.norm()), 1e-3 * gmax * b.numel() ** 0.5)

    from robocupvision_b200.model import upSampleTransposeConv
    noise = {f"{n}.conv.bias" for n, mod in m.named_modules() if isinstance(mod, upSampleTransposeConv)}
    names = {id(p): k for k, p in m.named_parameters()}
    for p in plan.params:
        k = names[id(p)]
        if k in noise:
            continue
        g64 = osd64[k].grad
        err, floor = rel_l2(views[id(p)], g64), rel_l2(osd32[k].grad, g64)
        assert err <= max(1e-3, 4 * floor), f"{tag}: grad {k} rel L2 err {err:.3e} (fp32 oracle {floor:.3e})"
    for k, b in m.named_buffers():
        if b.is_floating_point():
            assert torch.allclose(b, osd32[k], rtol=1e-5, atol=1e-6), (tag, k)
        else:
            assert int(b) == int(osd32[k]), (tag, k)
