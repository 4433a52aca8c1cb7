"""TrainStep(loss="dice") on the B200: the two-pass Dice head (rcv_head_dice_fwd / rcv_head_dice_train) against float64
autograd, the fused step against the unfused one and against the eager module loop (model(x) -> DiceLoss -> + L1 ->
backward -> torch.optim.Adam), a 50-step loss curve against a float64 oracle loop, and the step's features
(step_async, the single-rank communication schedule, an unfused 3x3 head, library kernels only)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import ref_model as R
from oracle.ref_transforms import dice_loss
from test_gpu_train import _cuda_kernel_names, _foreign
from util import assert_close

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("hw", [(7, 9), (12, 16)])
@pytest.mark.parametrize("classes", [2, 5, 8])
@pytest.mark.parametrize("cin", [8, 16])
def test_head_dice_kernels_match_float64(cin, classes, hw):
    """Pass 1 + pass 2 against float64 autograd over F.conv2d + ref_transforms.dice_loss: non-uniform class weights,
    the last class absent from the batch, an upstream gradient of 0.7; odd H*W (one pixel per thread) and even H*W
    (two).  Gates: sums and loss 1e-6 relative, dfeat / dW / db 2e-6 of their range, the correct count exact."""
    from robocupvision_b200 import ops
    g = torch.Generator().manual_seed(1000 * cin + 10 * classes + hw[0])
    n, (h, w) = 3, hw
    feat = torch.randn(n, cin, h, w, generator=g)
    weight = torch.randn(classes, cin, generator=g) * 0.5
    bias = torch.randn(classes, generator=g) * 0.1
    y = torch.randint(0, classes - 1, (n, h, w), generator=g)  # class classes-1 never occurs
    cw = torch.arange(1, classes + 1, dtype=torch.float32)
    wn = cw / cw.sum().item() * cw.shape[0]
    gscale = 0.7

    f64 = feat.double().requires_grad_(True)
    w64 = weight.double().requires_grad_(True)
    b64 = bias.double().requires_grad_(True)
    z = F.conv2d(f64, w64.view(classes, cin, 1, 1), b64)
    loss_ref = dice_loss(z, y, cw.double())
    (gscale * loss_ref).backward()
    p = torch.softmax(z.detach(), 1)
    oh = F.one_hot(y, classes).permute(0, 3, 1, 2).double()
    sums_ref = torch.cat([(p * oh).sum((0, 2, 3)), (p + oh).sum((0, 2, 3))])
    corr_ref = int((z.detach().argmax(1) == y).sum())

    dev = torch.device("cuda")
    fd, wd, bd, yd = feat.to(dev), weight.to(dev), bias.to(dev), y.to(dev)
    sums = torch.zeros(2 * classes, dtype=torch.float64, device=dev)
    corr = torch.zeros(1, dtype=torch.int64, device=dev)
    cell = torch.zeros(2, dtype=torch.float64, device=dev)
    dw = torch.zeros(classes, cin, device=dev)
    db = torch.zeros(classes, device=dev)
    ops.head_dice_fwd(fd, wd, bd, yd, sums, corr)
    dfeat = ops.head_dice_train(fd, wd, bd, yd, wn.to(dev), sums, 1e-7, cell, dw, db,
                                gscale=torch.tensor([gscale], device=dev))
    torch.cuda.synchronize()

    def rel(a, b):
        return float((a.cpu().double() - b).abs().max()) / float(b.abs().max())

    assert rel(sums, sums_ref) <= 1e-6, (sums.cpu(), sums_ref)
    assert abs(float(cell[0]) - float(loss_ref)) <= 1e-6 * abs(float(loss_ref)) and float(cell[1]) == 1.0
    assert int(corr) == corr_ref
    assert rel(dfeat, f64.grad) <= 2e-6, rel(dfeat, f64.grad)
    assert rel(dw, w64.grad) <= 2e-6, rel(dw, w64.grad)
    assert rel(db, b64.grad) <= 2e-6, rel(db, b64.grad)


def _make(net, eps=1e-3, **kw):
    """Adam eps 1e-3 by default: with 1e-8 the sign of rounding noise decides where a zero gradient moves a weight
    (test_step_async_matches_step)."""
    from robocupvision_b200.model import LabelProp, ROBO_UNet
    from robocupvision_b200.train import TrainStep
    torch.manual_seed(12345678)
    m = {"robo": lambda: ROBO_UNet(), "v2": lambda: ROBO_UNet(v2=True, classSize=3), "labelprop": lambda: LabelProp(5, 32, 0)}[net]()
    m = m.cuda()
    cw = synth.LP_CLASS_WEIGHTS if net == "labelprop" else synth.CLASS_WEIGHTS
    return m, TrainStep(m, cw, lr=1e-3, l1_decay=1e-6, eps=eps, use_graph=True, loss="dice", **kw)


def _batch(net, s):
    cin = 8 if net == "labelprop" else 3
    x = synth.images(4, cin, 48, 64, seed=300 + s)
    return x, synth.labels_learnable(x[:, :3])


def _same_weights(ma, mb, tol=2e-4):
    for (k, a), (_, b) in zip(ma.state_dict().items(), mb.state_dict().items()):
        if a.is_floating_point():
            assert_close(k, a, b, tol)
        else:
            assert torch.equal(a, b), k


@pytest.mark.parametrize("net", ["robo", "labelprop"])
def test_dice_fused_head_matches_separate_kernels(net):
    """Five graph-replayed Dice steps with the two-pass head against conv forward -> dice_fwd -> dice_bwd -> conv dgrad
    / wgrad: losses, correct counts and weights (gates of test_fused_head_matches_separate_kernels), and fewer
    kernels per step."""
    (ma, ta), (mb, tb) = _make(net, fused_head=True), _make(net, fused_head=False)
    assert ta._head == len(ta.plan.nodes) - 1 and tb._head == -1
    for s in range(5):
        x, y = (t.cuda() for t in _batch(net, s))
        got = []
        for ts in (ta, tb):
            ts.step(x, y)
            got.append((ts.loss_value(), int(ts.correct)))
        assert abs(got[0][0] - got[1][0]) <= 3e-5 * abs(got[1][0]) and abs(got[0][1] - got[1][1]) <= 8, (s, got)
    assert ta.kernels_per_step < tb.kernels_per_step, (ta.kernels_per_step, tb.kernels_per_step)
    _same_weights(ma, mb)


@pytest.mark.parametrize("net", ["robo", "v2"])
def test_dice_step_matches_eager_loop(net):
    """TrainStep(loss="dice") (fused head for ROBO_UNet, the unfused 3x3 head of ROBO_UNet(v2=True, classSize=3)) against the eager module loop
    on a twin model: model(x) -> DiceLoss -> + l1_decay * sum|p| -> backward -> torch.optim.Adam, five steps."""
    from robocupvision_b200.model import DiceLoss
    m, ts = _make(net)
    assert (ts._head >= 0) == (net == "robo")
    torch.manual_seed(12345678)
    twin = type(m)(v2=True, classSize=3).cuda() if net == "v2" else type(m)().cuda()
    twin.load_state_dict(m.state_dict())
    twin.train()
    crit = DiceLoss(synth.CLASS_WEIGHTS)
    opt = torch.optim.Adam(twin.parameters(), lr=1e-3, eps=1e-3)
    for s in range(5):
        x, y = (t.cuda() for t in _batch(net, s))
        ts.step(x, y)
        opt.zero_grad()
        out = twin(x)
        loss = crit(out, y) + 1e-6 * sum(p.abs().sum() for p in twin.parameters())
        loss.backward()
        opt.step()
        want, got = float(loss), ts.loss_value()
        assert abs(got - want) <= 3e-5 * abs(want), (s, got, want)
        assert abs(int(ts.correct) - int((out.detach().argmax(1) == y).sum())) <= 8
    _same_weights(m, twin)


def test_dice_loss_curve_against_float64_oracle():
    """50 graph-replayed Dice steps (ROBO_UNet, 4x3x48x64, learnable labels, seed 12345678, Adam 1e-3, L1 1e-6)
    against a float64 oracle loop (ref_model forward + dice_loss + L1 + torch.optim.Adam).  Gates: step 1 <= 1e-5
    relative, every step <= 2e-2, the mean of the last ten within 2 %; the loss falls."""
    m, ts = _make("robo", eps=1e-8)  # torch.optim.Adam's default, as the oracle loop uses it
    sd = R.leaf_state_dict({k: (v.detach().cpu().double() if v.is_floating_point() else v.detach().cpu().clone())
                            for k, v in m.state_dict().items()})
    params = [sd[k] for k in R.param_keys(sd)]
    opt = torch.optim.Adam(params, lr=1e-3)
    cw = torch.tensor(synth.CLASS_WEIGHTS, dtype=torch.float64)
    got, ref = [], []
    for s in range(50):
        x = synth.images(4, 3, 48, 64, seed=5000 + s)
        y = synth.labels_learnable(x)
        ts.step(x.cuda(), y.cuda())
        got.append(ts.loss_value())
        opt.zero_grad()
        loss = dice_loss(R.robo_unet_forward(sd, x.double(), training=True), y, cw) + 1e-6 * R.l1reg(params)
        loss.backward()
        opt.step()
        ref.append(float(loss.detach()))
    got, ref = np.array(got), np.array(ref)
    rel = np.abs(got - ref) / np.abs(ref)
    print(f"dice curve: step-1 rel {rel[0]:.2e}, max rel {rel.max():.2e} at step {int(rel.argmax())}, "
          f"final {got[-10:].mean():.5f} vs oracle {ref[-10:].mean():.5f}")
    assert rel[0] <= 1e-5, (got[0], ref[0])
    assert rel.max() <= 2e-2, (int(rel.argmax()), got[rel.argmax()], ref[rel.argmax()])
    assert abs(got[-10:].mean() - ref[-10:].mean()) <= 2e-2 * ref[-10:].mean()
    assert got[-10:].mean() < got[0], "the Dice loss must fall"


def test_dice_step_features():
    """step_async returns what step returns; the single-rank force_comm_path schedule matches the plain step; the
    unfused --v2 head trains; a profiled replay of a fused and of an unfused Dice step launches library kernels only."""
    (ma, ta), (mb, tb) = _make("robo"), _make("robo")
    batches = [_batch("robo", s) for s in range(5)]
    want = []
    for x, y in batches:
        ta.step(x.cuda(), y.cuda())
        want.append((ta.loss_value(), int(ta.correct)))
    got, prev = [], None
    for x, y in batches:
        h = tb.step_async(x.pin_memory(), y.pin_memory())
        if prev is not None:
            got.append(prev.wait())
        prev = h
    got.append(prev.wait())
    for (l0, c0), (dice, tot, c1) in zip(want, got):
        assert abs(l0 - tot) <= 3e-5 * abs(l0) and abs(c0 - c1) <= 8, (l0, tot, c0, c1)
        assert 0.0 < dice < 1.0
    _same_weights(ma, mb)
    assert ta.dice_sums.shape == (10,) and float(ta.dice_sums[5:].sum()) > 0

    (mc, tc), (md, td) = _make("robo", overlap_comm=False), _make("robo", force_comm_path=True)
    assert tc.comm_stream is None and td.comm_stream is not None
    for x, y in batches:
        for ts in (tc, td):
            ts.step(x.cuda(), y.cuda())
        assert abs(tc.loss_value() - td.loss_value()) <= 3e-5 * abs(tc.loss_value())
    _same_weights(mc, md)

    mv, tv = _make("v2")
    assert tv._head == -1
    losses = []
    for s in range(20):
        x, y = (t.cuda() for t in _batch("v2", s % 4))
        tv.step(x, y)
        losses.append(tv.loss_value())
    assert all(np.isfinite(losses)) and np.mean(losses[-4:]) < np.mean(losses[:4]), losses

    for ts in (ta, tv):
        x, y = (t.cuda() for t in _batch("robo", 0))
        names = _cuda_kernel_names(lambda: ts.step(x, y))
        assert len(names) >= 20, names
        assert not _foreign(names), _foreign(names)
    assert any("head_dice_fwd" in n for n in _cuda_kernel_names(lambda: ta.step(x, y)))
