"""Fixed-order (_det) reductions on the GPU: three runs on the same inputs give bitwise the same sums, the sums stay
within the plain forms' tolerances of a float64 reference, and the element-wise outputs are those of the plain forms.
The loss modules take the fixed-order forms under torch.use_deterministic_algorithms(True)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

RUNS = 3


def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-300)


@pytest.fixture
def deterministic_algorithms():
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=warn)


def _ce_case(n, c, h, w, seed):
    gen = torch.Generator().manual_seed(seed)
    z = torch.randn(n, c, h, w, generator=gen) * 3
    y = torch.randint(0, c, (n, h, w), generator=gen)
    cw = torch.rand(c, generator=gen) * 2 + 0.1  # non-integer class weights: the atomic weight sum is not exact
    return z, y, cw


def _ce_ref(z, y, cw):
    z, cw = z.double(), cw.double()
    nll = torch.logsumexp(z, 1) - z.gather(1, y.unsqueeze(1)).squeeze(1)
    wy = cw[y]
    return float((wy * nll).sum()), float(wy.sum())


@pytest.mark.parametrize("n,c,h,w", [(64, 5, 120, 160), (8, 5, 480, 640), (2, 3, 7, 9), (1, 8, 256, 300)])
def test_ce_fwd_det_repeatable_and_accurate(n, c, h, w):
    from robocupvision_b200 import ops
    z, y, cw = _ce_case(n, c, h, w, seed=n * 31 + c)
    zc, yc, cwc = z.cuda(), y.cuda(), cw.cuda()
    scratch = ops.det_scratch(ops.DET_CE_FWD, n, c, h * w, "cuda")
    outs = []
    for _ in range(RUNS):  # one scratch for every run: the kernels leave it ready for the next call
        sums, am, conf, corr = ops.ce_fwd(zc, yc, cwc, want_argmax=True, want_conf=True, want_correct=True,
                                          scratch=scratch)
        outs.append((sums.clone(), am, conf, corr))
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            assert torch.equal(a, b)
    lref, wref = _ce_ref(z, y, cw)
    s = outs[0][0].cpu()
    assert _rel(s[0], lref) <= 1e-6 and _rel(s[1], wref) <= 1e-12, (s, lref, wref)
    plain = ops.ce_fwd(zc, yc, cwc, want_argmax=True, want_conf=True, want_correct=True)
    assert _rel(plain[0][0], s[0]) <= 1e-9 and _rel(plain[0][1], s[1]) <= 1e-12
    for a, b in zip(plain[1:], outs[0][1:]):
        assert torch.equal(a, b)  # argmax, confusion, correct: integer results, unchanged
    assert int(torch.count_nonzero(scratch[:128])) == 0  # counter reset


def test_ce_fwd_det_accumulates_like_plain():
    """dst += sum: a caller-zeroed accumulator summed into twice holds twice the sums, as with the atomic form."""
    from robocupvision_b200 import ops
    z, y, cw = _ce_case(4, 5, 60, 80, seed=7)
    zc, yc, cwc = z.cuda(), y.cuda(), cw.cuda()
    scratch = ops.det_scratch(ops.DET_CE_FWD, 4, 5, 60 * 80, "cuda")
    once = ops.ce_fwd(zc, yc, cwc, scratch=scratch)[0].clone()
    acc = ops.zeros(2, torch.float64, "cuda")
    ops.ce_fwd(zc, yc, cwc, sums=acc, scratch=scratch)
    ops.ce_fwd(zc, yc, cwc, sums=acc, scratch=scratch)
    assert torch.equal(acc, once + once)


@pytest.mark.parametrize("count", [64 * 120 * 160, 5, 2048 * 600 + 3])
def test_ce_weight_sum_det_non_integer_weights(count):
    from robocupvision_b200 import ops
    gen = torch.Generator().manual_seed(count % 1000)
    y = torch.randint(-1, 5, (count,), generator=gen)  # -1: ignored label
    cw = torch.tensor([0.3, 1.7, 2.9, 0.11, 5.3])
    yc, cwc = y.cuda(), cw.cuda()
    scratch = ops.det_scratch(ops.DET_CE_WEIGHT_SUM, 1, 5, count, "cuda")
    got = []
    for _ in range(RUNS):
        out = ops.zeros(1, torch.float64, "cuda")
        ops.ce_weight_sum(yc, cwc, out, 5, scratch=scratch)
        got.append(out)
    assert all(torch.equal(got[0], g) for g in got[1:])
    valid = y >= 0
    ref = float(cw.double()[y[valid]].sum())
    assert _rel(got[0], ref) <= 1e-12


@pytest.mark.parametrize("n,c,h,w", [(64, 5, 120, 160), (3, 2, 17, 23), (8, 8, 240, 320)])
def test_dice_fwd_det_repeatable_and_accurate(n, c, h, w):
    from robocupvision_b200 import ops
    gen = torch.Generator().manual_seed(n + c)
    z = torch.randn(n, c, h, w, generator=gen) * 2
    y = torch.randint(0, c, (n, h, w), generator=gen)
    zc, yc = z.cuda(), y.cuda()
    scratch = ops.det_scratch(ops.DET_DICE_FWD, n, c, h * w, "cuda")
    got = [ops.dice_fwd(zc, yc, scratch=scratch) for _ in range(RUNS)]
    assert all(torch.equal(got[0], g) for g in got[1:])
    s = torch.softmax(z.double(), 1)
    oh = torch.nn.functional.one_hot(y, c).permute(0, 3, 1, 2).double()
    ref = torch.cat([(s * oh).sum((0, 2, 3)), (s + oh).sum((0, 2, 3))])
    assert float(((got[0].cpu() - ref).abs() / ref.abs()).max()) <= 1e-5
    plain = ops.dice_fwd(zc, yc)
    assert float(((plain - got[0]).abs() / got[0].abs()).max()) <= 1e-9


@pytest.mark.parametrize("n", [10007, 3_000_000])
@pytest.mark.parametrize("opt", ["adam", "sgd"])
def test_optimizer_l1_sum_det(opt, n):
    """The L1 sum in fixed order; the parameter update itself is element-wise and bitwise that of the plain form."""
    from robocupvision_b200 import ops
    gen = torch.Generator().manual_seed(n)
    p0 = torch.randn(n, generator=gen)
    mask = (torch.rand(n, generator=gen) < 0.2).to(torch.uint8).cuda()
    grads = [torch.randn(n, generator=gen).cuda() for _ in range(3)]
    scratch = ops.det_scratch(ops.DET_L1_SUM, 1, 1, n, "cuda")

    def run(det):
        p, m, v = p0.cuda(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
        sums = []
        for step, g in enumerate(grads, 1):
            l1 = ops.zeros(1, torch.float64, "cuda")
            kw = dict(scratch=scratch) if det else {}
            if opt == "adam":
                ops.adam_l1_step(p, g, m, v, lr=1e-3, step=step, l1_decay=1e-4, mask=mask, l1_sum=l1, **kw)
            else:
                ops.sgd_step(p, g, m, lr=1e-2, momentum=0.9, weight_decay=1e-4, mask=mask, first_step=step == 1,
                             l1_decay=1e-4, l1_sum=l1, **kw)
            sums.append(l1)
        return p, m, v, sums

    runs = [run(True) for _ in range(RUNS)]
    for r in runs[1:]:
        for a, b in zip(runs[0][:3], r[:3]):
            assert torch.equal(a, b)
        assert all(torch.equal(a, b) for a, b in zip(runs[0][3], r[3]))
    plain = run(False)
    for a, b in zip(plain[:3], runs[0][:3]):
        assert torch.equal(a, b)
    for a, b in zip(plain[3], runs[0][3]):
        assert _rel(a, b) <= 1e-9
    ref = float(p0.double().abs().sum())  # sum |p| before the first update
    assert _rel(runs[0][3][0], ref) <= 1e-5


def test_loss_modules_bitwise_under_deterministic_algorithms(deterministic_algorithms):
    """CrossEntropyLoss2d and DiceLoss, forward and backward, repeated on the same logits: bitwise the same loss and
    gradient, and the same values as with the mode off to summation order."""
    from robocupvision_b200.model import CrossEntropyLoss2d, DiceLoss
    z, y, cw = _ce_case(16, 5, 120, 160, seed=11)
    zc, yc = z.cuda(), y.cuda()
    for loss_fn in (CrossEntropyLoss2d(cw), DiceLoss(cw)):
        got = []
        for _ in range(RUNS):
            zi = zc.clone().requires_grad_(True)
            loss = loss_fn(zi, yc)
            (loss * 1.5).backward()
            got.append((loss.detach(), zi.grad))
        for a in got[1:]:
            assert torch.equal(a[0], got[0][0]) and torch.equal(a[1], got[0][1]), type(loss_fn).__name__
        torch.use_deterministic_algorithms(False)
        zi = zc.clone().requires_grad_(True)
        loss = loss_fn(zi, yc)
        (loss * 1.5).backward()
        torch.use_deterministic_algorithms(True)
        assert _rel(loss, got[0][0]) <= 1e-6
        assert float((zi.grad - got[0][1]).abs().max()) <= 1e-6 * float(got[0][1].abs().max())


def test_train_mode_model_refuses_under_deterministic_algorithms(deterministic_algorithms):
    """model(x) in train mode sums BatchNorm statistics, and its backward the weight gradients, with atomics: under
    torch.use_deterministic_algorithms(True) it raises a RuntimeError naming them, under warn_only=True it warns and
    runs.  Eval mode has no such sums and runs, bitwise repeatable."""
    from robocupvision_b200.model import ROBO_UNet
    torch.manual_seed(12345678)
    m = ROBO_UNet().cuda()
    x = torch.randn(2, 3, 48, 64, device="cuda")
    m.train()
    with pytest.raises(RuntimeError, match="BatchNorm batch statistics.*does not have a deterministic implementation"):
        m(x)
    torch.use_deterministic_algorithms(True, warn_only=True)
    with pytest.warns(UserWarning, match="does not have a deterministic implementation"):
        out = m(x)
    out.sum().backward()
    torch.use_deterministic_algorithms(True)
    m.eval()
    with torch.no_grad():
        a, b = m(x), m(x)
    assert torch.equal(a, b)
