"""CUDA graphs replayed after the same model ran at another batch size, the way a training loop trains at one batch
size and validates with another.

The plan replaces its conv workspace when a size needs more scratch, and its weight panels and pack tables when a
size needs another layout, while a graph captured earlier has the old addresses baked into its nodes.  Each scenario
therefore checks, before every replay, that every buffer the plan held at capture is still alive and referenced by
the graph's owner (TrainStep / EvalStep): a replay over freed memory is a device use-after-free, so the check comes
first.  Each scenario also asserts its premise (the second size needs a larger workspace, or a buffer was replaced),
so that a dispatch change that stops the growth fails loudly instead of leaving a test that tests nothing.  Results
are compared with the float64 oracle and with eager twins."""
import weakref

import pytest
import torch

import synth
from nets import pb_fcn_state, robo_state
from oracle import ref_model as R
from util import LOGIT_TOL, assert_close, check_eval_outputs, tensors_held_by

pytestmark = pytest.mark.gpu
CW = synth.CLASS_WEIGHTS


def _f64(sd):
    return {k: (v.detach().cpu().double() if v.is_floating_point() else v.detach().cpu()) for k, v in sd.items()}


def _assert_workspace_grows(plan, first, second):
    """Premise: Plan.workspace needs more at input size `second` (N, H, W) than at `first` (the same loop over the
    plan's tensor-core layers and both directions)."""
    from robocupvision_b200 import ops

    def need(n, h, w):
        out = 0
        for nd, (nn_, hh, ww) in zip(plan.nodes, plan._in_sizes(n, h, w)):
            if nd.kind == "conv":
                for d in (ops.PACK_FWD, ops.PACK_DGRAD):
                    if nd.uses_tc(d, plan.math):
                        out = max(out, ops.conv_workspace_bytes(nd.geom, nn_, hh, ww, d, plan.math))
        return out

    a, b = need(*first), need(*second)
    print(f"workspace need: {first} {a / 1e6:.2f} MB -> {second} {b / 1e6:.2f} MB")
    assert b > a, f"premise: the workspace need at {second} ({b} B) must exceed the one at {first} ({a} B)"


def _baked(plan):
    """The buffers a graph captured now can bake in, read off the plan's own fields (not Plan.capture_refs):
    [(label, weakref, address, bytes)]."""
    bufs = [("conv workspace", plan._workspace)]
    bufs += [(f"node {t} panel {d}", b) for t, nd in enumerate(plan.nodes) for d, b in enumerate(nd._pack)]
    bufs += [(f"pack table {k}", tbl.table) for k, tbl in plan._pack_tables.items()]
    return [(lbl, weakref.ref(t), t.data_ptr(), t.nbytes) for lbl, t in bufs if t is not None]


def _assert_held(owner, baked, what):
    """Before a replay: every buffer recorded at capture is still a live tensor, at the same address, that the graph's
    owner references."""
    held = tensors_held_by(owner)
    lost = [f"{lbl} ({nb} B at {ptr:#x})" for lbl, ref, ptr, nb in baked
            if ref() is None or id(ref()) not in held or ref().data_ptr() != ptr]
    assert not lost, f"{what}: its graph bakes in buffers its owner no longer holds: {lost}"


def _assert_replaced(plan, baked):
    """Premise: the plan no longer holds at least one of the buffers an earlier capture recorded."""
    held = tensors_held_by(plan)
    gone = [lbl for lbl, ref, _, _ in baked if ref() is None or id(ref()) not in held]
    print(f"replaced since the capture: {gone}")
    assert gone, "premise: the second size replaced none of the plan's buffers"


@pytest.mark.parametrize("math", ["parity", "bf16", "tf32"])
def test_eval_graphs_at_two_batch_sizes(math):
    """EvalStep(use_graph=True) on ROBO_UNet 48x64 at batch 4, then 8, then 4 again, for three rounds: each later call
    replays the graph of its size.  Parity math: the split workspace grows from batch 4 to 8.  The fast modes have no
    split workspace; there the pack table is rebuilt for each size.  Every output equals an eager EvalStep's bit for
    bit; in parity math the logits are also checked against the float64 oracle."""
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import EvalStep
    sd, _, _ = robo_state("robo_default")
    m = ROBO_UNet()
    m.load_state_dict(sd)
    m.cuda().eval().set_math(math)
    plan = m._get_plan()
    if math == "parity":
        _assert_workspace_grows(plan, (4, 48, 64), (8, 48, 64))
    sd64 = _f64(sd)
    graph, eager = EvalStep(m, CW, use_graph=True), EvalStep(m, CW)
    baked, worst = {}, 0.0
    for rnd in range(3):
        for n in (4, 8):
            x = synth.images(n, 3, 48, 64, seed=700 + 10 * rnd + n)
            y = synth.labels_random(n, 48, 64, seed=800 + 10 * rnd + n)
            key = ((n, 3, 48, 64), (n, 48, 64))
            if rnd > 0:
                _assert_held(graph, baked[n], f"eval graph at batch {n}")
                g0 = graph._graphs[key]["graph"]
            got = graph(x.cuda(), y.cuda())
            if rnd == 0:
                baked[n] = _baked(plan)
                if n == 8:
                    _assert_replaced(plan, baked[4])
            else:
                assert graph._graphs[key]["graph"] is g0, "the call captured again instead of replaying"
            want = eager(x.cuda(), y.cuda())
            for k in ("logits", "argmax", "conf", "correct", "loss"):
                assert torch.equal(got[k], want[k]), f"{math} round {rnd} batch {n}: graph {k} != eager {k}"
            if math == "parity":
                with torch.no_grad():
                    ref = R.robo_unet_forward(sd64, x.double())
                worst = max(worst, assert_close(f"round {rnd} batch {n} logits", got["logits"], ref, LOGIT_TOL))
    if math == "parity":
        print(f"eval graphs at batch 4 / 8: worst logit error against the float64 oracle {worst:.2e}")


@pytest.mark.parametrize("train_n,eval_n,h,w", [(4, 8, 48, 64), (64, 16, 120, 160)], ids=["48x64", "120x160"])
def test_train_graph_replays_after_a_larger_eval(train_n, eval_n, h, w):
    """TrainStep(use_graph=True) on ROBO_UNet, with an eval-mode EvalStep at a batch size whose workspace need is
    larger after every step, then the next training replay (120x160: the benchmarked training batch 64 and a
    validation batch of 16).  An eager TrainStep on a twin model runs the same sequence: losses, correct counts and
    final weights agree to the tolerances of test_step_async_matches_step (Adam eps = 1e-3, see there why).  Every
    eval's logits are checked against the float64 oracle on the weights the step just wrote."""
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import EvalStep, TrainStep
    models, steps = [], []
    for use_graph in (True, False):
        torch.manual_seed(12345678)
        m = ROBO_UNet().cuda()
        models.append(m)
        steps.append(TrainStep(m, CW, lr=1e-3, l1_decay=1e-6, eps=1e-3, use_graph=use_graph))
    plan = models[0]._get_plan()
    _assert_workspace_grows(plan, (train_n, h, w), (eval_n, h, w))
    evals = [EvalStep(m, CW) for m in models]
    baked, worst = None, 0.0
    for s in range(3):
        x = synth.images(train_n, 3, h, w, seed=900 + s)
        y = synth.labels_learnable(x)
        if s > 0:
            _assert_held(steps[0], baked, f"training graph at batch {train_n}, step {s}")
            g0 = steps[0].graph
        got = []
        for ts in steps:
            ts.step(x.cuda(), y.cuda())
            got.append((ts.loss_value(), int(ts.correct)))
        if s == 0:
            baked = _baked(plan)
        else:
            assert steps[0].graph is g0, "the step captured again instead of replaying"
        assert abs(got[0][0] - got[1][0]) <= 3e-5 * abs(got[1][0]) and abs(got[0][1] - got[1][1]) <= 8, (s, got)
        xe = synth.images(eval_n, 3, h, w, seed=950 + s).cuda()
        ye = synth.labels_random(eval_n, h, w, seed=960 + s).cuda()
        out = evals[0](xe, ye)
        evals[1](xe, ye)
        if s == 0:
            _assert_replaced(plan, baked)
        with torch.no_grad():
            ref = R.robo_unet_forward(_f64(models[0].state_dict()), xe.cpu().double())
        worst = max(worst, assert_close(f"eval after step {s}", out["logits"], ref, LOGIT_TOL))
    for (k, a), (_, b) in zip(models[0].state_dict().items(), models[1].state_dict().items()):
        if a.is_floating_point():
            assert_close(k, a, b, 2e-4)
        else:
            assert torch.equal(a, b), k
    print(f"train {train_n} / eval {eval_n} x {h}x{w}: eval logits vs float64 oracle, worst {worst:.2e}")


def test_pb_fcn_pruned_checkpoint_eval_graphs_at_256_and_64():
    """BASELINE configs[2] (PB_FCN from pth/bestModelSegFinetunedPruned.pth) at its benchmarked batch 256 x 3 x 120 x
    160 -- multi-wave grids and their own split plan -- through EvalStep(use_graph=True) at 256, then 64 (the workspace
    grows), then 256 again, replayed.  No reference-produced golden exists at this size; the float64 oracle, which
    reproduces the reference classes bit for bit, is the reference: the gates of _check_eval (util.check_eval_outputs)
    with the oracle's label map and weighted cross entropy."""
    from robocupvision_b200.model import PB_FCN, load_legacy_state_dict
    from robocupvision_b200.train import EvalStep
    osd, raw = pb_fcn_state("bestModelSegFinetunedPruned")
    m = PB_FCN(32, 5, 1, False, 0)
    load_legacy_state_dict(m, raw)
    m.cuda().eval()
    plan = m._get_plan()
    _assert_workspace_grows(plan, (256, 120, 160), (64, 120, 160))
    sd64 = _f64(osd)
    cw64 = torch.tensor(CW, dtype=torch.float64)
    ev = EvalStep(m, CW, use_graph=True)
    baked = {}
    for i, n in enumerate((256, 64, 256)):
        x = synth.images(n, 3, 120, 160, seed=1000 + i)
        y = synth.labels_random(n, 120, 160, seed=1100 + i)
        key = ((n, 3, 120, 160), (n, 120, 160))
        replay = n in baked
        if replay:
            _assert_held(ev, baked[n], f"eval graph at batch {n}")
            g0 = ev._graphs[key]["graph"]
        out = ev(x.cuda(), y.cuda())
        if replay:
            assert ev._graphs[key]["graph"] is g0, "the call captured again instead of replaying"
        else:
            baked[n] = _baked(plan)
        if i == 1:
            _assert_replaced(plan, baked[256])
        with torch.no_grad():
            ref = R.pb_fcn_forward(sd64, x.double(), False)
            loss_ref = float(R.cross_entropy_2d(ref, y, cw64))
        err, flips = check_eval_outputs(f"pb_fcn pruned batch {n}", out, ref, ref.argmax(1), y, loss_ref)
        scale = max(1.0, float(ref.abs().max()))
        print(f"pb_fcn pruned {n}x3x120x160 ({'replay' if replay else 'capture'}): logits max err {err:.2e} "
              f"({err / scale:.2e} of the logit scale {scale:.1f}), argmax flips {flips}, loss rel err "
              f"{abs(float(out['loss']) - loss_ref) / abs(loss_ref):.2e}")
