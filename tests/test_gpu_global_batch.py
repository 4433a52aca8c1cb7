"""TrainStep(global_batch=True) on the GPU: the small-vector peer exchange (rcv_peer_allreduce_f64 / _i64) bit for bit,
the one-rank schedule against the plain step, two ranks x B/2 against one process on all B, the kernels a global-batch
step launches, and the compiler's resource report of the BatchNorm and peer-exchange kernels."""
import json
import os
import re
import subprocess
import sys
import tempfile
from pathlib import Path

import pytest
import torch

import synth
from test_gpu_train import _cuda_kernel_names, _foreign

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu

B, H, W, STEPS = 8, 48, 64, 4  # global batch of the two-rank tests (4 per rank), graph-replayed steps


def _case(name):
    """-> (model constructor, class weights, input channels, TrainStep kwargs)."""
    from robocupvision_b200.model import LabelProp, ROBO_UNet
    return {
        "robo_ce": (ROBO_UNet, synth.CLASS_WEIGHTS, 3, {}),
        "robo_dice": (ROBO_UNet, synth.CLASS_WEIGHTS, 3, {"loss": "dice"}),
        "v2_ce": (lambda: ROBO_UNet(v2=True, classSize=3), synth.CLASS_WEIGHTS, 3, {}),  # 3x3 classifier: unfused
        "labelprop_ce": (lambda: LabelProp(5, 32, 0), synth.LP_CLASS_WEIGHTS, 8, {}),
    }[name]


def _batch(name, s):
    _, cw, cin, _ = _case(name)
    x = synth.images(B, cin, H, W, seed=700 + s)
    return x, synth.labels_learnable(x[:, :3], num_classes=len(cw))


def _run_steps(name, rank=0, world=1, **kw):
    """STEPS graph-replayed steps of case `name` on this rank's shard of the global batch -> record."""
    from robocupvision_b200.train import TrainStep
    ctor, cw, _, extra = _case(name)
    torch.manual_seed(12345678)
    m = ctor().cuda()
    ts = TrainStep(m, cw, lr=1e-3, l1_decay=1e-6, eps=1e-3, use_graph=True, **extra, **kw)
    losses, data_loss, correct = [], [], []
    lo, hi = rank * B // world, (rank + 1) * B // world
    for s in range(STEPS):
        x, y = _batch(name, s)
        ts.step(x[lo:hi].contiguous().cuda(), y[lo:hi].contiguous().cuda())
        losses.append(ts.loss_value())
        num, den = ts.loss_sums.tolist()
        data_loss.append(num / den)  # without the L1 term (an fp64 atomic sum over the weights on each rank)
        correct.append(int(ts.correct))
    torch.cuda.synchronize()
    return {"losses": losses, "data_loss": data_loss, "correct": correct, "global_batch": ts.global_batch,
            "state": {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}}


_RANK = r"""
import os, sys, torch
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import torch.distributed as dist
rank, world, port, mode, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4], sys.argv[5]
os.environ['MASTER_ADDR'] = '127.0.0.1'; os.environ['MASTER_PORT'] = port
os.environ.setdefault('RCV_PEER_TIMEOUT_S', '20')
torch.cuda.set_device(0)
dist.init_process_group('gloo', rank=rank, world_size=world)
res = {{}}
if mode == 'kernel':
    from robocupvision_b200.peer import PeerExchange
    n = 300
    px = PeerExchange(64, 'cuda:0', ndoubles=n)
    acc, acc_i = px.accum, px.accum.view(torch.int64)
    ranges = [(0, n, 1.0), (7, 40, 0.5), (299, 300, 1.0), (5, 6, 0.5), (0, n, 0.5)]
    bad = []
    for it in range(3):
        for k, (a, b, scale) in enumerate(ranges):
            g = torch.Generator().manual_seed(100 * it + k)
            data = torch.randn(world, n, generator=g, dtype=torch.float64) * 1e3
            acc.copy_(data[rank])
            px.allreduce_f64(acc[a:b], scale)
            torch.cuda.synchronize()
            s = data[0, a:b].clone()
            for q in range(1, world):
                s += data[q, a:b]          # rank order, as the kernel adds
            expect = data[rank].clone()
            expect[a:b] = s * scale
            if not torch.equal(acc.cpu(), expect):
                bad.append(('f64', it, k))
            dist.barrier()
            ints = torch.randint(-2 ** 40, 2 ** 40, (world, n), generator=g, dtype=torch.int64)
            acc_i.copy_(ints[rank])
            px.allreduce_i64(acc_i[a:b])
            torch.cuda.synchronize()
            expect = ints[rank].clone()
            expect[a:b] = ints[:, a:b].sum(0)
            if not torch.equal(acc_i.cpu(), expect):
                bad.append(('i64', it, k))
            dist.barrier()
    px.check()
    res = {{'bad': bad}}
else:
    from test_gpu_global_batch import _run_steps
    for name in ('robo_ce', 'robo_dice', 'v2_ce', 'labelprop_ce'):
        res[name] = _run_steps(name, rank, world, global_batch=True, reduce='peer')
    res['robo_ce_local'] = _run_steps('robo_ce', rank, world, global_batch=False, reduce='peer')
torch.save(res, out)
print('RANK_DONE'); sys.stdout.flush()
torch.cuda.synchronize(); dist.barrier(); os._exit(0)
"""


def _run_ranks(mode, port, world=2, timeout=600):
    """`world` processes on THIS GPU (the peer mapping, flags and barriers do not care that the peers share a device),
    gloo for the handle exchange and the shard check."""
    code = _RANK.format(root=str(ROOT), tests=str(ROOT / "tests"))
    with tempfile.TemporaryDirectory() as d:
        outs = [os.path.join(d, f"rank{r}.pt") for r in range(world)]
        procs = [subprocess.Popen([sys.executable, "-c", code, str(r), str(world), port, mode, outs[r]],
                                  stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(world)]
        try:
            for p in procs:
                o, e = p.communicate(timeout=timeout)
                assert "RANK_DONE" in o, o[-1500:] + e[-3000:]
        finally:
            for p in procs:
                if p.poll() is None:
                    p.kill()
        return [torch.load(f, weights_only=False) for f in outs]


def test_peer_small_allreduce_two_ranks():
    """rcv_peer_allreduce_f64 / _i64: the result equals the rank-order sum (times scale) bit for bit on both ranks,
    values outside the range stay untouched; whole region, interior, one-element ranges, scale 1/2, three rounds per
    slot."""
    for r in _run_ranks("kernel", "29693"):
        assert r == {"bad": []}, r


def _rel(a, b):
    return float((a.double() - b.double()).abs().max()) / max(1.0, float(b.double().abs().max()))


def test_global_batch_two_ranks_match_one_process():
    """Two ranks x B/2 with global_batch=True (peer path) against one process stepping on all B: per-step losses to
    1e-5 relative, weights within max(3e-4, 3x a one-process control), running statistics to 1e-5 relative,
    num_batches_tracked equal; the ranks' parameters, buffers, loss (without the L1 term) and counts bitwise identical.  Correct counts: exact at the first
    step (the same weights); after that the weights carry the floating-point-atomic noise of the weight gradients
    (Adam passes it on), which can flip an argmax tie, so they may differ by up to 1e-4 of the pixels or by what the
    one-process control shows.  Covers ROBO_UNet with CE (fused head) and Dice (fused), the unfused 3x3 head of
    ROBO_UNet(v2=True, classSize=3), and LabelProp.  Premise: the same ranks without global_batch miss the
    running-statistics gate."""
    ranks = _run_ranks("train", "29694")
    bad = []
    for name in ("robo_ce", "robo_dice", "v2_ce", "labelprop_ce", "robo_ce_local"):
        one = _run_steps(name.replace("_local", ""))
        ctl = _run_steps(name.replace("_local", ""))
        r0, r1 = ranks[0][name], ranks[1][name]
        assert r0["global_batch"] == (name != "robo_ce_local") and not one["global_batch"]
        if name == "robo_ce_local":
            worst = max(_rel(r0["state"][k], one["state"][k]) for k in r0["state"]
                        if k.endswith("running_var") or k.endswith("running_mean"))
            if not worst > 1e-5:
                bad.append(f"premise: rank-local BatchNorm is only {worst:.2e} from the full batch")
            continue
        bad += [f"{name}: {k} differs between the ranks" for k in r0["state"]
                if not torch.equal(r0["state"][k], r1["state"][k])]
        if r0["data_loss"] != r1["data_loss"] or r0["correct"] != r1["correct"]:
            bad.append(f"{name}: the ranks report different losses / counts")
        if any(abs(a - b) > 1e-5 * abs(b) for a, b in zip(r0["losses"], one["losses"])):
            bad.append(f"{name}: losses {r0['losses']} vs {one['losses']}")
        for s, (a, b, c) in enumerate(zip(r0["correct"], one["correct"], ctl["correct"])):
            if a != b and (s == 0 or abs(a - b) > max(1e-4 * B * H * W, abs(c - b))):
                bad.append(f"{name}: correct {r0['correct']} vs {one['correct']} (control {ctl['correct']})")
        for k, b in one["state"].items():
            a = r0["state"][k]
            if not b.is_floating_point():
                if not torch.equal(a, b):
                    bad.append(f"{name}: {k} {a} vs {b}")
            elif k.endswith("running_mean") or k.endswith("running_var"):
                if _rel(a, b) > 1e-5:
                    bad.append(f"{name}: {k} {_rel(a, b):.2e}")
            else:
                err, noise = _rel(a, b), _rel(ctl["state"][k], b)
                if err > max(3e-4, 3 * noise):
                    bad.append(f"{name}: {k} {err:.2e} (control {noise:.2e})")
        print(f"{name}: losses {r0['losses']} / {one['losses']}, correct {r0['correct']} / {one['correct']}")
    assert not bad, bad


def _bn_layers_leaving_the_cluster_kernel(plan, n, h, w):
    """BatchNorm layers whose backward rcv_bn_bwd runs as one cluster launch at this size: under global_batch they
    run as two passes."""
    from robocupvision_b200 import _lib
    lib = _lib.load()
    k = 0
    for nd, (nn_, ih, iw) in zip(plan.nodes, plan._in_sizes(n, h, w)):
        if nd.bn is not None:
            oh, ow = nd.geom.out_hw(ih, iw)
            k += int(lib.rcv_bn_bwd_is_fused(nn_, nd.geom.cout, oh * ow))
    return k


def test_global_batch_one_rank_matches_plain_step():
    """World 1: TrainStep(global_batch=True, force_comm_path=True) runs every exchange at world 1 (local flags) and
    must perform the plain step: losses within 2e-6, weights within max(3e-4, 3x a plain-vs-plain control).  Its
    launch count is the plain step's plus the bucket exchanges, one exchange per BatchNorm layer in each direction,
    the normaliser and the two end-of-step exchanges, plus one launch per BatchNorm backward that leaves the cluster
    kernel; a profiled replay launches library kernels only.  global_batch=True without force_comm_path is a no-op:
    the plain step's launches."""
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import TrainStep
    models, steps = [], []
    for kw in ({}, {"global_batch": True, "force_comm_path": True}, {}, {"global_batch": True}):
        torch.manual_seed(12345678)
        m = ROBO_UNet().cuda()
        models.append(m)
        steps.append(TrainStep(m, synth.CLASS_WEIGHTS, lr=1e-3, l1_decay=1e-6, eps=1e-3, use_graph=True, **kw))
    assert steps[1].global_batch and steps[1].peer is not None and not steps[3].global_batch
    for s in range(5):
        x = synth.images(8, 3, 120, 160, seed=200 + s).cuda()
        y = synth.labels_learnable(x.cpu()).cuda()
        losses = []
        for ts in steps:
            ts.step(x, y)
            losses.append(ts.loss_value())
        assert abs(losses[0] - losses[1]) <= 2e-6 * abs(losses[0]), (s, losses)
    plan = steps[1].plan
    n_bn = sum(1 for nd in plan.nodes if nd.bn is not None)
    assert n_bn == 15
    extra = len(steps[1].buckets) + 2 * n_bn + 1 + 2 + _bn_layers_leaving_the_cluster_kernel(plan, 8, 120, 160)
    print(f"launches: plain {steps[0].kernels_per_step}, global batch {steps[1].kernels_per_step} (+{extra})")
    assert steps[1].kernels_per_step == steps[0].kernels_per_step + extra
    assert steps[3].kernels_per_step == steps[0].kernels_per_step
    for (k, a), (_, b), (_, c) in zip(*(m.state_dict().items() for m in models[:3])):
        if a.is_floating_point():
            scale = max(1.0, float(a.abs().max()))
            noise = float((a - c).abs().max()) / scale
            err = float((a - b).abs().max()) / scale
            assert err <= max(3e-4, 3.0 * noise), f"{k}: global-batch deviation {err:.2e}, control {noise:.2e}"
        else:
            assert torch.equal(a, b), k
    names = _cuda_kernel_names(lambda: steps[1].step(x, y))
    assert any("peer_small_allreduce" in n for n in names), names
    assert len(names) >= 20 and not _foreign(names), f"non-library kernels in a global-batch step: {_foreign(names)}"
    plain = _cuda_kernel_names(lambda: steps[0].step(x, y))
    assert sorted(_cuda_kernel_names(lambda: steps[3].step(x, y))) == sorted(plain)


_KEY = re.compile(r"_ZN\d+_GLOBAL__N__[0-9a-f]{8}_\d+_\w+?_cu_[0-9a-f]{8}")


def _ptxas(src: Path, tmp: Path) -> dict:
    """{kernel: {registers, smem, spill: [stores, loads]}} of `nvcc -Xptxas -v` for one source file."""
    from robocupvision_b200.build import NVCC_FLAGS, _nvcc
    r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-Xptxas", "-v", "-c", str(src), "-o", str(tmp / (src.stem + ".o"))],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '([^']+)'", line)
        if m:
            cur = _KEY.sub("_ZN_anon_", m.group(1))
            out[cur] = {}
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            out[cur]["spill"] = [int(m.group(1)), int(m.group(2))]
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            s = re.search(r"(\d+) bytes smem", line)
            out[cur]["registers"], out[cur]["smem"] = int(m.group(1)), int(s.group(1)) if s else 0
    return out


def test_batchnorm_and_peer_kernels_keep_their_resources(tmp_path):
    """-Xptxas -v: every kernel of rcv_bn.cu and rcv_peer.cu that existed before the global-batch exchange keeps its
    registers, spills and shared memory (tests/golden/ptxas_bn_peer.json); the new exchange kernels do not spill."""
    golden = json.loads((ROOT / "tests" / "golden" / "ptxas_bn_peer.json").read_text())
    for fname, want in golden.items():
        got = _ptxas(ROOT / "robocupvision_b200" / "csrc" / fname, tmp_path)
        for k, v in want.items():
            assert got.get(k) == v, (fname, k, got.get(k), v)
        new = {k: v for k, v in got.items() if k not in want}
        if fname == "rcv_peer.cu":
            assert len(new) == 2 and all("peer_small_allreduce" in k for k in new), new
        else:
            assert not new, new
        for k, v in new.items():
            assert v["spill"] == [0, 0], (k, v)
