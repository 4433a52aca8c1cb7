"""TrainStep(global_batch=True) without a GPU: the engine hooks (Plan.forward / Plan.backward with `batch_reduce`)
on two gloo ranks, each running the REAL plan on its half of the batch with ATen stand-ins of the kernels, against
autograd over the oracle forward on the FULL batch; argument validation of the new entry points; the refusal of
unequal shard shapes and of an unknown `reduce`."""
import ctypes as C
import os
import socket
import types

import pytest
import torch
import torch.nn.functional as F

CASES = ["robo_default", "robo_unet_pool", "pb_fcn", "labelprop"]
HEAD_CASES = ["robo_default", "labelprop"]
B, H, W = 2, 24, 32  # global batch: one image per rank


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


# ---- stand-ins for the entry points the global-batch schedule adds (fake_ops has the rest)
def _fake_module():
    import fake_ops
    mod = types.ModuleType("fake_ops_global_batch")
    mod.__dict__.update(fake_ops.__dict__)

    def bn_finalize_apply(z, stats, gamma, beta, running_mean, running_var, momentum, eps, relu, residual=None,
                          num_batches_tracked=None, count=None):
        if count is None:
            return fake_ops.bn_finalize_apply(z, stats, gamma, beta, running_mean, running_var, momentum, eps, relu,
                                              residual, num_batches_tracked)
        fake_ops.calls.append(("bn_finalize_apply_count", count))
        scale, shift, mean, invstd = fake_ops.bn_finalize(stats, count, gamma, beta, running_mean, running_var,
                                                          momentum, eps, num_batches_tracked)
        fake_ops.calls.pop()
        y = fake_ops.bn_apply(z, scale, shift, relu, residual)
        fake_ops.calls.pop()
        return y, scale, shift, mean, invstd

    def _g_xhat(order, dy, z, scale, shift, mean, invstd):
        g = dy
        if order == fake_ops.EPI_AFFINE_RELU:
            g = torch.where(z * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1) > 0, dy, torch.zeros_like(dy))
        return g, (z - mean.view(1, -1, 1, 1)) * invstd.view(1, -1, 1, 1)

    def bn_bwd_reduce(order, dy, z, scale, shift, mean, invstd, sums):
        fake_ops.calls.append(("bn_bwd_reduce", None))
        g, xhat = _g_xhat(order, dy, z, scale, shift, mean, invstd)
        c = z.shape[1]
        sums[:c] += g.double().sum((0, 2, 3))
        sums[c:] += (g.double() * xhat.double()).sum((0, 2, 3))

    def bn_bwd_apply(order, dy, z, scale, shift, mean, invstd, sums, dgamma=None, dbeta=None, dbias=None):
        """rcv_bn_bwd_apply: the channel means are sums / (N*HW of THIS z), subtracted at (better than) fp32 precision
        as the kernel's hi + lo pairs do."""
        fake_ops.calls.append(("bn_bwd_apply", None))
        g, xhat = _g_xhat(order, dy, z, scale, shift, mean, invstd)
        c, m = z.shape[1], z.numel() // z.shape[1]
        d = (g.double() - (sums[:c] / m).view(1, -1, 1, 1) - xhat.double() * (sums[c:] / m).view(1, -1, 1, 1))
        dz = scale.view(1, -1, 1, 1) * d.float()
        if order == fake_ops.EPI_RELU_AFFINE:
            dz = torch.where(z > 0, dz, torch.zeros_like(dz))
        if dgamma is not None:
            dgamma += sums[c:].float()
        if dbeta is not None:
            dbeta += sums[:c].float()
        if dbias is not None:
            dbias += dz.sum((0, 2, 3))
        return dz

    mod.bn_finalize_apply, mod.bn_bwd_reduce, mod.bn_bwd_apply = bn_finalize_apply, bn_bwd_reduce, bn_bwd_apply
    return mod


class _GlooReduce:
    """Plan's batch_reduce over dist.all_reduce (what TrainStep does with reduce="nccl")."""

    def __init__(self, world):
        self.world = world
        self.calls = 0

    def sum(self, buf):
        import torch.distributed as dist
        self.calls += 1
        dist.all_reduce(buf)

    def mean(self, buf):
        import torch.distributed as dist
        self.calls += 1
        dist.all_reduce(buf)
        buf /= self.world


def _views(plan):
    total = sum(p.numel() for p in plan.params)
    flat = torch.zeros(total)
    views, o = {}, 0
    for p in plan.params:
        views[id(p)] = flat[o:o + p.numel()].view(p.shape)
        o += p.numel()
    return flat, views


def _check_case(tag, rank, world, fused_head, reduce_batch):
    """One rank's run of one case -> list of failures (empty: the gradients summed over the ranks and the running
    statistics are those of the full batch)."""
    import torch.distributed as dist

    import synth
    from oracle import ref_model as R
    from robocupvision_b200.model import upSampleTransposeConv
    from test_plan_host import _cases
    make, oracle, cin = _cases()[tag]
    torch.manual_seed(12345678)
    m = make().train()
    plan = m._get_plan()
    x = synth.images(B, cin, H, W, seed=5)
    y = synth.labels_learnable(x[:, :3])
    cw = torch.tensor(synth.LP_CLASS_WEIGHTS if tag == "labelprop" else synth.CLASS_WEIGHTS)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    lo, hi = rank * B // world, (rank + 1) * B // world
    xl, yl = x[lo:hi].contiguous(), y[lo:hi].contiguous()

    def oracle_run(dtype):
        osd = R.leaf_state_dict({k: (v.clone().to(dtype) if v.is_floating_point() else v.clone()) for k, v in sd.items()})
        logits = oracle(osd, x.to(dtype), training=True)
        loss = R.cross_entropy_2d(logits, y, cw.to(dtype))
        loss.backward()
        return float(loss.detach()), logits.detach(), osd

    loss32, logits32, osd32 = oracle_run(torch.float32)
    loss64, _, osd64 = oracle_run(torch.float64)
    br = _GlooReduce(world) if reduce_batch else None
    fails = []
    with torch.no_grad():
        flat, views = _views(plan)
        sums = torch.zeros(2, dtype=torch.float64)
        corr = torch.zeros(1, dtype=torch.int64)
        if fused_head:
            head = plan.fusable_head()
            assert head == len(plan.nodes) - 1
            nd = plan.nodes[head]
            import fake_ops
            fake_ops.ce_weight_sum(yl, cw, sums[1:2], nd.geom.cout)
            if br is not None:
                br.sum(sums[1:2])
            _, saved = plan.forward(xl, training=True, save=True, stop_before=head, batch_reduce=br)
            dfeat = fake_ops.head_ce_train(saved[0][nd.src], nd.conv.weight, nd.conv.bias, yl, cw, sums, corr,
                                           views[id(nd.conv.weight)], views[id(nd.conv.bias)])
            plan.backward(saved, [None], False, views, seed={nd.src: dfeat}, batch_reduce=br)
            dist.all_reduce(sums[0:1])
            dist.all_reduce(corr)
        else:
            outs, saved = plan.forward(xl, training=True, save=True, batch_reduce=br)
            lg = outs[0].detach().clone().requires_grad_(True)
            den = cw.double()[yl].sum().reshape(1)
            dist.all_reduce(den)  # the weighted-mean normaliser of the GLOBAL batch
            with torch.enable_grad():
                nll = F.cross_entropy(lg, yl, weight=cw, reduction="sum")
                (nll / float(den)).backward()
            sums[0], sums[1] = float(nll), float(den)
            corr += (outs[0].argmax(1) == yl).sum()
            plan.backward(saved, [lg.grad], False, views, batch_reduce=br)
            dist.all_reduce(sums[0:1])
            dist.all_reduce(corr)
        dist.all_reduce(flat)  # the gradient all-reduce of the step: a SUM under global_batch
    n_bn = sum(1 for nd in plan.nodes if nd.bn is not None)
    if br is not None and br.calls != 2 * n_bn + (1 if fused_head else 0):
        fails.append(f"{tag}: {br.calls} exchanges for {n_bn} BatchNorm layers")
    if abs(float(sums[0] / sums[1]) - loss64) > 1e-5 * abs(loss64):
        fails.append(f"{tag}: loss {float(sums[0] / sums[1])} vs {loss64}")
    if int(corr) != int((logits32.argmax(1) == y).sum()):
        fails.append(f"{tag}: correct {int(corr)} vs {int((logits32.argmax(1) == y).sum())}")
    gmax = max(float(v.grad.abs().max()) for v in osd64.values() if v.grad is not None)

    def rel_l2(a, b):
        return float((a.double() - b).norm()) / max(float(b.norm()), 1e-3 * gmax * b.numel() ** 0.5)

    noise = {f"{n}.conv.bias" for n, mod in m.named_modules() if isinstance(mod, upSampleTransposeConv)}
    names = {id(p): k for k, p in m.named_parameters()}
    for p in plan.params:
        k = names[id(p)]
        if k in noise:
            continue
        g64 = osd64[k].grad
        err, floor = rel_l2(views[id(p)], g64), rel_l2(osd32[k].grad, g64)
        if err > max(1e-3, 4 * floor):
            fails.append(f"{tag}: grad {k} rel L2 err {err:.3e} (fp32 oracle {floor:.3e})")
    for k, b in m.named_buffers():
        if b.is_floating_point():
            if not torch.allclose(b, osd32[k], rtol=1e-5, atol=1e-6):
                fails.append(f"{tag}: buffer {k} max err {float((b - osd32[k]).abs().max()):.3e}")
        elif int(b) != int(osd32[k]):
            fails.append(f"{tag}: {k} {int(b)} vs {int(osd32[k])}")
    return fails


def _worker(rank, world, port, mode, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = {}
    try:
        if mode == "shards":
            from robocupvision_b200.train import check_equal_shards
            check_equal_shards(torch.zeros(2, 3, 24, 32), torch.zeros(2, 24, 32, dtype=torch.long))
            out["equal"] = "ok"
            try:
                check_equal_shards(torch.zeros(2 + rank, 3, 24, 32), torch.zeros(2 + rank, 24, 32, dtype=torch.long))
                out["unequal"] = "accepted"
            except ValueError as e:
                out["unequal"] = "refused" if "same shard shape" in str(e) else str(e)
        else:
            from robocupvision_b200 import engine
            engine.ops = _fake_module()
            engine.WGRAD_SIDE_STREAM = False
            for tag in CASES:
                out[("plain", tag)] = _check_case(tag, rank, world, False, True)
                # control: the same shards without the exchange (rank-local BatchNorm)
                ctl = _check_case(tag, rank, world, False, False)
                out[("control", tag)] = [f for f in ctl if "running_var" in f]
            for tag in HEAD_CASES:
                out[("head", tag)] = _check_case(tag, rank, world, True, True)
    except Exception as e:  # noqa: BLE001  (reported through the queue)
        import traceback
        out["error"] = f"{type(e).__name__}: {e}\n{traceback.format_exc()}"
    q.put((rank, out))
    dist.destroy_process_group()


def _run(mode, world=2):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, mode, q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    return outs


def test_global_batch_engine_hooks_match_full_batch_oracle_gloo():
    """Two gloo ranks, each with half of the batch, through the real Plan.forward / Plan.backward with batch_reduce
    (BatchNorm statistics summed over the ranks before finalize, which divides by the global count; the BatchNorm
    backward as two passes with the sums averaged between them): the gradients summed over the ranks equal autograd
    over the oracle forward on the FULL batch, and so do the running mean and variance (the unbiased factor of the
    global count) -- for ROBO_UNet, the --UNet pool variant, PB_FCN (AFFINE_RELU order) and LabelProp (partial skip),
    and through the fused-CE-head wiring (normaliser summed before the forward).  Control: without batch_reduce the
    running variances miss that gate."""
    outs = _run("hooks")
    for rank, out in outs.items():
        assert "error" not in out, out["error"]
        for tag in CASES:
            assert out[("plain", tag)] == [], (rank, out[("plain", tag)])
            assert out[("control", tag)], (rank, tag, "rank-local BatchNorm must miss the full-batch running variance")
        for tag in HEAD_CASES:
            assert out[("head", tag)] == [], (rank, out[("head", tag)])


def test_unequal_shard_shapes_are_refused_gloo():
    outs = _run("shards")
    for rank, out in outs.items():
        assert out == {"equal": "ok", "unequal": "refused"}, (rank, out)


def test_train_step_refuses_unknown_reduce():
    from robocupvision_b200.model import ROBO_UNet
    from robocupvision_b200.train import TrainStep
    with pytest.raises(ValueError, match="reduce"):
        TrainStep(ROBO_UNet(), reduce="bogus", global_batch=True)


def test_global_batch_entry_points_validate_without_gpu():
    from robocupvision_b200 import _lib
    lib = _lib.load()
    BAD = _lib.RCV_ERR_BAD_ARG
    p = C.c_void_p(16)  # never dereferenced: every case below is refused before a launch
    ptrs = (C.c_void_p * 2)(16, 32)
    st = C.c_void_p(64)
    assert lib.rcv_peer_allreduce_f64(2, 0, 14, ptrs, ptrs, 0, 4097, 1.0, st, None) == BAD
    assert b"4096" in lib.rcv_last_error()
    assert lib.rcv_peer_allreduce_f64(2, 0, 14, ptrs, ptrs, 0, 0, 1.0, st, None) == BAD
    assert lib.rcv_peer_allreduce_f64(2, 0, 16, ptrs, ptrs, 0, 4, 1.0, st, None) == BAD
    assert lib.rcv_peer_allreduce_f64(2, 2, 14, ptrs, ptrs, 0, 4, 1.0, st, None) == BAD
    assert lib.rcv_peer_allreduce_f64(9, 0, 14, ptrs, ptrs, 0, 4, 1.0, st, None) == BAD
    assert lib.rcv_peer_allreduce_f64(2, 0, 14, ptrs, ptrs, -1, 4, 1.0, st, None) == BAD
    assert lib.rcv_peer_allreduce_f64(2, 0, 14, ptrs, ptrs, 0, 4, 1.0, None, None) == BAD
    assert lib.rcv_peer_allreduce_i64(2, 0, 14, ptrs, ptrs, 0, 4097, st, None) == BAD
    assert lib.rcv_peer_allreduce_i64(2, 0, 14, None, ptrs, 0, 1, st, None) == BAD
    unaligned = (C.c_void_p * 2)(16, 36)
    assert lib.rcv_peer_allreduce_i64(2, 0, 14, unaligned, ptrs, 0, 1, st, None) == BAD
    args = [4, 8, 100, 0, p, p, p, p, p, 0.1, 1e-5, p, 0, None, 0, p, p, p, p, p, None, None]
    assert lib.rcv_bn_finalize_apply_count(*args) == BAD  # count 0
    args[3], args[4] = 800, None
    assert lib.rcv_bn_finalize_apply_count(*args) == BAD  # no statistics
