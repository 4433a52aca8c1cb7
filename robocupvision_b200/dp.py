"""Data-parallel gradient exchange: host-side bucket planning (backend-agnostic, so the gloo tests cover it).

Training is batch-sharded: rank r owns samples [r*B, (r+1)*B); BatchNorm statistics stay local
(the reference has no SyncBN); the only exchange per step is a sum all-reduce of the flat
gradient arena.  The arena is in ``model.parameters()`` order (encoder first, head last) and backward
visits the plan's nodes last to first, so the arena's TAIL holds final gradients first: it is cut
into a few contiguous buckets at plan-node boundaries, and ``train.TrainStep`` all-reduces bucket k
(and runs its optimiser pass) on a side stream as soon as backward has passed the bucket's first
node, while the remaining (encoder) backward still runs.  Only the last, small bucket is exposed.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple


def plan_buckets(node_params: Sequence[Sequence[Tuple[int, int]]], table: Sequence[Tuple[int, int]], total: int,
                 n_buckets: int = 3, tail_fraction: float = 0.02) -> List[Tuple[int, int, int]]:
    """Cut the arena [0, total) into <= n_buckets contiguous ranges at plan-node boundaries.

    node_params[t]: (offset, numel) of every parameter plan node t owns; table: (offset, numel) of every
    parameter in the arena (parameters no node owns -- e.g. PB_FCN's unused classification head -- never
    receive a gradient and may sit in any bucket).  Returns [(first_node, start, end)] in the order backward
    completes them (arena tail first): every gradient in [start, end) is final once backward has passed node
    `first_node`; the last entry has first_node = 0 and start = 0.  The buckets partition [0, total).

    Sizing: the LAST bucket's all-reduce cannot overlap anything (it waits for the last weight gradient), so it
    is kept small (about tail_fraction of the arena); the others split the rest evenly."""
    if total <= 0:
        return []
    nn = len(node_params)
    owned = {o for ps in node_params for o, _ in ps}
    # lo[t] = smallest arena offset owned by nodes >= t
    lo, cur = [total] * (nn + 1), total
    for t in range(nn - 1, -1, -1):
        for o, _ in node_params[t]:
            cur = min(cur, o)
        lo[t] = cur
    # a cut at node t (arena offset lo[t]) is valid if every OWNED parameter at or after lo[t] belongs to nodes >= t
    later = set()
    valid = []  # (t, offset)
    for t in range(nn - 1, 0, -1):
        later.update(o for o, _ in node_params[t])
        off = lo[t]
        if off >= total or (valid and off == valid[-1][1]):
            continue
        if all((o in later) or (o not in owned) for o, _ in table if o >= off):
            valid.append((t, off))
    # targets, from the tail: even shares of the arena above the small last bucket
    nb = max(1, int(n_buckets))
    cuts: List[Tuple[int, int]] = []
    if nb > 1 and valid:
        head = tail_fraction * total
        targets = [total - (total - head) * (k + 1) / (nb - 1) for k in range(nb - 1)]
        for tg in targets:
            # the valid cut closest to the target that lies strictly below the previous cut
            prev = cuts[-1][1] if cuts else total
            cands = [(abs(off - tg), t, off) for t, off in valid if 0 < off < prev]
            if not cands:
                break
            _, t, off = min(cands)
            cuts.append((t, off))
    out, end = [], total
    for t, off in cuts:
        out.append((t, off, end))
        end = off
    out.append((0, 0, end))
    return out


def allreduce_buckets(flat, buckets: Sequence[Tuple[int, int, int]], group=None):
    """Sum all-reduce every bucket in completion order (test / reference form of what TrainStep interleaves
    with backward)."""
    import torch.distributed as dist
    works = [dist.all_reduce(flat[a:b], group=group, async_op=True) for _, a, b in buckets]
    for w in works:
        w.wait()
    return flat


def self_check(model_ctor, class_weights, batch: int, cin: int, h: int, w: int, steps: int = 3, group=None,
               lr: float = 1e-3, l1_decay: float = 1e-6, seed: int = 777, use_graph: bool = True,
               force_comm_path: bool = True, tol: float = 5e-4, reduce=None, global_batch: bool = False) -> dict:
    """Numerical check of the data-parallel product path on THIS job's ranks (bench.py emits it as `dp_check`).

    Every rank trains `steps` steps of TrainStep (bucketed all-reduce + optimiser on the comm stream, captured in a
    CUDA graph, exactly the schedule of the timed run) on its own shard, and ALSO replays the same steps serially
    on one GPU with the single-GPU autograd path of the same kernels: gradients of all N shards accumulated with
    weight 1/N (per-shard BatchNorm statistics, as every rank computes them), + l1_decay*sign(p), torch.optim.Adam.
    The single-GPU path is pinned against the CPU oracle by tests/, so agreement here extends that pin to N ranks.
    Adam runs with eps = 1e-3 on both sides (with torch's default 1e-8 a gradient that is analytically zero moves
    its weight by +-lr according to the sign of rounding noise; see tests/test_gpu_models.py::test_step_async).
    Gate: weights within `tol` = 5e-4 of the largest weight after `steps` steps.  Two runs of the SAME schedule differ
    by up to ~1e-4 here (floating-point atomics in the weight-gradient kernels, passed on by Adam's normalisation:
    the control in tests/test_gpu_train.py::test_comm_path_schedule_matches_plain_step); a missing or mis-scaled
    all-reduce, or an optimiser pass racing a gradient, moves weights by the order of lr = 1e-3 per step.
    global_batch: check TrainStep(global_batch=True) instead; the serial reference is then one process stepping on
    the N shards concatenated into one batch (BatchNorm statistics and loss over all of it).

    -> {"ok", "world", "steps", "max_weight_err", "max_loss_err", "weights_identical_across_ranks"}"""
    import copy

    import torch
    import torch.distributed as dist

    from .model import CrossEntropyLoss2d
    from .train import TrainStep
    have_pg = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if have_pg else 1
    rank = dist.get_rank(group) if have_pg else 0
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(12345678)
    model = model_ctor().to(dev)
    if have_pg:
        for t in list(model.parameters()) + [b for b in model.buffers()]:
            dist.broadcast(t.data, 0, group=group)
    emu = copy.deepcopy(model)
    eps = 1e-3
    ts = TrainStep(model, class_weights, lr=lr, l1_decay=l1_decay, eps=eps, use_graph=use_graph,
                   process_group=group, force_comm_path=force_comm_path, reduce=reduce, global_batch=global_batch)
    crit = CrossEntropyLoss2d(torch.tensor(class_weights)).to(dev)
    opt = torch.optim.Adam(emu.parameters(), lr=lr, eps=eps)
    gen = torch.Generator().manual_seed(seed)
    max_loss = 0.0
    for s in range(steps):
        xs = torch.randn(world, batch, cin, h, w, generator=gen)
        ys = (torch.nn.functional.avg_pool2d(xs[:, :, 0], 5, 1, 2) * 3 + 2).clamp(0, len(class_weights) - 1).long()
        xs, ys = xs.to(dev), ys.to(dev)
        ts.step(xs[rank].contiguous(), ys[rank].contiguous())
        dp_loss = float(ts.loss_sums[0] / ts.loss_sums[1])
        emu.train()
        opt.zero_grad()
        if global_batch:
            loss_g = crit(emu(xs.flatten(0, 1)), ys.flatten(0, 1))
            max_loss = max(max_loss, abs(float(loss_g.detach()) - dp_loss) / max(1.0, abs(dp_loss)))
            loss_g.backward()
        for r in range(0 if global_batch else world):
            loss_r = crit(emu(xs[r].contiguous()), ys[r].contiguous())
            if r == rank:
                max_loss = max(max_loss, abs(float(loss_r.detach()) - dp_loss) / max(1.0, abs(dp_loss)))
            (loss_r / world).backward()
        with torch.no_grad():
            for p in emu.parameters():
                if p.grad is not None:
                    p.grad.add_(torch.sign(p), alpha=l1_decay)
        opt.step()
        emu._get_plan().epoch += 1  # the optimiser wrote the weights behind the plan's caches
    torch.cuda.synchronize()
    if ts.peer is not None:
        ts.peer.check()
    max_w = 0.0
    for p, q in zip(model.parameters(), emu.parameters()):
        max_w = max(max_w, float((p.detach() - q.detach()).abs().max()) / max(1.0, float(q.detach().abs().max())))
    identical = True
    if have_pg and world > 1:
        chk = torch.stack([ts.arena.double().sum(), ts.arena.double().abs().sum()])
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
        identical = bool(torch.equal(lo, hi))
        t = torch.tensor([max_w, max_loss], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        max_w, max_loss = float(t[0]), float(t[1])
    return {"ok": bool(max_w <= tol and max_loss <= 1e-4 and identical), "world": world, "steps": steps,
            "batch_per_rank": batch, "max_weight_err": max_w, "max_loss_err": max_loss,
            "weights_identical_across_ranks": identical, "buckets": [list(b) for b in ts.buckets],
            "graph": bool(use_graph), "reduce": ts.reduce if world > 1 or ts.peer is not None else "none", "reference": "serial N-shard gradient accumulation on one GPU "
            "(autograd path of the same kernels, pinned against the CPU oracle by tests/)"}
