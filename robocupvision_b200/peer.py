"""Gradient exchange over NVLink peer memory: host side of ``rcv_peer_allreduce`` (csrc/rcv_peer.cu).

One ``PeerExchange`` per ``TrainStep``: it owns the rank's flat GRADIENT arena (a cudaMalloc block every rank of the
group maps through a cudaIpc handle), followed by the flag words of the kernel's two barriers.  The process group is
used ONCE, to exchange the 64-byte handles (any backend: the data path never touches it); after that
``allreduce(slot, a, b)`` is one kernel launch on the current stream that leaves the sum over ranks of
``grads[a:b]`` in every rank's arena -- bitwise identical on all ranks (each element is summed once, in rank order, by
the rank that owns its share).  Replaces ``dist.all_reduce(grads[a:b])`` of the bucketed schedule in train.py.

With ``ndoubles`` > 0 the block also holds an fp64 region after the arena, ``accum`` ([grads | accum | flags]):
``allreduce_f64`` / ``allreduce_i64`` sum small slices of it over the ranks (rcv_peer_allreduce_f64 / _i64, one CTA),
which is how TrainStep(global_batch=True) shares BatchNorm statistics, loss normalisers and correct counts.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Tuple

import torch

from . import _lib

SLOTS = 16
SMALL_SLOT = SLOTS - 2  # the small-vector exchanges of a global-batch step (main stream); buckets use 0, 1, ...


def share_bounds(count: int, world: int, rank: int) -> Tuple[int, int]:
    """[lo, hi) of the range [0, count) (floats, count % 4 == 0) that `rank` sums: ceil-divided in float4 units, the
    rule of peer_allreduce_kernel."""
    if count % 4 or count < 0 or not 0 <= rank < world:
        raise ValueError(f"share_bounds: count {count}, world {world}, rank {rank}")
    c4 = count // 4
    per = -(-c4 // world)
    lo = min(rank * per, c4)
    return 4 * lo, 4 * min(lo + per, c4)


class _RawCuda:
    """A raw device range as a __cuda_array_interface__ object (torch.as_tensor wraps it without copying)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class PeerUnavailable(RuntimeError):
    """The ranks' GPUs cannot map each other's memory (raised on EVERY rank of the group, or on none)."""


class PeerExchange:
    def __init__(self, nfloats: int, device, group=None, ndoubles: int = 0):
        import torch.distributed as dist
        if nfloats <= 0 or nfloats % 4:
            raise ValueError(f"PeerExchange: arena of {nfloats} floats (must be a positive multiple of 4)")
        if ndoubles < 0:
            raise ValueError(f"PeerExchange: {ndoubles} doubles")
        self.dev = torch.device(device)
        have = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if have else 1
        self.rank = dist.get_rank(group) if have else 0
        if self.world > 8:
            raise ValueError(f"PeerExchange: {self.world} ranks (one NVSwitch node: at most 8)")

        def gather(obj):
            if self.world == 1:
                return [obj]
            every: List = [None] * self.world
            dist.all_gather_object(every, obj, group=group)
            return every

        lib = _lib.load()
        self.arena_bytes = 4 * nfloats
        self.accum_bytes = -(-8 * ndoubles // 16) * 16
        self.flag_bytes = int(lib.rcv_peer_flag_bytes())
        self._own, self._opened = None, []
        # every step below ends in a gather of its outcome, so the ranks fail together or not at all
        handle, why = None, ""
        try:
            with torch.cuda.device(self.dev):
                torch.cuda.synchronize()
                base = C.c_void_p()
                hbuf = (C.c_ubyte * 64)()
                _lib.call("rcv_peer_alloc", C.c_uint64(self.arena_bytes + self.accum_bytes + self.flag_bytes),
                          C.byref(base), hbuf)
            self._own, handle = base.value, bytes(hbuf)
        except Exception as e:  # noqa: BLE001  (whatever went wrong here, the other ranks must hear of it)
            why = f"{type(e).__name__}: {e}"
        every = sorted(gather((self.rank, handle, why)), key=lambda t: t[0])
        if any(h is None for _, h, _ in every):
            self._release()
            raise PeerUnavailable("; ".join(f"rank {r}: {w}" for r, h, w in every if h is None))
        bases, why = [], ""
        try:
            with torch.cuda.device(self.dev):
                for r, h, _ in every:
                    if r == self.rank:
                        bases.append(self._own)
                        continue
                    ptr = C.c_void_p()
                    _lib.call("rcv_peer_open", (C.c_ubyte * 64).from_buffer_copy(h), C.byref(ptr))
                    self._opened.append(ptr.value)
                    bases.append(ptr.value)
        except Exception as e:  # noqa: BLE001  (whatever went wrong here, the other ranks must hear of it)
            why = f"{type(e).__name__}: {e}"
        outcome = gather((self.rank, why))
        if any(w for _, w in outcome):
            self._release()
            raise PeerUnavailable("; ".join(f"rank {r}: {w}" for r, w in outcome if w))
        self._arenas = (C.c_void_p * self.world)(*bases)
        self._accums = (C.c_void_p * self.world)(*[b + self.arena_bytes for b in bases])
        self._flags = (C.c_void_p * self.world)(*[b + self.arena_bytes + self.accum_bytes for b in bases])
        self._raw = _RawCuda(self._own, self.arena_bytes)
        self.grads = torch.as_tensor(self._raw, device=self.dev).view(torch.float32)
        self.accum = None
        if ndoubles:
            self._raw_acc = _RawCuda(self._own + self.arena_bytes, 8 * ndoubles)
            self.accum = torch.as_tensor(self._raw_acc, device=self.dev).view(torch.float64)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.dev)
        # one real exchange before anything depends on it: rank r contributes r + 1, everyone must read N(N+1)/2
        why = ""
        try:
            with torch.cuda.device(self.dev):
                self.grads[:4] = float(self.rank + 1)
                self.allreduce(SLOTS - 1, 0, 4)
                got = self.grads[:4].tolist()
                if int(self.status.item()) != 0 or got != [self.world * (self.world + 1) / 2.0] * 4:
                    why = f"self-test read {got}"
                self.grads[:4] = 0.0
                torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            why = f"{type(e).__name__}: {e}"
        outcome = gather((self.rank, why))
        if any(w for _, w in outcome):
            self._release()
            raise PeerUnavailable("; ".join(f"rank {r}: {w}" for r, w in outcome if w))

    def _release(self) -> None:
        try:
            with torch.cuda.device(self.dev):
                torch.cuda.synchronize()
                for p in self._opened:
                    _lib.call("rcv_peer_close", C.c_void_p(p))
                if self._own is not None:
                    _lib.call("rcv_peer_free", C.c_void_p(self._own))
        except Exception:  # noqa: BLE001  (clean-up on a failure path: the failure itself is what gets reported)
            pass
        self._opened, self._own, self.grads, self.accum = [], None, None, None

    def allreduce(self, slot: int, a: int, b: int) -> None:
        """grads[a:b] <- sum over ranks, on the current stream (capture-safe)."""
        from . import ops
        if not 0 <= slot < SLOTS:
            raise ValueError(f"PeerExchange.allreduce: slot {slot} of {SLOTS}")
        ops._call("rcv_peer_allreduce", 1, self.world, self.rank, slot, self._arenas, self._flags, a, b - a,
                  ops._ptr(self.status), ops._stream())

    def _acc_offset(self, t: torch.Tensor) -> int:
        """Element offset of t (a contiguous 8-byte slice of `accum`) in the fp64 region."""
        off = -1 if self.accum is None else t.data_ptr() - self.accum.data_ptr()
        if (t.element_size() != 8 or not t.is_contiguous() or off < 0 or off % 8
                or off + 8 * t.numel() > 8 * self.accum.numel()):
            raise ValueError("PeerExchange: the tensor is not a slice of the peer-mapped fp64 region")
        return off // 8

    def allreduce_f64(self, t: torch.Tensor, scale: float = 1.0, slot: int = SMALL_SLOT) -> None:
        """t <- scale * sum over ranks, t a float64 slice of `accum`; on the current stream (capture-safe)."""
        from . import ops
        ops._call("rcv_peer_allreduce_f64", 1, self.world, self.rank, slot, self._accums, self._flags,
                  self._acc_offset(t), t.numel(), float(scale), ops._ptr(self.status), ops._stream())

    def allreduce_i64(self, t: torch.Tensor, slot: int = SMALL_SLOT) -> None:
        """t <- sum over ranks, t an int64 view of a slice of `accum`; on the current stream (capture-safe)."""
        from . import ops
        ops._call("rcv_peer_allreduce_i64", 1, self.world, self.rank, slot, self._accums, self._flags,
                  self._acc_offset(t), t.numel(), ops._ptr(self.status), ops._stream())

    def check(self) -> None:
        """Raise if a launch gave up waiting for a peer (host read: call where the step's scalars are read)."""
        if int(self.status.item()) != 0:
            raise RuntimeError("robocupvision_b200: a rank did not reach rcv_peer_allreduce within RCV_PEER_TIMEOUT_S; "
                               "the gradients of that step are invalid")

    def close(self) -> None:
        """Unmap the peers' blocks and free the own one.  Collective in spirit: call it on every rank once no rank
        will launch another exchange (a peer that still reads a freed block faults)."""
        if self._own is not None:
            self._release()
