"""Rank plumbing for the one exchange step of the path (global extrema).

``torch.distributed`` carries the collectives: NCCL over NVLink/NVSwitch on the GPU box
(tensors stay on the device), gloo in the CPU tests.  The payloads are tiny (bucket totals
of the radix histograms, a few scalars), so latency, not bandwidth, is what matters.
"""

from __future__ import annotations

import numpy as np


def rank_world():
    """``(rank, world size, torch.distributed)`` of this process; ``(0, 1, None)`` outside an initialised job."""
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size(), dist
    except ImportError:
        pass
    return 0, 1, None


def current_device() -> int:
    """The calling thread's CUDA device (``torchrun`` workers select theirs with ``torch.cuda.set_device``).
    Read it on the thread that was called: a new host thread starts on device 0."""
    try:
        import torch

        if torch.cuda.is_available():
            return int(torch.cuda.current_device())
    except ImportError:
        pass
    return 0


def block_of(n: int, rank: int, world: int) -> tuple[int, int]:
    """``[lo, hi)``: the rank's contiguous block of ``n`` ordered items, ``ceil(n / world)`` per rank (ranks past
    the end get an empty block, ``lo >= hi``)."""
    per = -(-n // world)
    return rank * per, min(n, (rank + 1) * per)


class TorchComm:
    def __init__(self, dist, device=None, group=None):
        """``group``: the process group the collectives run in (``None``: the default group)."""
        import torch

        self.torch = torch
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.size = dist.get_world_size(group)
        self.device = device if device is not None else torch.device("cpu")

    def allgather(self, arr: np.ndarray) -> list[np.ndarray]:
        """All-gather equally shaped numpy arrays (histogram-merge payload)."""
        torch = self.torch
        arr = np.ascontiguousarray(arr)
        view = arr.view(np.uint8).reshape(-1)
        t = torch.from_numpy(view.copy()).to(self.device)
        outs = [torch.empty_like(t) for _ in range(self.size)]
        self.dist.all_gather(outs, t, group=self.group)
        return [o.cpu().numpy().view(arr.dtype).reshape(arr.shape) for o in outs]

    def allgather_object(self, obj):
        outs = [None] * self.size
        self.dist.all_gather_object(outs, obj, group=self.group)
        return outs

    def barrier(self):
        self.dist.barrier(group=self.group)

    # ---- device-pointer collectives (NCCL): the payload never leaves HBM, nothing blocks the host
    def _tensor(self, ptr: int, nbytes: int):
        key = (ptr, nbytes)
        cache = self.__dict__.setdefault("_tensors", {})
        t = cache.get(key)
        if t is None:
            holder = type("CudaPtr", (), {})()
            holder.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
            t = cache[key] = self.torch.as_tensor(holder, device=self.device)
        return t

    def _on(self, stream_handle: int):
        """Order the collective behind (and the following work after) the given cudaStream_t --
        the libcsgpu context's stream -- whatever torch's current stream happens to be."""
        torch = self.torch
        if not stream_handle:
            return torch.cuda.stream(torch.cuda.current_stream(self.device))
        cache = self.__dict__.setdefault("_streams", {})
        ext = cache.get(stream_handle)
        if ext is None:
            ext = cache[stream_handle] = torch.cuda.ExternalStream(stream_handle, device=self.device)
        return torch.cuda.stream(ext)

    def stream_scope(self, stream_handle: int):
        """Context manager: inside it the device collectives may be called with
        ``stream_handle=None`` (no per-call stream switch -- a dozen tiny collectives per step)."""
        return self._on(stream_handle)

    def allgather_dev(self, src_ptr: int, dst_ptr: int, nbytes: int, stream_handle: int | None = 0):
        """dst[rank][nbytes] <- every rank's src[nbytes], enqueued behind the context stream's work."""
        dst, src = self._tensor(dst_ptr, nbytes * self.size), self._tensor(src_ptr, nbytes)
        if stream_handle is None:
            self.dist.all_gather_into_tensor(dst, src, group=self.group)
            return
        with self._on(stream_handle):
            self.dist.all_gather_into_tensor(dst, src, group=self.group)

    def allreduce_max_dev(self, ptr: int, count: int, kind: str, stream_handle: int | None = 0):
        key = (ptr, count, kind)
        cache = self.__dict__.setdefault("_typed", {})
        t = cache.get(key)
        if t is None:
            torch = self.torch
            dt = {"i8": torch.int64, "f8": torch.float64, "i4": torch.int32}[kind]
            t = cache[key] = self._tensor(ptr, count * dt.itemsize).view(dt)
        if stream_handle is None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
            return
        with self._on(stream_handle):
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)


# ----------------------------------------------------------------------------------------
# Exchanges: "every rank contributes nbytes, every rank sees all of them", on the context
# stream, device memory in and out.  The pooled-extrema selection (pool_select.py) is written
# against this one call.
# ----------------------------------------------------------------------------------------
class LocalExchange:
    """One rank: the payload is its own gather."""

    rank, size, kind = 0, 1, "local"
    error_ptr = None

    def ensure(self, slot_bytes: int):
        pass

    def allgather(self, src_ptr: int, nbytes: int) -> int:
        return src_ptr


class NcclExchange:
    """NCCL all-gather (``torch.distributed``) into a persistent device buffer; everything is
    stream-ordered, so one buffer serves every exchange of a step."""

    kind = "nccl"
    error_ptr = None

    def __init__(self, comm: TorchComm, ctx):
        self.comm, self.ctx = comm, ctx
        self.rank, self.size = comm.rank, comm.size
        self.buf = None

    def ensure(self, slot_bytes: int):
        if self.buf is None or self.buf.nbytes < slot_bytes * self.size:
            self.buf = self.ctx.alloc(slot_bytes * self.size)

    def allgather(self, src_ptr: int, nbytes: int) -> int:
        self.comm.allgather_dev(src_ptr, self.buf.ptr, nbytes, None)  # inside TorchComm.stream_scope
        return self.buf.ptr


class PeerExchange:
    """Mailboxes in every rank's HBM, written by the peers over NVLink (``csrc/peer.cu``)."""

    kind = "peer"

    def __init__(self, ctx, rank: int, size: int):
        self.ctx, self.rank, self.size = ctx, rank, size
        self.handle = None
        self.slot_bytes = 0
        self.error_ptr = None

    def _create(self, slot_bytes: int) -> bytes:
        import ctypes as C

        self.destroy()
        out, ipc = C.c_void_p(), (C.c_ubyte * 64)()
        self.ctx._check(self.ctx.lib.csg_peer_create(self.ctx.handle, self.rank, self.size, slot_bytes, C.byref(out), ipc))
        self.handle, self.slot_bytes = out.value, slot_bytes
        self.error_ptr = self.ctx.lib.csg_peer_error_word(self.handle)
        return bytes(ipc)

    def mailbox(self) -> int:
        return self.ctx.lib.csg_peer_mailbox(self.handle)

    def connect_ipc(self, handles: list[bytes]):
        import ctypes as C

        blob = b"".join(handles)
        self.ctx._check(self.ctx.lib.csg_peer_connect_ipc(self.ctx.handle, self.handle, C.c_char_p(blob)))

    def connect_ptrs(self, mailboxes: list[int]):
        import ctypes as C

        arr = (C.c_void_p * len(mailboxes))(*mailboxes)
        self.ctx._check(self.ctx.lib.csg_peer_connect_ptrs(self.ctx.handle, self.handle, arr))

    def ensure(self, slot_bytes: int):
        """Collective when the mailboxes must grow (every rank computes the same sizes)."""
        if self.handle is not None and self.slot_bytes >= slot_bytes:
            return
        self._grow(slot_bytes)

    def _grow(self, slot_bytes: int):
        """Abstract: (re)create the mailboxes with room for ``slot_bytes`` per rank and wire the ranks up
        (CUDA IPC in :class:`IpcPeerExchange`, raw pointers in :class:`_SharedPeer`)."""
        raise NotImplementedError(f"{type(self).__name__} must implement _grow()")

    def wait_stats(self, last_n: int = 64) -> dict:
        """``{"mean_us", "max_us"}`` of the time the last ``last_n`` exchanges spent waiting for the other
        ranks' epochs (rank skew + link latency; ``clock64`` inside the exchange kernel)."""
        import ctypes as C

        if self.handle is None:
            return {"mean_us": 0.0, "max_us": 0.0}
        mean, top = C.c_double(), C.c_double()
        self.ctx._check(self.ctx.lib.csg_peer_wait_stats(self.ctx.handle, self.handle, int(last_n), C.byref(mean), C.byref(top)))
        return {"mean_us": mean.value, "max_us": top.value}

    def trace(self, last_n: int = 12) -> list[list[float]]:
        """Timeline of the last ``last_n`` exchanges, oldest first: ``[kernel start, epoch published, every
        peer's epoch seen]`` in microseconds since the first entry's start (``%globaltimer`` of this GPU)."""
        import ctypes as C

        import numpy as np

        if self.handle is None:
            return []
        ns = np.zeros(3 * 64, dtype=np.uint64)
        n = C.c_int()
        self.ctx._check(self.ctx.lib.csg_peer_trace(self.ctx.handle, self.handle, int(last_n), ns.ctypes.data, C.byref(n)))
        rows = ns[: 3 * n.value].reshape(-1, 3).astype(np.int64)
        if not len(rows):
            return []
        return [[round(float(v - rows[0, 0]) / 1e3, 2) for v in row] for row in rows]

    def allgather(self, src_ptr: int, nbytes: int) -> int:
        import ctypes as C

        out = C.c_void_p()
        self.ctx._check(self.ctx.lib.csg_peer_allgather(self.ctx.handle, self.handle, src_ptr, nbytes, C.byref(out)))
        return out.value

    def clear_error(self):
        self.ctx._check(self.ctx.lib.csg_peer_clear_error(self.ctx.handle, self.handle))

    def destroy(self):
        if self.handle is not None:
            self.ctx.lib.csg_peer_destroy(self.ctx.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class IpcPeerExchange(PeerExchange):
    """One process per GPU: mailboxes mapped through CUDA IPC handles exchanged once over
    ``torch.distributed`` (plumbing); the data path never touches a library collective."""

    def __init__(self, comm: TorchComm, ctx):
        super().__init__(ctx, comm.rank, comm.size)
        self.comm = comm

    def _grow(self, slot_bytes: int):
        self.ctx.sync()
        self.comm.barrier()  # nobody may still be writing into a mailbox that is about to go away
        if self.handle is not None:  # growing: every rank unmaps its imports before any exporter frees
            self.ctx.lib.csg_peer_disconnect(self.ctx.handle, self.handle)
            self.comm.barrier()
        mine = self._create(int(slot_bytes * 1.25))
        handles = self.comm.allgather_object(mine)
        ok = all(h != bytes(64) for h in handles)
        if ok:
            try:
                self.connect_ipc(handles)
            except Exception:  # e.g. no peer access between two of the GPUs
                ok = False
        # the decision is collective: either every rank talks through mailboxes or none does
        if not all(self.comm.allgather_object(ok)):
            self.close()  # two-phase: some ranks may have mapped this mailbox already
            raise RuntimeError("CUDA IPC / peer access is unavailable on at least one rank")
        self.comm.barrier()


    def close(self):
        """Collective teardown (every rank calls it): unmap the other ranks' mailboxes, meet, and only then
        free the own one -- an exporter must not free memory an importer still has mapped.  ``destroy()`` /
        ``__del__`` alone are only safe once every peer process has closed or exited."""
        if self.handle is None:
            return
        self.ctx.sync()
        self.ctx.lib.csg_peer_disconnect(self.ctx.handle, self.handle)
        self.comm.barrier()
        self.destroy()


class SharedPeerGroup:
    """Several ranks living in ONE process (one context / stream each): mailboxes wired by raw
    device pointers.  Used by the single-GPU tests to run the multi-rank selection for real."""

    def __init__(self, contexts):
        self.members = [_SharedPeer(self, ctx, r, len(contexts)) for r, ctx in enumerate(contexts)]
        self.slot_bytes = 0

    def grow(self, slot_bytes: int):
        if self.slot_bytes >= slot_bytes:
            return
        for m in self.members:
            m.ctx.sync()
        for m in self.members:
            m._create(slot_bytes)
        boxes = [m.mailbox() for m in self.members]
        for m in self.members:
            m.connect_ptrs(boxes)
        self.slot_bytes = slot_bytes


class _SharedPeer(PeerExchange):
    def __init__(self, group, ctx, rank, size):
        super().__init__(ctx, rank, size)
        self.group = group

    def ensure(self, slot_bytes: int):
        self.group.grow(slot_bytes)


def make_exchange(comm, ctx):
    """The exchange a selection on ``ctx`` uses: peer mailboxes over NVLink by default,
    ``CSG_EXCHANGE=nccl`` selects the library collectives (A/B measurements)."""
    import os

    if comm is None or getattr(comm, "size", 1) == 1:
        return LocalExchange()
    if not hasattr(comm, "allgather_dev"):
        raise TypeError("multi-rank selection needs a TorchComm (device collectives)")
    if os.environ.get("CSG_EXCHANGE", "peer").lower() == "nccl" or comm.device.type != "cuda":
        return NcclExchange(comm, ctx)
    return IpcPeerExchange(comm, ctx)
