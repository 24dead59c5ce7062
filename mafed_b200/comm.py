"""Peer-memory communicator for the batch-sharded step (one process per GPU, one NVLink box).

`torch.distributed` is only the plumbing here: it carries the 64-byte CUDA IPC handles once, at set-up.
After that the per-step exchanges (<= 2L+2 doubles) happen inside the path's own kernels with NVLink peer stores
of self-validating words (``csrc/distill_comm.cuh``): the token counts leave when the batch is drawn
(``prefetch_counts``), the sums are exchanged by the fused kernel's last CTA -- no NCCL call and no extra launch on
the step's critical path.  If the ranks are not on one host, or a mailbox cannot be mapped, every rank falls back to
the NCCL allreduce together.
"""
from __future__ import annotations

import ctypes
import os
import socket
from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import cabi

_cache: Dict[tuple, Optional["PeerComm"]] = {}
# Bumped whenever the communicators are torn down: a compiled step reads it (Dynamo guards on its value), so a graph
# traced against a communicator is retraced instead of replaying a stale handle.
_generation = 0


class PeerComm:
    def __init__(self, handle: ctypes.c_void_p, world: int, rank: int):
        self.handle, self.world, self.rank = handle, world, rank

    def status(self) -> int:
        """0 = ok, 1 = a peer did not arrive within the spin bound.  A plain read of a word in mapped pinned host
        memory (no synchronisation): it reflects every exchange of the kernels that have finished."""
        out = ctypes.c_int(0)
        cabi.check(cabi.load().mafed_comm_status(self.handle, ctypes.byref(out)), "mafed_comm_status")
        return out.value

    def set_timeout(self, seconds: float):
        """Spin bound of one in-kernel wait (default 60 s, ``MAFED_B200_COMM_TIMEOUT_S``)."""
        cabi.check(cabi.load().mafed_comm_set_timeout(self.handle, float(seconds)), "mafed_comm_set_timeout")

    def check(self):
        """Raise if a peer did not arrive within the spin bound in any exchange so far (the losses and gradients
        of that step are NaN).  Does not synchronise: it sees the kernels that have finished; synchronise the stream
        first for a verdict on the steps still queued."""
        if self.status() != 0:
            raise cabi.MafedDistillError(
                f"rank {self.rank}: a peer did not reach a distillation exchange within the spin bound "
                "(MAFED_B200_COMM_TIMEOUT_S); the results of that step are NaN")

    def trace(self):
        """SM-cycle totals ``[counts exchange, publish, wait for peers, sums exchanges]`` (synchronises the device)."""
        out = (ctypes.c_ulonglong * 4)()
        cabi.check(cabi.load().mafed_comm_trace(self.handle, out), "mafed_comm_trace")
        return list(out)

    def trace_into(self, out4: torch.Tensor):
        """The same four totals as a stream-ordered snapshot: an asynchronous copy into ``out4`` (a pinned or device
        uint64/int64 tensor of 4 elements) behind the work queued on the current stream; no synchronisation."""
        assert out4.numel() >= 4 and out4.element_size() == 8 and out4.is_contiguous()
        cabi.check(cabi.load().mafed_comm_trace_async(self.handle, out4.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream), "mafed_comm_trace_async")

    def close(self):
        if self.handle:
            cabi.load().mafed_comm_destroy(self.handle)
            self.handle = None


def _build(group) -> Optional[PeerComm]:
    lib = cabi.load()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if world > 16:
        return None
    n = lib.mafed_comm_handle_bytes()
    buf = ctypes.create_string_buffer(n)
    handle = ctypes.c_void_p()
    ok = lib.mafed_comm_create(world, rank, buf, ctypes.byref(handle)) == 0
    infos = [None] * world
    dist.all_gather_object(infos, (socket.gethostname(), bytes(buf.raw) if ok else None), group=group)
    same_host = len({h for h, _ in infos}) == 1
    if ok and same_host and all(b is not None for _, b in infos):
        ok = lib.mafed_comm_connect(handle, b"".join(b for _, b in infos)) == 0
    else:
        ok = False
    flags = [None] * world
    dist.all_gather_object(flags, bool(ok), group=group)   # also a barrier: every mailbox is zeroed and mapped
    if not all(flags):
        if handle:
            lib.mafed_comm_destroy(handle)
        return None
    return PeerComm(handle, world, rank)


def get_peer_comm(group=None) -> Optional[PeerComm]:
    """The communicator of `group` (default group if None) on the current device; None -> use NCCL."""
    if os.environ.get("MAFED_B200_DIST", "peer").lower() == "nccl":
        return None
    key = (id(group) if group is not None else 0, torch.cuda.current_device())
    if key not in _cache:
        _cache[key] = _build(group)
    return _cache[key]


def peek_peer_comm(group=None) -> Optional[PeerComm]:
    """The communicator of `group` if one has been built already (never builds one: not a collective call)."""
    return _cache.get((id(group) if group is not None else 0, torch.cuda.current_device()))


def reset():
    global _generation
    _generation += 1
    for c in _cache.values():
        if c is not None:
            c.close()
    _cache.clear()
