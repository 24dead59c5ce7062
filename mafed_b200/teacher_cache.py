"""Per-task cache of the frozen teacher's hidden states over the episodic memory (``FeatureDistillation(teacher_cache=True)``).

The teacher (``past_model``) and the memory are both fixed for a task, and every replay step draws its batch from that
memory, so the teacher forward of a replay step recomputes hidden states it has computed before.  ``build`` runs the
teacher once per task over the whole memory and keeps, per distilled layer, one ``[M, T_c, D]`` tensor; a replay step
then gathers its samples' rows from it (``TeacherCache.gather``: one launch of ``libmafed_teacher_gather.so`` per dtype
of the cached layers, ``include/mafed_teacher_gather.h``) instead of running the teacher -- or, where the one-pass step
takes the shape, has the step's kernels read the rows straight from the cache (``TeacherCache.step_inputs``,
``libmafed_cached_step.so``, ``include/mafed_cached_step.h``), with no gathered copy at all.

Layout: ``T_c = n_vis + the longest text of the memory set``; every sample is computed with its text left-padded to
that length, as the collate pads a batch.  A batch at length ``T <= T_c`` takes the visual rows ``t < n_vis`` from the
start of its samples' cache rows and the text rows from their right-aligned end.

Sharded (``shard_teacher_cache=True``, one process per GPU of one box): ``build_sharded`` runs only this rank's share of
the same build batches into one device buffer per rank (``ShardedTeacherCache``), maps every peer's buffer through CUDA
IPC, and a step's gather reads each sample's rows from whichever GPU holds them, in the same single launch per dtype.
Build batch ``k`` (the ``k``-th batch of ``batch_size`` samples of the memory, in order) belongs to rank ``k % N``
(``shard_owners``), so every row is computed by the same batch as in ``build`` and is bit for bit the replicated row.

Sample identity: the memory loader yields ``batch["memory_index"]``, a Python list of the samples' indices into the
memory ``ConcatDataset`` (``IndexedDataset`` + ``IndexedCollate``); a list is left on the host by the prefetch loader,
so a step never reads a device tensor back.
"""
from __future__ import annotations

import ctypes
import logging
import os
import socket
import threading
from typing import Dict, List, Sequence, Tuple

import torch

from mafed_b200.cabi import MafedDistillError

_log = logging.getLogger(__name__)

ABI_VERSION = 2
MAX_RANKS = 16
_ALIGN = 256                    # byte alignment of each layer's block in a shard
_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib", "libmafed_teacher_gather.so")

_lib = None
_lock = threading.Lock()


def load():
    """Load libmafed_teacher_gather.so (built in-tree by ``mafed_b200.build``); raise if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise MafedDistillError(f"{LIB_PATH} not found: build it with `python -m mafed_b200.build` "
                                        "(the teacher cache has no eager fallback)")
            lib = ctypes.CDLL(LIB_PATH)
            lib.mafed_teacher_gather_abi_version.restype = ctypes.c_int
            lib.mafed_teacher_gather_error_string.restype = ctypes.c_char_p
            lib.mafed_teacher_gather_error_string.argtypes = [ctypes.c_int]
            lib.mafed_teacher_gather.restype = ctypes.c_int
            i32 = ctypes.c_int
            lib.mafed_teacher_gather.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                                 ctypes.POINTER(ctypes.c_int64), i32, i32, ctypes.c_int64, i32, i32,
                                                 i32, i32, i32, ctypes.c_void_p]
            vp, i64 = ctypes.c_void_p, ctypes.c_int64
            lib.mafed_teacher_gather_sharded.restype = i32
            lib.mafed_teacher_gather_sharded.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(vp), i32,
                                                         ctypes.POINTER(i64), ctypes.POINTER(ctypes.c_int32),
                                                         ctypes.POINTER(i64), i32, i32, i64, i32, i32, i32, i32, i32, vp]
            lib.mafed_teacher_shard_handle_bytes.restype = i32
            lib.mafed_teacher_shard_create.restype = i32
            lib.mafed_teacher_shard_create.argtypes = [i32, i32, i64, ctypes.c_char_p, ctypes.POINTER(vp)]
            lib.mafed_teacher_shard_connect.restype = i32
            lib.mafed_teacher_shard_connect.argtypes = [vp, ctypes.c_char_p]
            lib.mafed_teacher_shard_base.restype = i32
            lib.mafed_teacher_shard_base.argtypes = [vp, i32, ctypes.POINTER(vp)]
            lib.mafed_teacher_shard_destroy.restype = i32
            lib.mafed_teacher_shard_destroy.argtypes = [vp]
            if lib.mafed_teacher_gather_abi_version() != ABI_VERSION:
                raise MafedDistillError("libmafed_teacher_gather.so ABI version mismatch; rebuild")
            _lib = lib
    return _lib


def _check(rc, what):
    if rc != 0:
        raise MafedDistillError(f"{what} failed: {load().mafed_teacher_gather_error_string(rc).decode()} (code {rc})")


def gather_raw(out_ptrs, cache_ptrs, idx, B, M, T, T_c, n_vis, D, dtype_code, stream):
    """``mafed_teacher_gather`` as it is (plain ints and pointers); raise ``MafedDistillError`` on a non-zero code."""
    lib = load()
    n = len(out_ptrs)
    rc = lib.mafed_teacher_gather((ctypes.c_void_p * n)(*out_ptrs), (ctypes.c_void_p * len(cache_ptrs))(*cache_ptrs),
                                  (ctypes.c_int64 * len(idx))(*idx) if idx is not None else None, n, B, M, T, T_c,
                                  n_vis, D, dtype_code, stream)
    _check(rc, "mafed_teacher_gather")


def _array(ctype, values):
    return (ctype * len(values))(*values) if values is not None else None


def gather_sharded_raw(out_ptrs, bases, layer_off, src_rank, slot, B, slots, T, T_c, n_vis, D, dtype_code, stream):
    """``mafed_teacher_gather_sharded`` as it is (plain ints and pointers; ``None`` passes NULL); raise
    ``MafedDistillError`` on a non-zero code."""
    lib = load()
    rc = lib.mafed_teacher_gather_sharded(
        _array(ctypes.c_void_p, out_ptrs), _array(ctypes.c_void_p, bases), len(bases) if bases is not None else 0,
        _array(ctypes.c_int64, layer_off), _array(ctypes.c_int32, src_rank), _array(ctypes.c_int64, slot),
        len(out_ptrs if out_ptrs is not None else layer_off), B, slots, T, T_c, n_vis, D, dtype_code, stream)
    _check(rc, "mafed_teacher_gather_sharded")


def _checked(idx: Sequence[int], T: int, M: int, T_c: int, n_vis: int) -> List[int]:
    """The memory indices of a step as ints, after the range and length checks every read of the cache makes."""
    idx = [int(i) for i in idx]
    bad = [i for i in idx if not 0 <= i < M]
    if bad:
        raise MafedDistillError(f"memory index {bad[0]} out of range for a teacher cache of {M} samples")
    if not n_vis <= T <= T_c:
        raise MafedDistillError(f"a batch of {T} tokens does not fit the teacher cache (n_vis = {n_vis}, T_c = {T_c}): "
                                "the memory set changed since the cache was built")
    return idx


def gather(cache: Sequence[torch.Tensor], idx: Sequence[int], T: int, n_vis: int) -> List[torch.Tensor]:
    """``[B, T, D]`` teacher states of the memory samples ``idx`` from ``[M, T_c, D]`` cache tensors (one kernel launch
    per dtype among them), stream-ordered on the current stream."""
    M, T_c, D = cache[0].shape
    idx = _checked(idx, T, M, T_c, n_vis)
    out = [torch.empty((len(idx), T, D), dtype=c.dtype, device=c.device) for c in cache]
    stream = torch.cuda.current_stream(cache[0].device).cuda_stream
    for dtype in dict.fromkeys(c.dtype for c in cache):
        pick = [i for i, c in enumerate(cache) if c.dtype == dtype]
        gather_raw([out[i].data_ptr() for i in pick], [cache[i].data_ptr() for i in pick], idx, len(idx), M, T, T_c,
                   n_vis, D, _DTYPES[dtype], stream)
    return out


def reference_gather(cache: Sequence[torch.Tensor], idx: Sequence[int], T: int, n_vis: int) -> List[torch.Tensor]:
    """Torch restatement of ``gather`` (index_select + the two row blocks); an index ``>= M`` gives NaN rows, as the
    kernel writes them."""
    out = []
    for c in cache:
        M, T_c, D = c.shape
        rows = torch.cat([torch.arange(n_vis), torch.arange(n_vis, T) + (T_c - T)]).to(c.device)
        ix = torch.as_tensor(list(idx), dtype=torch.int64, device=c.device)
        valid = (ix >= 0) & (ix < M)
        g = c.index_select(0, torch.where(valid, ix, 0)).index_select(1, rows)
        out.append(torch.where(valid[:, None, None], g, torch.full_like(g, float("nan"))))
    return out


class IndexedDataset(torch.utils.data.Dataset):
    """A dataset whose item ``i`` is ``(i, dataset[i])``: the memory index travels with the sample."""

    def __init__(self, dataset):
        self.dataset = dataset

    def __len__(self):
        return len(self.dataset)

    def __getitem__(self, i):
        return i, self.dataset[i]


class IndexedCollate:
    """The memory collate over ``IndexedDataset`` items; adds ``batch["memory_index"]`` (a list of ints)."""

    def __init__(self, collate=None):
        self.collate = collate if collate is not None else torch.utils.data.default_collate

    def __call__(self, items):
        batch = self.collate([item for _, item in items])
        batch["memory_index"] = [int(i) for i, _ in items]
        return batch


def repad_left(batch: Dict[str, object], text_len: int) -> Dict[str, object]:
    """``input_ids`` / ``attention_mask`` padded on the left to ``text_len`` tokens, as the collate pads (mask 0; the id
    the collate put under a 0 of the mask, else 0)."""
    ids, am = batch["input_ids"], batch["attention_mask"]
    pad = text_len - ids.shape[1]
    if pad < 0:
        raise ValueError(f"a batch of {ids.shape[1]} text tokens cannot be padded to {text_len}")
    if pad == 0:
        return batch
    under = ids[am == 0]
    pad_id = int(under[0]) if under.numel() else 0
    out = dict(batch)
    out["input_ids"] = torch.cat([ids.new_full((ids.shape[0], pad), pad_id), ids], dim=1)
    out["attention_mask"] = torch.cat([am.new_zeros((am.shape[0], pad)), am], dim=1)
    return out


class TeacherCache:
    """The teacher states of every memory sample for the distilled ``layers``: ``states[k]`` is ``[M, T_c, D]``."""

    def __init__(self, layers: List[int], states: List[torch.Tensor], T_c: int, n_vis: int):
        self.layers, self.states, self.T_c, self.n_vis = list(layers), states, T_c, n_vis

    @property
    def nbytes(self) -> int:
        return sum(s.numel() * s.element_size() for s in self.states)

    def gather(self, idx: Sequence[int], T: int, layers: Sequence[int]) -> List[torch.Tensor]:
        if list(layers) != self.layers:
            raise MafedDistillError(f"the teacher cache holds layers {self.layers}, the step distils {list(layers)}")
        return gather(self.states, idx, T, self.n_vis)

    def step_inputs(self, idx: Sequence[int], T: int, layers: Sequence[int]):
        """What a step that reads the teacher rows straight from the cache needs instead of ``gather``'s tensors:
        ``(states, idx, T, T_c)`` with ``idx`` checked as ``gather`` checks it (``distill_op.cached_distill_loss``)."""
        if list(layers) != self.layers:
            raise MafedDistillError(f"the teacher cache holds layers {self.layers}, the step distils {list(layers)}")
        return self.states, _checked(idx, T, self.states[0].shape[0], self.T_c, self.n_vis), T, self.T_c


def _build_batches(strategy):
    """The build batches: the memory ``ConcatDataset`` in order, in batches of ``strategy.batch_size`` (host inputs,
    each with its ``memory_index``), the longest text of the whole memory, and M."""
    from torch.utils.data import ConcatDataset, DataLoader

    memory = ConcatDataset(strategy.datasets)
    collate, _ = strategy._data_hooks()
    loader = DataLoader(IndexedDataset(memory), batch_size=strategy.batch_size, shuffle=False, num_workers=0,
                        collate_fn=IndexedCollate(collate))
    batches = list(loader)                   # host inputs, kept: for ~500 samples a few hundred MB
    return batches, max(b["input_ids"].shape[1] for b in batches), len(memory)


def _teacher_states(strategy, batch, text_len, layers, device):
    """One build batch through the teacher at ``text_len`` text tokens: ``(memory indices, [B, T_c, D] per layer)``."""
    from mafed_b200.capture import HiddenStateCapture

    model = strategy.past_model
    idx = batch.pop("memory_index")
    batch.pop("labels", None)
    batch = {k: v.to(device, non_blocking=True) if torch.is_tensor(v) else v
             for k, v in repad_left(batch, text_len).items()}
    with torch.no_grad(), torch.autocast(device.type, dtype=torch.bfloat16), strategy._teacher_forward(batch):
        with HiddenStateCapture(model, layers, detach=True, stop_after_last=True) as cap:
            model(**batch, output_hidden_states=False, return_dict=True)
    return idx, [strategy._as_teacher_dtype(cap.hidden_states[l]) for l in layers]


def build(strategy) -> TeacherCache:
    """Run ``strategy.past_model`` once over the whole episodic memory (``strategy.datasets``) and cache its distilled
    hidden states, as ``replay()`` would hand them to the step: the same bf16 autocast region, ``teacher_dtype``
    autocast and rounding, and a forward that stops after the last distilled entry."""
    batches, text_len, M = _build_batches(strategy)
    n_vis = strategy.num_vision_tokens
    T_c = n_vis + text_len
    layers = strategy.loss_weights.get_distillation_layers()
    device = next(strategy.past_model.parameters()).device
    states = None
    for batch in batches:
        idx, hs = _teacher_states(strategy, batch, text_len, layers, device)
        if states is None:
            need = sum(M * T_c * h.shape[-1] * h.element_size() for h in hs)
            _log.info("teacher cache: %d samples x %d layers x T_c %d x D %d = %d bytes", M, len(layers), T_c,
                      hs[0].shape[-1], need)
            try:
                states = [torch.empty((M, T_c, h.shape[-1]), dtype=h.dtype, device=device) for h in hs]
            except torch.OutOfMemoryError as exc:
                raise torch.OutOfMemoryError(
                    f"the teacher cache needs {need} bytes ({M} memory samples x {len(layers)} layers x T_c {T_c} x "
                    f"D {hs[0].shape[-1]}): {exc}") from exc
        rows = torch.as_tensor(idx, dtype=torch.int64, device=device)
        for s, h in zip(states, hs):
            s.index_copy_(0, rows, h)
    return TeacherCache(layers, states, T_c, n_vis)


# ---------------------------------------------------------------- the cache sharded across the ranks of one box
def shard_owners(M: int, batch_size: int, world: int) -> Tuple[List[int], List[int], List[int]]:
    """Where each memory sample lives in a sharded cache: ``(rank[i], slot[i], count[r])``.  Build batch
    ``k = i // batch_size`` belongs to rank ``k % world``; a rank's batches fill its slots in order, so sample ``i``
    takes slot ``(k // world) * batch_size + i % batch_size``.  A pure function of its arguments: every rank computes
    it with no exchange.  A rank with no build batch (fewer batches than ranks) holds no sample."""
    if M < 0 or batch_size < 1 or world < 1:
        raise ValueError(f"shard_owners needs M >= 0, batch_size >= 1 and world >= 1, not {M}, {batch_size}, {world}")
    rank = [(i // batch_size) % world for i in range(M)]
    slot = [(i // batch_size // world) * batch_size + i % batch_size for i in range(M)]
    count = [0] * world
    for r in rank:
        count[r] += 1
    return rank, slot, count


def shard_layout(capacity: int, T_c: int, D: int, element_sizes: Sequence[int]) -> Tuple[List[int], int]:
    """Byte offset of each layer's ``[capacity, T_c, D]`` block in a shard (each 256-byte aligned) and the shard's
    size.  The same on every rank: every rank allocates the largest share."""
    offsets, at = [], 0
    for e in element_sizes:
        offsets.append(at)
        at += -(-capacity * T_c * D * e // _ALIGN) * _ALIGN
    return offsets, max(at, _ALIGN)


class _DeviceMemory:
    """A raw device range as a torch tensor (``__cuda_array_interface__``); the memory stays the shard's."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class ShardedTeacherCache:
    """This rank's share of the teacher cache, with every peer's share mapped (``build_sharded``).  Same surface as
    ``TeacherCache``: ``layers``, ``T_c``, ``n_vis`` and ``gather``, which reads each sample's rows from the GPU that
    holds them (one launch per dtype of the layers).  ``local_states[k]`` is ``[count, T_c, D]``: this rank's samples
    (``owner``/``slot`` map memory indices to ranks and slots).  ``nbytes`` is this rank's shard.  ``release()`` is a
    collective of the group the cache was built over."""

    def __init__(self, layers, dtypes, T_c, n_vis, M, D, owner, slot, count, capacity, offsets, nbytes, handle, group,
                 rank, device):
        self.layers, self.dtypes, self.T_c, self.n_vis, self.M, self.D = list(layers), list(dtypes), T_c, n_vis, M, D
        self.owner, self.slot, self.count, self.capacity = owner, slot, count, capacity
        self.offsets, self.nbytes, self.group, self.rank, self.device = offsets, nbytes, group, rank, device
        self._handle = handle
        lib = load()
        self.bases = []
        for r in range(len(count)):
            base = ctypes.c_void_p()
            _check(lib.mafed_teacher_shard_base(handle, r, ctypes.byref(base)), "mafed_teacher_shard_base")
            self.bases.append(base.value)
        raw = torch.as_tensor(_DeviceMemory(self.bases[rank], nbytes), device=device)
        self._slots = [raw[o:o + capacity * T_c * D * torch.empty((), dtype=d).element_size()].view(d)
                       .view(capacity, T_c, D) for o, d in zip(offsets, self.dtypes)]
        self.local_states = [s[: count[rank]] for s in self._slots]

    def gather(self, idx: Sequence[int], T: int, layers: Sequence[int]) -> List[torch.Tensor]:
        if list(layers) != self.layers:
            raise MafedDistillError(f"the teacher cache holds layers {self.layers}, the step distils {list(layers)}")
        if self._handle is None:
            raise MafedDistillError("the sharded teacher cache has been released")
        idx = [int(i) for i in idx]
        bad = [i for i in idx if not 0 <= i < self.M]
        if bad:
            raise MafedDistillError(f"memory index {bad[0]} out of range for a teacher cache of {self.M} samples")
        if not self.n_vis <= T <= self.T_c:
            raise MafedDistillError(f"a batch of {T} tokens does not fit the teacher cache (n_vis = {self.n_vis}, "
                                    f"T_c = {self.T_c}): the memory set changed since the cache was built")
        out = [torch.empty((len(idx), T, self.D), dtype=d, device=self.device) for d in self.dtypes]
        ranks, slots = [self.owner[i] for i in idx], [self.slot[i] for i in idx]
        stream = torch.cuda.current_stream(self.device).cuda_stream
        for dtype in dict.fromkeys(self.dtypes):
            pick = [k for k, d in enumerate(self.dtypes) if d == dtype]
            gather_sharded_raw([out[k].data_ptr() for k in pick], self.bases, [self.offsets[k] for k in pick], ranks,
                               slots, len(idx), self.capacity, T, self.T_c, self.n_vis, self.D, _DTYPES[dtype], stream)
        return out

    def release(self):
        """Free the shards, collectively over the cache's group: wait for this device's work and for every rank
        (a peer may still be gathering from this shard), then unmap the peers' shards and free this one."""
        if self._handle is None:
            return
        torch.cuda.synchronize(self.device)
        torch.distributed.barrier(group=self.group)
        self.local_states, self._slots = [], []
        load().mafed_teacher_shard_destroy(self._handle)
        self._handle = None


def build_sharded(strategy, group=None) -> ShardedTeacherCache:
    """``build`` split across the ranks of ``group`` (the default group if None), one process per GPU of one host:
    rank ``r`` runs the build batches ``k % N == r`` (the same inputs at the same ``T_c`` as ``build``) into its own
    shard, and maps every peer's shard through CUDA IPC.  Collective: every rank of the group calls it."""
    dist = torch.distributed
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if world > MAX_RANKS:
        raise MafedDistillError(f"a sharded teacher cache spans at most {MAX_RANKS} ranks, the group has {world}")
    lib = load()
    batches, text_len, M = _build_batches(strategy)
    n_vis = strategy.num_vision_tokens
    T_c = n_vis + text_len
    layers = strategy.loss_weights.get_distillation_layers()
    device = next(strategy.past_model.parameters()).device
    owner, slot, count = shard_owners(M, strategy.batch_size, world)
    mine = batches[rank::world]
    # this rank's first batch gives the layers' width and dtypes (rank 0 always has one)
    first = _teacher_states(strategy, mine[0], text_len, layers, device) if mine else None
    spec = None if first is None else (first[1][0].shape[-1], [str(h.dtype) for h in first[1]])
    every = [None] * world
    dist.all_gather_object(every, (socket.gethostname(), spec), group=group)
    hosts = sorted({h for h, _ in every})
    if len(hosts) != 1:
        raise MafedDistillError(f"shard_teacher_cache needs every rank of the group on one host (CUDA IPC over "
                                f"NVLink); the ranks run on {hosts}")
    D, names = every[0][1]
    if any(sp is not None and sp != every[0][1] for _, sp in every):
        raise MafedDistillError(f"the ranks' teachers give different hidden-state widths or dtypes: {[sp for _, sp in every]}")
    dtypes = [getattr(torch, n.split(".")[-1]) for n in names]
    capacity = max(count)
    offsets, nbytes = shard_layout(capacity, T_c, D, [torch.empty((), dtype=d).element_size() for d in dtypes])
    _log.info("sharded teacher cache: rank %d/%d holds %d of %d samples (capacity %d) x %d layers x T_c %d x D %d = "
              "%d bytes", rank, world, count[rank], M, capacity, len(layers), T_c, D, nbytes)

    handle = ctypes.c_void_p()
    hbytes = ctypes.create_string_buffer(lib.mafed_teacher_shard_handle_bytes())
    rc = lib.mafed_teacher_shard_create(world, rank, nbytes, hbytes, ctypes.byref(handle))
    every = [None] * world
    dist.all_gather_object(every, (rc, hbytes.raw), group=group)
    if any(r != 0 for r, _ in every):
        lib.mafed_teacher_shard_destroy(handle)
        failed = [r for r, (c, _) in enumerate(every) if c != 0]
        raise MafedDistillError(f"rank(s) {failed} could not allocate a teacher-cache shard of {nbytes} bytes "
                                f"({capacity} samples x {len(layers)} layers x T_c {T_c} x D {D}): "
                                f"{lib.mafed_teacher_gather_error_string(every[failed[0]][0]).decode()}")
    rc = lib.mafed_teacher_shard_connect(handle, b"".join(h for _, h in every))
    flags = [None] * world
    dist.all_gather_object(flags, rc, group=group)
    if any(flags):
        lib.mafed_teacher_shard_destroy(handle)
        raise MafedDistillError(f"rank(s) {[r for r, c in enumerate(flags) if c]} could not map the peers' teacher-cache "
                                "shards")
    cache = ShardedTeacherCache(layers, dtypes, T_c, n_vis, M, D, owner, slot, count, capacity, offsets, nbytes,
                                handle, group, rank, device)
    for k, batch in enumerate(mine):
        idx, hs = first if k == 0 else _teacher_states(strategy, batch, text_len, layers, device)
        lo = slot[idx[0]]
        for s, h in zip(cache._slots, hs):
            s[lo:lo + len(idx)].copy_(h)
    first = None
    # every row is written before any peer reads it
    torch.cuda.synchronize(device)
    dist.barrier(group=group)
    every = [None] * world
    mine_spec = (M, T_c, layers, D, names)
    dist.all_gather_object(every, mine_spec, group=group)
    if any(e != mine_spec for e in every):
        cache.release()
        raise MafedDistillError(f"the ranks' teacher caches differ in (M, T_c, layers, D, dtypes): {every}")
    return cache
