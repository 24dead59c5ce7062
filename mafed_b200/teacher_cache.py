"""Per-task cache of the frozen teacher's hidden states over the episodic memory (``FeatureDistillation(teacher_cache=True)``).

The teacher (``past_model``) and the memory are both fixed for a task, and every replay step draws its batch from that
memory, so the teacher forward of a replay step recomputes hidden states it has computed before.  ``build`` runs the
teacher once per task over the whole memory and keeps, per distilled layer, one ``[M, T_c, D]`` tensor; a replay step
then gathers its samples' rows from it (``TeacherCache.gather``: one launch of ``libmafed_teacher_gather.so`` per dtype
of the cached layers, ``include/mafed_teacher_gather.h``) instead of running the teacher.

Layout: ``T_c = n_vis + the longest text of the memory set``; every sample is computed with its text left-padded to
that length, as the collate pads a batch.  A batch at length ``T <= T_c`` takes the visual rows ``t < n_vis`` from the
start of its samples' cache rows and the text rows from their right-aligned end.

Sample identity: the memory loader yields ``batch["memory_index"]``, a Python list of the samples' indices into the
memory ``ConcatDataset`` (``IndexedDataset`` + ``IndexedCollate``); a list is left on the host by the prefetch loader,
so a step never reads a device tensor back.
"""
from __future__ import annotations

import ctypes
import logging
import os
import threading
from typing import Dict, List, Sequence

import torch

from mafed_b200.cabi import MafedDistillError

_log = logging.getLogger(__name__)

ABI_VERSION = 1
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
            if lib.mafed_teacher_gather_abi_version() != ABI_VERSION:
                raise MafedDistillError("libmafed_teacher_gather.so ABI version mismatch; rebuild")
            _lib = lib
    return _lib


def gather_raw(out_ptrs, cache_ptrs, idx, B, M, T, T_c, n_vis, D, dtype_code, stream):
    """``mafed_teacher_gather`` as it is (plain ints and pointers); raise ``MafedDistillError`` on a non-zero code."""
    lib = load()
    n = len(out_ptrs)
    rc = lib.mafed_teacher_gather((ctypes.c_void_p * n)(*out_ptrs), (ctypes.c_void_p * len(cache_ptrs))(*cache_ptrs),
                                  (ctypes.c_int64 * len(idx))(*idx) if idx is not None else None, n, B, M, T, T_c,
                                  n_vis, D, dtype_code, stream)
    if rc != 0:
        raise MafedDistillError(f"mafed_teacher_gather failed: {lib.mafed_teacher_gather_error_string(rc).decode()} "
                                f"(code {rc})")


def gather(cache: Sequence[torch.Tensor], idx: Sequence[int], T: int, n_vis: int) -> List[torch.Tensor]:
    """``[B, T, D]`` teacher states of the memory samples ``idx`` from ``[M, T_c, D]`` cache tensors (one kernel launch
    per dtype among them), stream-ordered on the current stream."""
    M, T_c, D = cache[0].shape
    idx = [int(i) for i in idx]
    bad = [i for i in idx if not 0 <= i < M]
    if bad:
        raise MafedDistillError(f"memory index {bad[0]} out of range for a teacher cache of {M} samples")
    if not n_vis <= T <= T_c:
        raise MafedDistillError(f"a batch of {T} tokens does not fit the teacher cache (n_vis = {n_vis}, T_c = {T_c}): "
                                "the memory set changed since the cache was built")
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


def build(strategy) -> TeacherCache:
    """Run ``strategy.past_model`` once over the whole episodic memory (``strategy.datasets``) and cache its distilled
    hidden states, as ``replay()`` would hand them to the step: the same bf16 autocast region, ``teacher_dtype``
    autocast and rounding, and a forward that stops after the last distilled entry."""
    from torch.utils.data import ConcatDataset, DataLoader

    from mafed_b200.capture import HiddenStateCapture

    memory = ConcatDataset(strategy.datasets)
    collate, _ = strategy._data_hooks()
    loader = DataLoader(IndexedDataset(memory), batch_size=strategy.batch_size, shuffle=False, num_workers=0,
                        collate_fn=IndexedCollate(collate))
    batches = list(loader)                   # host inputs, kept: for ~500 samples a few hundred MB
    n_vis = strategy.num_vision_tokens
    text_len = max(b["input_ids"].shape[1] for b in batches)
    T_c = n_vis + text_len
    layers = strategy.loss_weights.get_distillation_layers()
    model = strategy.past_model
    device = next(model.parameters()).device
    M = len(memory)
    states = None
    for batch in batches:
        idx = batch.pop("memory_index")
        batch.pop("labels", None)
        batch = {k: v.to(device, non_blocking=True) if torch.is_tensor(v) else v
                 for k, v in repad_left(batch, text_len).items()}
        with torch.no_grad(), torch.autocast(device.type, dtype=torch.bfloat16), strategy._teacher_forward(batch):
            with HiddenStateCapture(model, layers, detach=True, stop_after_last=True) as cap:
                model(**batch, output_hidden_states=False, return_dict=True)
        hs = [strategy._as_teacher_dtype(cap.hidden_states[l]) for l in layers]
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
