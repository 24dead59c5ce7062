"""The fused distillation operator: host tables -> C ABI -> sm_100a kernels, with autograd.

Two ways to run a step, same results:

* two-pass  -- fused forward over all selected layers (the loss algebra runs in the kernel's last CTA),
  later one fused backward: 5*D*e bytes of HBM traffic per token*layer, two launches;
* one-pass  -- the gradient scale depends only on the token counts and the host weight tables, not
  on the loss, so one kernel produces the loss sums AND the gradients from a single read of student
  and teacher (3*D*e bytes).  The upstream gradient is assumed (``plan.assumed_grad_out``, i.e.
  ``1 / accumulate_grad_batches`` under Lightning); ``backward`` launches a fix-up that returns at
  once when the real upstream gradient equals the assumed one and otherwise recomputes exactly.
  The whole step -- modality masks, scale table, loss sums, gradients, losses, and across batch
  shards the NVLink exchange of counts and sums -- is ONE kernel launch (``mafed_distill_step``).

Under ``torch.distributed`` with batch sharding, the per-rank ``[2L+2]`` fp64 partial sums / counts
are combined by allreduce; the backward needs no collective (SURVEY.md 8e).  Nothing here
synchronises the host with the device.

Host side: ``distill_loss`` hands the whole step to the compiled autograd node (``csrc/torch_node.cpp``,
``mafed_b200.node``) -- pointer tables, workspace and gradient allocation, stream lookup, the launch and the
backward gate all run in C++.  The ctypes functions below (``distill_forward`` / ``distill_fused`` /
``distill_backward``) are the same C-ABI calls one at a time: the NCCL sequence, the kernel-level benchmarks and
the tests use them.

Replaces the per-layer Python loop of ``mafed/methods/distillation.py:105-166`` and the autograd
chains behind ``:226-249``.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import torch

from . import cabi, node
from . import comm as _comm
from .comm import get_peer_comm

_DTYPES = {torch.float32: cabi.F32, torch.bfloat16: cabi.BF16, torch.float16: cabi.F16}
# (student, teacher) dtype pairs the kernels read as they are besides one dtype on both sides
_TEACHER_PAIRS = {(torch.float32, torch.bfloat16), (torch.float32, torch.float16)}


def _native_dtypes(students, teachers) -> bool:
    """True when the kernels take these layers without an up-cast: one dtype everywhere, or fp32 students with
    teachers of one half-precision dtype.  ``distill_loss`` splits a step into dtype groups first
    (``dtype_groups``), so a launch-sized step that fails this is the one group of pairs the kernels refuse (a
    half-precision student against an fp32 teacher, bf16 against fp16): that group alone is up-cast to fp32."""
    s_types, t_types = {t.dtype for t in students}, {t.dtype for t in teachers}
    if len(s_types) != 1 or len(t_types) != 1:
        return False
    pair = (next(iter(s_types)), next(iter(t_types)))
    return pair[0] == pair[1] or pair in _TEACHER_PAIRS


def dtype_groups(pairs: Sequence[tuple]) -> Optional[List[List[int]]]:
    """The layers of a step partitioned by their ``(student dtype, teacher dtype)`` pair, or ``None`` when one launch
    takes them all (every layer has the same pair).

    One group per pair the kernels read as it is (one dtype, or fp32 with bf16 / fp16), in the order of each pair's
    first layer; then, if any, one group of every layer whose pair the kernels refuse, which that step up-casts to
    fp32.  Layer order is kept inside each group.  A single group is ``None`` as well."""
    first = pairs[0]
    if all(p == first for p in pairs):
        return None
    native, refused = {}, []
    for i, p in enumerate(pairs):
        if p[0] == p[1] or p in _TEACHER_PAIRS:
            native.setdefault(p, []).append(i)
        else:
            refused.append(i)
    groups = list(native.values()) + ([refused] if refused else [])
    return groups if len(groups) > 1 else None


def sub_steps(n: int, groups: Optional[List[List[int]]]) -> Optional[List[List[int]]]:
    """The layer indices of each launch of a step over ``n`` layers: each dtype group (``dtype_groups``) cut into
    chunks of at most ``MAFED_MAX_LAYERS``.  ``None``: one launch over all of them."""
    if groups is None:
        if n <= cabi.MAX_LAYERS:
            return None
        groups = [list(range(n))]
    return [g[lo:lo + cabi.MAX_LAYERS] for g in groups for lo in range(0, len(g), cabi.MAX_LAYERS)]


def aux_runs(steps: List[List[int]]):
    """How to lay the sub-steps' ``aux`` vectors back out in the caller's layer order: ``(k, lo, hi)`` for each maximal
    run of caller positions that are layers ``lo:hi`` of sub-step ``k``, in caller order."""
    where = {}
    for k, idx in enumerate(steps):
        for j, i in enumerate(idx):
            where[i] = (k, j)
    runs = []
    for i in range(len(where)):
        k, j = where[i]
        if runs and runs[-1][0] == k and runs[-1][2] == j:
            runs[-1][2] = j + 1
        else:
            runs.append([k, j, j + 1])
    return [tuple(r) for r in runs]


@dataclass
class DistillPlan:
    """Host-side description of one distillation step (which layers, which weights)."""
    layers: List[int]                       # indices into the hidden-state tuple
    layer_coeffs: List[float]               # get_layer_loss_weight(layer) per selected layer
    distill_coeff: float = 1.0
    modality_kind: int = cabi.MODW_EQUAL
    lang_weights: Optional[List[float]] = None   # MODW_TABLE: language weight per selected layer
    loss_kind: int = cabi.LOSS_MSE
    cls: bool = False
    n_vis: int = 256
    grad_multiplier: float = 1.0            # e.g. world_size to undo DDP's gradient averaging
    single_pass: bool = True                # one-pass step when gradients are needed
    assumed_grad_out: float = 1.0           # upstream gradient the one-pass step bakes in
    _weights: Optional[cabi.Weights] = field(default=None, repr=False)
    _node_plan: object = field(default=None, repr=False)
    _splits: dict = field(default_factory=dict, repr=False)

    def split(self, pairs: tuple):
        """The launches of a step whose layers have these ``(student, teacher)`` dtype pairs: ``None`` for one
        launch over every layer, else ``(steps, runs)`` -- ``(layer indices, sub-plan)`` per launch, and
        ``aux_runs``.  Built once per dtype signature (a plan's host tables cost ~50 us of Python)."""
        if pairs not in self._splits:
            idx_lists = sub_steps(len(pairs), dtype_groups(pairs))
            if idx_lists is None:
                self._splits[pairs] = None
            else:
                steps = [(idx, self._sub_plan(idx)) for idx in idx_lists]
                self._splits[pairs] = (steps, aux_runs(idx_lists))
        return self._splits[pairs]

    def _sub_plan(self, idx: List[int]) -> "DistillPlan":
        return DistillPlan(layers=[self.layers[i] for i in idx], layer_coeffs=[self.layer_coeffs[i] for i in idx],
                           distill_coeff=self.distill_coeff, modality_kind=self.modality_kind,
                           lang_weights=None if self.lang_weights is None else [self.lang_weights[i] for i in idx],
                           loss_kind=self.loss_kind, cls=self.cls, n_vis=self.n_vis,
                           grad_multiplier=self.grad_multiplier, single_pass=self.single_pass,
                           assumed_grad_out=self.assumed_grad_out)

    def weights(self) -> cabi.Weights:
        if self._weights is None:
            if len(self.layers) > cabi.MAX_LAYERS:
                raise ValueError(f"at most {cabi.MAX_LAYERS} layers per call")
            self._weights = cabi.make_weights(
                cabi.MODW_CLS if self.cls else self.modality_kind, self.distill_coeff,
                self.layer_coeffs, self.lang_weights)
        return self._weights

    def node_plan(self):
        """The same tables as the compiled node's ``Plan`` (built once per DistillPlan)."""
        if self._node_plan is None:
            self._node_plan = node.load().Plan(
                cabi.MODW_CLS if self.cls else self.modality_kind, float(self.distill_coeff),
                [float(c) for c in self.layer_coeffs],
                None if self.lang_weights is None else [float(c) for c in self.lang_weights],
                self.loss_kind, bool(self.cls), int(self.n_vis), float(self.grad_multiplier), bool(self.single_pass),
                float(self.assumed_grad_out))
        return self._node_plan


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream_ptr(device) -> int:
    """cudaStream_t of torch's current stream on `device` (fast path avoids building a Stream object)."""
    if _raw_stream is not None and device.index is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


class _on_device:
    """`with torch.cuda.device(dev)` that costs nothing when `dev` is already current (the usual case)."""
    __slots__ = ("ctx",)

    def __init__(self, device):
        same = _raw_device is not None and device.index is not None and _raw_device() == device.index
        self.ctx = None if same else torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise cabi.MafedDistillError(
            f"{what} is on {t.device}: the distillation path runs only as sm_100a CUDA kernels "
            "(there is no CPU fallback)")


def _prepare(tensors: Sequence[torch.Tensor]):
    return [t if t.is_contiguous() else t.contiguous() for t in tensors]


class _DevicePtr:
    """A raw device address inside a torch allocation that it keeps alive (``.data_ptr()`` like a tensor)."""
    __slots__ = ("owner", "ptr")

    def __init__(self, owner, ptr):
        self.owner, self.ptr = owner, ptr

    def data_ptr(self):
        return self.ptr


class _Launch:
    """Geometry + pointer tables of one step; keeps the tensors alive until the kernels are queued."""

    def __init__(self, students, teachers, attn_mask, plan: DistillPlan):
        s0 = students[0]
        _require_cuda(s0, "hidden_states")
        if s0.dtype not in _DTYPES:
            raise TypeError(f"unsupported hidden-state dtype {s0.dtype} (float32, bfloat16, float16)")
        if s0.dim() != 3:
            raise ValueError("hidden states must be [B, T, D]")
        shape, dtype, device = s0.shape, s0.dtype, s0.device
        t_dtype = teachers[0].dtype
        if t_dtype != dtype and (dtype, t_dtype) not in _TEACHER_PAIRS:
            raise ValueError(f"student / teacher dtype mismatch ({dtype} / {t_dtype}): the kernels take one dtype, "
                             "or float32 students with bfloat16 or float16 teachers")
        self.B, self.T, self.D = shape
        for group, want in ((students, dtype), (teachers, t_dtype)):
            for t in group:
                if t.shape != shape:
                    raise ValueError("all selected hidden states must share one [B, T, D] shape")
                if t.dtype != want or t.device != device:
                    raise ValueError("student / teacher dtype or device mismatch")
        self.device = device
        self.dtype = dtype
        n_vis = plan.n_vis
        if plan.cls:
            self.mask = None
        else:
            if attn_mask is None:
                raise ValueError("attention_mask is required")
            _require_cuda(attn_mask, "attention_mask")
            if attn_mask.dtype != torch.int64:
                attn_mask = attn_mask.to(torch.int64)
            if attn_mask.shape != (self.B, self.T - n_vis):
                raise ValueError(
                    f"attention_mask shape {tuple(attn_mask.shape)} != (B, T - n_vis) = {(self.B, self.T - n_vis)}")
            self.mask = attn_mask.contiguous()
        self.n_layers = len(students)
        self.shape = cabi.make_shape(self.n_layers, self.B, self.T, n_vis if not plan.cls else min(n_vis, self.T),
                                     self.D, _DTYPES[self.dtype], plan.loss_kind, plan.cls, _DTYPES[t_dtype])
        self.shape_ref = ctypes.byref(self.shape)
        self.students = students
        self.teachers = teachers
        self.s_ptrs = cabi.ptr_array([t.data_ptr() for t in students])
        self.t_ptrs = cabi.ptr_array([t.data_ptr() for t in teachers])
        self.mask_ptr = self.mask.data_ptr() if self.mask is not None else None

    def alloc_scalars(self, lib):
        """(workspace, out, bwd_scale): the partial-sum workspace and the scale table share one scratch
        allocation; `bwd_scale` is returned as a `_DevicePtr` view that keeps the scratch alive."""
        L, dev = self.n_layers, self.device
        ws_bytes = (lib.mafed_distill_ws_bytes(L) + 255) & ~255
        scratch = torch.empty(ws_bytes + 8 * L, dtype=torch.uint8, device=dev)
        out = torch.empty(1 + 3 * L, dtype=torch.float32, device=dev)
        base = scratch.data_ptr()
        return _DevicePtr(scratch, base), out, _DevicePtr(scratch, base + ws_bytes)


def modality_masks(attn_mask: torch.Tensor, n_vis: int):
    """``[B, n_vis + txt]`` int64 language / image masks (``distillation.py:134-144``) in one launch."""
    lib = cabi.load()
    _require_cuda(attn_mask, "attention_mask")
    am = attn_mask if attn_mask.dtype == torch.int64 else attn_mask.to(torch.int64)
    am = am.contiguous()
    B, txt = am.shape
    both = torch.empty((2, B, n_vis + txt), dtype=torch.int64, device=am.device)
    shape = cabi.make_shape(1, B, n_vis + txt, n_vis, 1, cabi.F32, cabi.LOSS_MSE)
    with _on_device(am.device):
        cabi.check(lib.mafed_distill_modality_masks(ctypes.byref(shape), am.data_ptr(), both[0].data_ptr(),
                                                    both[1].data_ptr(), _stream_ptr(am.device)),
                   "mafed_distill_modality_masks")
    lang, image = both[0], both[1]
    if attn_mask.dtype != torch.int64:
        lang, image = lang.to(attn_mask.dtype), image.to(attn_mask.dtype)
    return lang, image


def modality_masks_into(attn_mask: torch.Tensor, n_vis: int, lang: torch.Tensor, image: torch.Tensor):
    """``modality_masks`` into pre-allocated int64 ``[B, n_vis + txt]`` outputs (``attn_mask`` int64, contiguous)."""
    lib = cabi.load()
    B, txt = attn_mask.shape
    shape = cabi.make_shape(1, B, n_vis + txt, n_vis, 1, cabi.F32, cabi.LOSS_MSE)
    with _on_device(attn_mask.device):
        cabi.check(lib.mafed_distill_modality_masks(ctypes.byref(shape), attn_mask.data_ptr(), lang.data_ptr(),
                                                    image.data_ptr(), _stream_ptr(attn_mask.device)),
                   "mafed_distill_modality_masks")


def token_norm_sums(tensors: Sequence[torch.Tensor], attn_mask: torch.Tensor, n_vis: int, group=False) -> torch.Tensor:
    """Masked per-modality sums of the per-token L2 norms of ``len(tensors)`` ``[B, T, D]`` tensors in one
    fused pass (``distillation_loss_weights.py:122-137``).  Returns device fp64 ``[2L + 2]``:
    ``(text sum, vision sum)`` per tensor, then ``(n_text, n_vision)``.  No host synchronisation.

    Tensors of several dtypes (the gradients w.r.t. a bf16 model's hidden states next to the fp32 output of its final
    layer norm) take one pass per dtype; the per-tensor sums are laid out in the caller's order, the counts taken once.

    ``group``: ``False`` (the default) returns this process's vector.  Otherwise (``None``: the default process group;
    see ``resolve_group``) the tensors are this rank's batch shard and every rank gets the vector of the whole batch,
    identical on every rank; every rank of the group must make the call.  With a peer-memory communicator the pass's
    reduce launch sums the vector over the ranks in rank order (no extra launch, no NCCL call); without one
    (``MAFED_B200_DIST=nccl``, ranks on several hosts) the vector is allreduced.  Tensors of several dtypes are exchanged
    once, as the assembled vector, by the allreduce: the reduce launch exchanges the vector of its own pass only."""
    distributed, pg = resolve_group(group)
    by_dtype = {}
    for i, t in enumerate(tensors):
        by_dtype.setdefault(t.dtype, []).append(i)
    if len(by_dtype) == 1:
        peer = get_peer_comm(pg) if distributed else None
        sums = _token_norm_sums(tensors, attn_mask, n_vis, peer)
        if distributed and peer is None:
            allreduce_sums(sums, pg)
        return sums
    rows = [None] * len(tensors)
    for idx in by_dtype.values():
        sums = _token_norm_sums([tensors[i] for i in idx], attn_mask, n_vis)
        for j, i in enumerate(idx):
            rows[i] = sums[2 * j:2 * j + 2]
    sums = torch.cat(rows + [sums[2 * len(idx):]])
    if distributed:
        allreduce_sums(sums, pg)
    return sums


def _token_norm_sums(tensors: Sequence[torch.Tensor], attn_mask: torch.Tensor, n_vis: int, peer=None) -> torch.Tensor:
    """``token_norm_sums`` over tensors of one dtype: one pass (summed over the ranks of ``peer``, a ``PeerComm``)."""
    lib = cabi.load()
    tensors = _prepare([t.detach() for t in tensors])
    plan = DistillPlan(layers=list(range(len(tensors))), layer_coeffs=[1.0] * len(tensors), n_vis=n_vis)
    ln = _Launch(tensors, tensors, attn_mask, plan)
    L, dev = ln.n_layers, ln.device
    with _on_device(dev):
        stream = _stream_ptr(dev)
        ws = torch.empty(lib.mafed_distill_ws_bytes(L), dtype=torch.uint8, device=dev)
        sums = torch.empty(2 * L + 2, dtype=torch.float64, device=dev)
        cabi.check(lib.mafed_distill_token_norm_sums(ln.shape_ref, ln.s_ptrs, ln.mask_ptr, ws.data_ptr(), stream),
                   "mafed_distill_token_norm_sums")
        cabi.check(cabi.reduce_stage(lib, ln.shape_ref, ln.mask_ptr, ws.data_ptr(), sums.data_ptr(), stream,
                                     peer.handle if peer is not None else None), "mafed_distill_scalar_stage(reduce)")
    return sums


def resolve_group(group):
    """``None``: the default process group if one is initialised with more than one rank;
    ``False``: never communicate; otherwise an explicit ``ProcessGroup``."""
    if group is False:
        return False, None
    dist = torch.distributed
    if group is None or group is True:
        on = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        return on, None
    return dist.get_world_size(group) > 1, group


def allreduce_sums(sums: torch.Tensor, group=None) -> torch.Tensor:
    """The path's collective: SUM-allreduce of fp64 partial sums and/or token counts (<= 2L+2 values)."""
    torch.distributed.all_reduce(sums, op=torch.distributed.ReduceOp.SUM, group=group)
    return sums


def distill_forward(students, teachers, attn_mask, plan: DistillPlan, group=None):
    """Two-pass step, first half: the fused forward; its last CTA reduces the partial sums and forms the
    losses and the backward scale table (one launch).  Returns ``(out, bwd_scale, launch)``.

    ``out`` is a device fp32 vector ``[1 + 3L]``: total loss, L layer losses (what the reference
    logs to W&B, ``distillation.py:165``), then L x (text loss, vision loss).
    """
    lib = cabi.load()
    ln = _Launch(students, teachers, attn_mask, plan)
    L, dev = ln.n_layers, ln.device
    with _on_device(dev):
        stream = _stream_ptr(dev)
        ws, out, bwd_scale = ln.alloc_scalars(lib)
        w = ctypes.byref(plan.weights())
        distributed, pg = resolve_group(group)
        peer = get_peer_comm(pg) if distributed else None
        if distributed and peer is None:
            cabi.check(lib.mafed_distill_fwd(ln.shape_ref, ln.s_ptrs, ln.t_ptrs, ln.mask_ptr, ws.data_ptr(), stream),
                       "mafed_distill_fwd")
            sums = torch.empty(2 * L + 2, dtype=torch.float64, device=dev)
            cabi.check(cabi.reduce_stage(lib, ln.shape_ref, ln.mask_ptr, ws.data_ptr(), sums.data_ptr(), stream),
                       "mafed_distill_scalar_stage(reduce)")
            allreduce_sums(sums, pg)
            cabi.check(cabi.finalize_stage(lib, ln.shape_ref, w, sums.data_ptr(), out.data_ptr(),
                                           bwd_scale.data_ptr(), stream), "mafed_distill_scalar_stage(finalize)")
        else:
            # forward + reduce + counts (+ NVLink peer allreduce) + losses + scale: one launch, no NCCL call
            sums = torch.empty(2 * L + 2, dtype=torch.float64, device=dev) if peer is not None else None
            cabi.check(lib.mafed_distill_fwd_step(
                ln.shape_ref, ln.s_ptrs, ln.t_ptrs, ln.mask_ptr, w, ws.data_ptr(), out.data_ptr(),
                bwd_scale.data_ptr(), sums.data_ptr() if sums is not None else None,
                peer.handle if peer is not None else None, stream), "mafed_distill_fwd_step")
    return out, bwd_scale, ln


def distill_backward(ln: _Launch, grads: Sequence[Optional[torch.Tensor]], bwd_scale: torch.Tensor,
                     grad_out: Optional[torch.Tensor], skip_if_equals: Optional[float] = None,
                     grad_out_scale: float = 1.0, seen: Optional[torch.Tensor] = None):
    """Fused backward into pre-allocated ``grads`` (``None`` entries are skipped).  With ``skip_if_equals`` the
    launch is the one-pass step's gate: a 1-CTA kernel that does nothing when the upstream gradient (times
    ``grad_out_scale``) equals that value and otherwise starts the backward from the device.  ``seen``: optional
    pinned float tensor that receives the upstream gradient the gate saw."""
    lib = cabi.load()
    g_ptrs = cabi.ptr_array([g.data_ptr() if g is not None else None for g in grads])
    skip = ctypes.byref(ctypes.c_float(skip_if_equals)) if skip_if_equals is not None else None
    with _on_device(ln.device):
        cabi.check(lib.mafed_distill_bwd(ln.shape_ref, ln.s_ptrs, ln.t_ptrs, g_ptrs, ln.mask_ptr,
                                         bwd_scale.data_ptr(), grad_out.data_ptr() if grad_out is not None else None,
                                         float(grad_out_scale), skip, seen.data_ptr() if seen is not None else None,
                                         _stream_ptr(ln.device)), "mafed_distill_bwd")


def _ticket_ptr(ticket):
    """Device address of a counts ticket (``node.prefetch_counts``); the current stream is made to wait for the
    side-stream launch that fills it."""
    if ticket is None:
        return None
    if hasattr(ticket, "wait"):
        ticket.wait()
    return ticket.data_ptr()


def distill_fused(students, teachers, grads, attn_mask, plan: DistillPlan, group=None, mask_out=None, ticket=None):
    """One-pass step: counts -> gradient scale, loss sums + gradients from one read of student and teacher,
    losses -- a single launch of the fused kernel (``mafed_distill_step``); ``mask_out = (lang, image)`` int64
    ``[B, T]`` tensors are filled by the same kernel.  Returns ``(out, bwd_scale, launch)``."""
    lib = cabi.load()
    ln = _Launch(students, teachers, attn_mask, plan)
    L, dev = ln.n_layers, ln.device
    fixed = float(plan.assumed_grad_out) * float(plan.grad_multiplier)
    g_ptrs = cabi.ptr_array([g.data_ptr() if g is not None else None for g in grads])
    with _on_device(dev):
        stream = _stream_ptr(dev)
        ws, out, bwd_scale = ln.alloc_scalars(lib)
        w = ctypes.byref(plan.weights())
        distributed, pg = resolve_group(group)
        peer = get_peer_comm(pg) if distributed else None
        if not distributed or peer is not None:
            # one launch, on one GPU and across batch shards alike: with a communicator the counts are exchanged
            # inside the kernel behind its first tiles and the sums by its last CTA (NVLink peer stores, no NCCL;
            # the epochs live on the device, so the step can be captured into a CUDA graph and replayed)
            sums = torch.empty(2 * L + 2, dtype=torch.float64, device=dev) if peer is not None else None
            lang, image = mask_out if mask_out is not None else (None, None)
            cabi.check(lib.mafed_distill_step(
                ln.shape_ref, ln.s_ptrs, ln.t_ptrs, g_ptrs, ln.mask_ptr, w, fixed, ws.data_ptr(), out.data_ptr(),
                bwd_scale.data_ptr(), sums.data_ptr() if sums is not None else None,
                lang.data_ptr() if lang is not None else None, image.data_ptr() if image is not None else None,
                peer.handle if peer is not None else None, _ticket_ptr(ticket), stream),
                "mafed_distill_step")
            return out, bwd_scale, ln
        if mask_out is not None:
            modality_masks_into(ln.mask, plan.n_vis, *mask_out)
        sums = torch.empty(2 * L + 2, dtype=torch.float64, device=dev)
        # NCCL: counts allreduce -> scale table -> fused pass -> sums allreduce -> losses
        cabi.check(lib.mafed_distill_scalar_stage(ln.shape_ref, None, cabi.STAGE_COUNTS, ln.mask_ptr, None,
                                                  sums.data_ptr(), None, None, None, 0, stream), "counts")
        allreduce_sums(sums[2 * L:], pg)
        cabi.check(lib.mafed_distill_scalar_stage(ln.shape_ref, w, cabi.STAGE_SCALE, None, None, sums.data_ptr(), None,
                                                  bwd_scale.data_ptr(), None, 0, stream), "scale")
        cabi.check(lib.mafed_distill_fused(ln.shape_ref, ln.s_ptrs, ln.t_ptrs, g_ptrs, ln.mask_ptr, None,
                                           bwd_scale.data_ptr(), fixed, ws.data_ptr(), None, stream),
                   "mafed_distill_fused")
        cabi.check(lib.mafed_distill_scalar_stage(ln.shape_ref, None, cabi.STAGE_REDUCE, None, ws.data_ptr(),
                                                  sums.data_ptr(), None, None, None, 0, stream), "reduce")
        allreduce_sums(sums[: 2 * L], pg)
        cabi.check(cabi.finalize_stage(lib, ln.shape_ref, w, sums.data_ptr(), out.data_ptr(), None, stream),
                   "mafed_distill_scalar_stage(finalize)")
    return out, bwd_scale, ln


def _alloc_grads(students, needs: Sequence[bool], cls: bool):
    """Gradient buffers for the layers that need them: ONE allocation carved into per-layer views (the
    caching allocator and the Python overhead are paid once, not L times)."""
    idx = [i for i, need in enumerate(needs) if need]
    if not idx:
        return [None] * len(students)
    s0 = students[idx[0]]
    make = torch.zeros if cls else torch.empty   # cls: only row 0 of each sample is written by the kernel
    buf = make((len(idx),) + tuple(s0.shape), dtype=s0.dtype, device=s0.device)
    views = buf.unbind(0)
    grads = [None] * len(students)
    for j, i in enumerate(idx):
        grads[i] = views[j]
    return grads


class _DistillFunction(torch.autograd.Function):
    """The step as a Python autograd Function over the ctypes calls: used when the ranks have no peer-memory
    communicator (NCCL sequence) -- every other step goes through the compiled node (``_node_step``).  Inputs: (plan, attention_mask, group, teachers tuple, mask_out, *students).  The teachers ride in a plain
    tuple: they never need gradients, so autograd does not have to look at them.  ``mask_out``: ``None`` or the
    pre-allocated ``(lang_masks, image_masks)`` pair to fill (``distillation.py:134-144``)."""

    @staticmethod
    def forward(ctx, plan: DistillPlan, attn_mask, group, teachers, mask_out, *students):
        students = _prepare(students)
        needs = ctx.needs_input_grad[5:]
        ctx.plan, ctx.needs, ctx.grads = plan, needs, None
        if plan.single_pass and any(needs):
            grads = _alloc_grads(students, needs, plan.cls)
            out, bwd_scale, ln = distill_fused(students, teachers, grads, attn_mask, plan, group, mask_out)
            ctx.grads = grads
        else:
            out, bwd_scale, ln = distill_forward(students, teachers, attn_mask, plan, group)
            if mask_out is not None:
                modality_masks_into(ln.mask, plan.n_vis, *mask_out)
        ctx.launch, ctx.bwd_scale = ln, bwd_scale
        # registered with autograd so that an in-place modification of a hidden state between forward and
        # backward is detected (the backward / fix-up kernel would otherwise read the modified values)
        ctx.save_for_backward(*students, *teachers)
        total, aux = out[0], out[1:]
        ctx.mark_non_differentiable(aux)
        return total, aux

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_total, _grad_aux):
        ln, plan = ctx.launch, ctx.plan
        if grad_total is None or ln is None or not any(ctx.needs):
            return (None,) * (5 + len(ctx.needs))
        _ = ctx.saved_tensors   # version-counter check of students / teachers
        g = grad_total
        if g.dtype != torch.float32 or g.device != ln.device:
            g = g.to(device=ln.device, dtype=torch.float32)
        if not g.is_contiguous():
            g = g.contiguous()
        mul = float(plan.grad_multiplier)
        if ctx.grads is not None:
            # one-pass step: gradients already exist; fix them up only if the upstream gradient differs
            grads, ctx.grads = ctx.grads, None
            fixed = float(plan.assumed_grad_out) * mul
            distill_backward(ln, grads, ctx.bwd_scale, g, skip_if_equals=fixed, grad_out_scale=mul)
        else:
            grads = _alloc_grads(ln.students, ctx.needs, plan.cls)
            distill_backward(ln, grads, ctx.bwd_scale, g, grad_out_scale=mul)
        return (None, None, None, None, None, *grads)


# Pinned words that receive the upstream gradient a backward gate saw.  The gate stores into its word when it
# RUNS, which can be after every Python object of the step is gone, so the words are never freed: one pinned
# allocation per process, slots handed out round-robin (a slot shared by two strategies after 1024 of them can
# only mislead the `assumed_grad_out` heuristic, never the results -- the gate itself decides on the device).
_SEEN_POOL = None
_seen_next = 0


def seen_slot() -> torch.Tensor:
    """A pinned float32[1] view for ``distill_loss(..., seen=...)``."""
    global _SEEN_POOL, _seen_next
    if _SEEN_POOL is None:
        _SEEN_POOL = torch.zeros(1024, dtype=torch.float32).pin_memory()
    i = _seen_next % 1024
    _seen_next += 1
    slot = _SEEN_POOL[i:i + 1]
    slot.zero_()
    return slot


def _step(plan: DistillPlan, attn_mask, group, teachers, mask_out, students, ticket=None, seen=None):
    """One launch-sized step (<= MAX_LAYERS layers): the compiled node, or the NCCL sequence without a communicator."""
    _require_cuda(students[0], "hidden_states")
    if attn_mask is not None and not plan.cls:
        _require_cuda(attn_mask, "attention_mask")
    distributed, pg = resolve_group(group)
    peer = get_peer_comm(pg) if distributed else None
    if distributed and peer is None:
        if mask_out is True:
            mask_out = torch.empty((2, attn_mask.shape[0], plan.n_vis + attn_mask.shape[1]), dtype=torch.int64,
                                   device=attn_mask.device)
        both = (mask_out[0], mask_out[1]) if mask_out is not None else None
        if not _native_dtypes(students, teachers):
            students, teachers = [s.float() for s in students], [t.float() for t in teachers]
        total, aux = _DistillFunction.apply(plan, attn_mask, group, tuple(_prepare(teachers)), both, *students)
        return total, aux, mask_out
    ext = node.load()
    return ext.distill(plan.node_plan(), students, teachers, None if plan.cls else attn_mask, mask_out,
                       peer.handle.value if peer is not None else 0, ticket, seen, cabi.active_tuning_address())


@torch._dynamo.assume_constant_result
def _compiled_comm(group, generation: int) -> int:
    """The peer communicator's handle for a compiled step: 0 on one rank, -1 for the NCCL sequence.  It is a host object
    Dynamo cannot trace, so it is read when the step is traced and becomes a constant of the graph; ``generation``
    (``comm._generation``, which ``comm.reset()`` bumps) is read by the traced code, so Dynamo guards on it and a graph
    is retraced rather than handed a torn-down communicator.  Tracing also puts the in-place pass back in front if the
    caller replaced Inductor's post-grad pre-pass after the extension loaded."""
    from . import ops
    ops.install_graph_pass()
    distributed, pg = resolve_group(group)
    peer = get_peer_comm(pg) if distributed else None
    return -1 if distributed and peer is None else (peer.handle.value if peer is not None else 0)


def _op_step(plan: DistillPlan, attn_mask, teachers, mask_out, students, comm, tuning):
    """One launch-sized step through the ``mafed::`` ops (``mafed_b200.ops``): what ``torch.compile`` traces."""
    if not _native_dtypes(students, teachers):
        students, teachers = [s.float() for s in students], [t.float() for t in teachers]
    needs = [torch.is_grad_enabled() and s.requires_grad for s in students]
    mask = None
    if not plan.cls:
        mask = attn_mask if attn_mask.dtype == torch.int64 else attn_mask.to(torch.int64)
    want_masks = mask_out is not None and not plan.cls
    args = (list(students), list(teachers), mask, [float(c) for c in plan.layer_coeffs],
            None if plan.lang_weights is None else [float(c) for c in plan.lang_weights],
            cabi.MODW_CLS if plan.cls else plan.modality_kind, float(plan.distill_coeff), plan.loss_kind,
            bool(plan.cls), int(plan.n_vis))
    if plan.single_pass and any(needs):
        out, _, _, masks = torch.ops.mafed.step(*args, float(plan.assumed_grad_out), float(plan.grad_multiplier), needs,
                                                comm, want_masks, tuning)
    else:
        out, _, masks = torch.ops.mafed.fwd_step(*args, float(plan.grad_multiplier), needs, comm, want_masks, tuning)
    if not want_masks:
        masks = None
    elif torch.is_tensor(mask_out):
        mask_out.copy_(masks)
        masks = mask_out
    return out[0], out[1:], masks


# The NCCL sequence (a process group without a peer communicator) is host-driven: it runs eagerly, behind a graph break.
_step_eager = torch.compiler.disable(_step)


def _any_step(plan, attn_mask, group, teachers, mask_out, students, ticket, seen):
    if not torch.compiler.is_compiling():
        return _step(plan, attn_mask, group, teachers, mask_out, students, ticket, seen)
    node.load()
    comm = _compiled_comm(group, _comm._generation)
    # a plain int global: Dynamo guards on it, so a step traced inside `with cabi.tuning(...)` is retraced outside it
    tuning = cabi._active_tuning_address
    if comm == -1:
        return _step_eager(plan, attn_mask, group, teachers, mask_out, students, ticket, seen)
    return _op_step(plan, attn_mask, teachers, mask_out, students, comm, tuning)


def distill_loss(students: Sequence[torch.Tensor], teachers: Sequence[torch.Tensor], attn_mask, plan: DistillPlan,
                 group=None, teachers_detached: bool = False, mask_out=None, ticket=None, seen=None,
                 return_masks: bool = False):
    """Differentiable fused distillation loss over ``len(students)`` selected layers.

    Returns ``(total, aux)``: ``total`` is the 0-dim fp32 loss (gradients flow to ``students``),
    ``aux`` the non-differentiable ``[3L]`` vector of layer losses then (text, vision) losses.
    ``mask_out``: optional pre-allocated int64 ``[2, B, T]`` tensor, or ``True`` to have one allocated; the step's
    own kernel fills ``[0]`` with ``lang_masks`` and ``[1]`` with ``image_masks`` (``attn_mask`` must then be a
    contiguous int64 CUDA tensor); ``return_masks=True`` appends ``(lang_masks, image_masks)`` (or ``None``) to
    the result.
    ``ticket``: the token counts sent ahead of the step (``prefetch_counts``).  ``seen``: pinned float32 tensor
    that receives the upstream gradient the backward gate saw.
    Layers may differ in dtype: each ``(student, teacher)`` dtype group runs as its own launch (``dtype_groups``).

    Under ``torch.compile`` the step runs through the ``mafed::`` ops (``mafed_b200.ops``), which Dynamo traces into the
    caller's graph; ``ticket`` and ``seen`` are ignored there (the kernel exchanges the counts itself; nothing records
    the upstream gradient).  A process group without a peer communicator (the NCCL sequence) is not compiled: the
    step runs eagerly behind a graph break.
    """
    if not teachers_detached:
        teachers = [t.detach() for t in teachers]
    if len(students) != len(teachers) or len(students) != len(plan.layers):
        raise ValueError("students / teachers / plan.layers length mismatch")
    # Layers of several dtype pairs, or more of them than one launch carries (MAFED_MAX_LAYERS): one launch per dtype
    # group and chunk.  Each group runs natively at its own width; only a group of pairs the kernels refuse is up-cast
    # to fp32 on both sides (inside its step), as the reference's autocast region does to the inputs of its loss
    # functions (distillation.py:90,244).  Every launch has its own backward gate, and across batch shards its own
    # exchange: the groups come from the model's dtypes, so every rank runs the same sequence.  A counts ticket is only
    # read by a step, so every launch may take it.
    split = _split(plan, students, teachers)
    if split is None:
        total, aux, both = _any_step(plan, attn_mask, group, teachers, mask_out, students, ticket, seen)
    else:
        steps, runs = split
        total, aux, both = _joined(steps, runs, [
            _any_step(sub, attn_mask, group, [teachers[i] for i in idx], mask_out if k == 0 else None,
                      [students[i] for i in idx], ticket, seen) for k, (idx, sub) in enumerate(steps)])
    if not return_masks:
        return total, aux
    return total, aux, (None if both is None else (both[0], both[1]))


def _split(plan: DistillPlan, students, teachers):
    """``None`` when one launch takes every layer, else ``plan.split`` of the layers' dtype pairs."""
    s_type, t_type = students[0].dtype, teachers[0].dtype
    one_launch = len(students) <= cabi.MAX_LAYERS
    for s, t in zip(students, teachers):
        one_launch = one_launch and s.dtype == s_type and t.dtype == t_type
    return None if one_launch else plan.split(tuple([(s.dtype, t.dtype) for s, t in zip(students, teachers)]))


def _joined(steps, runs, results):
    """``(total, aux, masks)`` of a step run as several launches (``results``: each launch's ``(total, aux, masks)``),
    with ``aux`` in the caller's layer order: layer losses, then (text, vision) pairs."""
    total, parts = None, []
    for part, aux, _ in results:
        total = part if total is None else total + part
        parts.append(aux)
    aux = torch.cat([parts[k][lo:hi] for k, lo, hi in runs] +
                    [parts[k][len(steps[k][0]) + 2 * lo:len(steps[k][0]) + 2 * hi] for k, lo, hi in runs])
    return total, aux, results[0][2]


def cached_distill_loss(students: Sequence[torch.Tensor], cache: Sequence[torch.Tensor], idx: Sequence[int], T_c: int,
                        attn_mask, plan: DistillPlan, mask_out=None, seen=None, return_masks: bool = False):
    """``distill_loss`` of one rank's one-pass step whose teacher rows come straight from the teacher cache: ``cache``
    holds one contiguous ``[M, T_c, D]`` tensor per selected layer (``TeacherCache.step_inputs``) and sample ``b`` of
    the batch is memory sample ``idx[b]``.  The step's kernels read the rows where they are, so no ``[B, T, D]`` copy
    of the teacher is made; the loss, gradients, masks and ``aux`` are bit-identical to ``distill_loss`` on the
    gathered teachers (``teacher_cache.gather``).

    Returns ``None``, having launched nothing, when some launch of the step is not one ``libmafed_cached_step.so``
    takes (``mafed_cached_step_supported``; a launch without gradients, i.e. the two-pass form; a dtype group the
    kernels refuse): the caller then gathers and calls ``distill_loss``, so a step never mixes the two libraries.
    The same ``dtype_groups`` split as ``distill_loss``; CLS, the two-pass form, batch sharding and ``torch.compile``
    are the caller's to route to ``distill_loss``."""
    if len(students) != len(cache) or len(students) != len(plan.layers):
        raise ValueError("students / cache / plan.layers length mismatch")
    if plan.cls or not plan.single_pass or not torch.is_grad_enabled():
        return None
    ext = node.load_cached()
    tuning = cabi.active_tuning_address()
    split = _split(plan, students, cache)
    steps = [(None, plan)] if split is None else split[0]
    launches = []
    for lidx, sub in steps:
        s = list(students) if lidx is None else [students[i] for i in lidx]
        c = list(cache) if lidx is None else [cache[i] for i in lidx]
        if not any(x.requires_grad for x in s) or not ext.cached_supported(sub.node_plan(), s, c, T_c, tuning):
            return None
        launches.append((sub, s, c))
    idx = [int(i) for i in idx]
    results = [ext.distill_cached(sub.node_plan(), s, c, idx, T_c, attn_mask, mask_out if k == 0 else None, seen, tuning)
               for k, (sub, s, c) in enumerate(launches)]
    total, aux, both = results[0] if split is None else _joined(split[0], split[1], results)
    if not return_masks:
        return total, aux
    return total, aux, (None if both is None else (both[0], both[1]))
