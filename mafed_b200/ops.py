"""The distillation step as ``torch.library`` ops, so that ``torch.compile`` traces it into the caller's graph.

``csrc/torch_node.cpp`` declares ``mafed::step`` (the one-pass step, ``mafed_distill_step``), ``mafed::fwd_step`` (the
two-pass first half, ``mafed_distill_fwd_step``) and ``mafed::bwd`` (``mafed_distill_bwd``, mutating its ``grads``)
with their CUDA implementations.  This module gives them what the compiler needs besides: fake implementations
(shapes and dtypes only), the autograd formula of the two forward ops, and a graph pass that lets Inductor run
``mafed::bwd`` in place.  ``node.load()`` calls ``register()`` once the extension is loaded.

The autograd formula saves students, teachers and the mask as the compiled node does (the gate's exact fallback reads
them).  One-pass step: the backward is the 1-CTA gate over the saved gradient buffer.  Two-pass step: the backward runs
into a freshly allocated buffer.  Either way the per-layer gradients are views of one ``[n_need, B, T, D]`` buffer.
"""
from __future__ import annotations

import operator
import warnings

import torch
from torch._inductor.custom_graph_pass import CustomGraphPass

_registered = False


def _masks_fake(s0, want_masks, cls):
    shape = (2, s0.shape[0], s0.shape[1]) if want_masks and not cls else (0,)
    return s0.new_empty(shape, dtype=torch.int64)


def _step_fake(students, teachers, mask, layer_coeffs, lang_weights, modality_kind, distill_coeff, loss_kind, cls,
               n_vis, assumed_grad_out, grad_multiplier, needs, comm, want_masks, tuning):
    s0, L = students[0], len(students)
    out = s0.new_empty((1 + 3 * L,), dtype=torch.float32)
    grads = s0.new_empty((sum(bool(n) for n in needs),) + tuple(s0.shape))
    return out, grads, s0.new_empty((2 * L,), dtype=torch.float32), _masks_fake(s0, want_masks, cls)


def _fwd_step_fake(students, teachers, mask, layer_coeffs, lang_weights, modality_kind, distill_coeff, loss_kind, cls,
                   n_vis, grad_multiplier, needs, comm, want_masks, tuning):
    s0, L = students[0], len(students)
    out = s0.new_empty((1 + 3 * L,), dtype=torch.float32)
    return out, s0.new_empty((2 * L,), dtype=torch.float32), _masks_fake(s0, want_masks, cls)


def _bwd_fake(students, teachers, mask, grads, bwd_scale, grad_out, grad_out_scale, skip_if_equals, needs, loss_kind,
              cls, n_vis, tuning):
    return None


def _save(ctx, students, teachers, mask, extra, needs, loss_kind, cls, n_vis, tuning):
    ctx.n, ctx.has_mask = len(students), mask is not None
    ctx.save_for_backward(*students, *teachers, *([mask] if mask is not None else []), *extra)
    ctx.needs, ctx.loss_kind, ctx.cls, ctx.n_vis, ctx.tuning = list(needs), loss_kind, cls, n_vis, tuning
    ctx.set_materialize_grads(False)


def _unpack(ctx):
    saved, n = ctx.saved_tensors, ctx.n
    mask = saved[2 * n] if ctx.has_mask else None
    return list(saved[:n]), list(saved[n:2 * n]), mask, saved[2 * n + int(ctx.has_mask):]


def _per_layer(buf, needs):
    views = iter(buf.unbind(0))
    return [next(views) if need else None for need in needs]


def _step_setup(ctx, inputs, output):
    (students, teachers, mask, _coeffs, _lang, _kind, _dc, loss_kind, cls, n_vis, assumed, mul, needs, _comm, _want,
     tuning) = inputs
    out, grads, bwd_scale, masks = output
    ctx.mark_non_differentiable(grads, bwd_scale, masks)
    _save(ctx, students, teachers, mask, (grads, bwd_scale), needs, loss_kind, cls, n_vis, tuning)
    ctx.fixed, ctx.mul = float(assumed) * float(mul), float(mul)


def _no_grads(ctx, n_rest):
    # one entry per input: per-layer lists for the two Tensor[] inputs, None for the rest
    return ([None] * ctx.n, [None] * ctx.n) + (None,) * n_rest


def _step_backward(ctx, d_out, _d_grads, _d_scale, _d_masks):
    if d_out is None:
        return _no_grads(ctx, 14)
    students, teachers, mask, (grads, bwd_scale) = _unpack(ctx)
    # the gate: nothing happens when the upstream gradient is the assumed one, else the exact backward into `grads`
    torch.ops.mafed.bwd(students, teachers, mask, grads, bwd_scale, d_out.float().contiguous(), ctx.mul, ctx.fixed,
                        ctx.needs, ctx.loss_kind, ctx.cls, ctx.n_vis, ctx.tuning)
    return (_per_layer(grads, ctx.needs), [None] * ctx.n) + (None,) * 14


def _fwd_step_setup(ctx, inputs, output):
    (students, teachers, mask, _coeffs, _lang, _kind, _dc, loss_kind, cls, n_vis, mul, needs, _comm, _want,
     tuning) = inputs
    out, bwd_scale, masks = output
    ctx.mark_non_differentiable(bwd_scale, masks)
    _save(ctx, students, teachers, mask, (bwd_scale,), needs, loss_kind, cls, n_vis, tuning)
    ctx.mul = float(mul)


def _fwd_step_backward(ctx, d_out, _d_scale, _d_masks):
    if d_out is None or not any(ctx.needs):
        return _no_grads(ctx, 13)
    students, teachers, mask, (bwd_scale,) = _unpack(ctx)
    s0 = students[0]
    make = torch.zeros if ctx.cls else torch.empty      # cls: only row 0 of each sample is written by the kernel
    grads = make((sum(ctx.needs),) + tuple(s0.shape), dtype=s0.dtype, device=s0.device)
    torch.ops.mafed.bwd(students, teachers, mask, grads, bwd_scale, d_out.float().contiguous(), ctx.mul, None,
                        ctx.needs, ctx.loss_kind, ctx.cls, ctx.n_vis, ctx.tuning)
    return (_per_layer(grads, ctx.needs), [None] * ctx.n) + (None,) * 13


class _BwdInPlace(CustomGraphPass):
    """Post-grad graph pass: let Inductor run ``mafed::bwd`` in place on the saved gradient buffer.

    In the backward graph the one-pass step's gradient buffer is a graph input (a saved activation).  Inductor
    re-inplaces a functionalized mutation of a graph input only when the graph writes the result back into it (a
    ``copy_`` epilogue); otherwise it clones the buffer first, a 2*D*e pass per token*layer that the eager path does not
    have.  The buffer is dead once the gate has run, so writing back is what the step means: this pass adds that
    ``copy_`` for every ``mafed::bwd`` whose buffer is a graph input.  After re-inplacing, the ``copy_`` is a copy of the
    buffer onto itself, which Inductor lowers to nothing.  It runs before a pre-pass the caller had installed, and a
    compiled step that is traced after the caller replaced the pre-pass installs it again in front (see
    ``distill_op._compiled_comm``).  A ``mafed::bwd`` in a functionalization layout this pass does not know raises a
    RuntimeWarning instead of silently costing a copy."""

    def __init__(self, then=None):
        self.then = then

    def __call__(self, graph):
        hop = torch.ops.higher_order.auto_functionalized_v2
        output = next(n for n in reversed(graph.nodes) if n.op == "output")
        for node in list(graph.nodes):
            if (node.op == "call_function" and node.target is not hop and node.args
                    and node.args[0] is torch.ops.mafed.bwd.default):
                # another functionalization layout (auto_functionalized v1, a newer HOP): nothing here matches it, so
                # Inductor may clone the gradient buffer before the backward writes into it
                warnings.warn(f"mafed_b200: mafed::bwd reached Inductor as {node.target}, which the in-place pass does "
                              "not handle; the compiled backward may copy the gradient buffer once per step",
                              RuntimeWarning, stacklevel=2)
                continue
            if node.target is not hop or node.args[0] is not torch.ops.mafed.bwd.default:
                continue
            bases = node.kwargs["_all_bases"]
            first = len(node.meta["val"]) - len(bases)    # the op's own outputs, then one per base
            for i, base in enumerate(bases):
                if base.op != "placeholder":
                    continue
                new = next((u for u in node.users if u.target is operator.getitem and u.args[1] == first + i), None)
                if new is None:
                    with graph.inserting_after(node):
                        new = graph.call_function(operator.getitem, (node, first + i))
                    new.meta["val"] = node.meta["val"][first + i]
                with graph.inserting_before(output):
                    copy = graph.call_function(torch.ops.aten.copy_.default, (base, new))
                copy.meta["val"] = base.meta["val"]
        if self.then is not None:
            self.then(graph)

    def uuid(self):
        then = self.then.uuid() if self.then is not None and hasattr(self.then, "uuid") else None
        return ("mafed_b200.ops._BwdInPlace", 1, then)


def install_graph_pass():
    """Install ``_BwdInPlace`` as Inductor's post-grad pre-pass, in front of one the caller set (idempotent)."""
    from torch._inductor import config
    current = config.post_grad_custom_pre_pass
    if not isinstance(current, _BwdInPlace):
        config.post_grad_custom_pre_pass = _BwdInPlace(current)


def register():
    """Fake implementations and autograd formulas of the ``mafed`` ops, and the in-place pass (once per process).
    The ops themselves are defined by the compiled extension, which must be loaded first."""
    global _registered
    if _registered:
        return
    torch.library.register_fake("mafed::step", _step_fake)
    torch.library.register_fake("mafed::fwd_step", _fwd_step_fake)
    torch.library.register_fake("mafed::bwd", _bwd_fake)
    torch.library.register_autograd("mafed::step", _step_backward, setup_context=_step_setup)
    torch.library.register_autograd("mafed::fwd_step", _fwd_step_backward, setup_context=_fwd_step_setup)
    install_graph_pass()
    _registered = True
