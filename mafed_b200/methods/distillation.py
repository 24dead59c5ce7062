"""Modality-aware feature distillation on sm_100a kernels.

Mirror of ``mafed/methods/distillation.py:16-257``: same constructor arguments, attributes, hook
methods and return types (``distill`` -> 0-dim loss, ``replay`` -> ``(loss, n_ex)``), so it drops in
behind ``CLMethod["featdistill"]`` (``mafed/train.py:119-134``,
``mafed/model/vqa_cont_learner.py:213-254``).

What changed underneath: the reference loops over layers in Python and, per layer, builds two masks
on the CPU, runs two masked token-loss passes through ~16 ATen kernels and synchronises the host for
W&B.  Here one step is ONE kernel launch over all selected layers (masks, gradient scale, loss sums,
gradients and the loss algebra; ``mafed_distill_step``) plus, in ``backward``, a 1-CTA gate that returns at
once unless the upstream gradient differs from the assumed one (then it starts the exact backward from the
device) -- no host synchronisation; the per-layer values the reference logs (``task_{k}/distill_loss_{layer}``)
stay on the device and are logged a step or two late.  The host side of a step is one call into a compiled
autograd node (``mafed_b200.node``).
"""
from __future__ import annotations

import contextlib
from collections import deque
from copy import deepcopy
from typing import Dict, List, Optional

import numpy as np
import torch

from mafed_b200 import cabi
from mafed_b200 import comm as _comm
from mafed_b200.capture import HiddenStateCapture, HiddenStateTuple
from mafed_b200.distill_op import (DistillPlan, cached_distill_loss, distill_loss, modality_masks, resolve_group,
                                   seen_slot)
from mafed_b200.methods.base import CLStrategy
from mafed_b200.methods.distillation_loss_weights import DistillationWeights

try:  # W&B is optional here; the reference requires it
    import wandb as _wandb
except Exception:  # pragma: no cover
    _wandb = None


def _identity(x):
    """A plan-cache key part: plain values by value, objects by identity (Dynamo traces ``id()`` of objects only)."""
    return x if x is None or isinstance(x, (bool, int, float, str)) else id(x)


class _CapturedOutput:
    """Model output whose ``hidden_states`` holds only the captured (distilled) entries."""

    def __init__(self, output, hidden_states):
        self._output = output
        self.hidden_states = hidden_states

    def __getattr__(self, name):
        return getattr(self._output, name)


class FeatureDistillation(CLStrategy):
    """Feature distillation with separate vision / language weights (MAFED).

    ``teacher_cache=True`` computes the teacher's distilled hidden states of the whole episodic memory once per task
    (in ``update()``) and gathers each replay step's rows from them instead of running the teacher (INTEGRATION.md:
    the text rows' targets change).  Under ``torch.compile`` the option does not apply: the teacher forward runs.
    ``shard_teacher_cache=True`` on top of it splits the cache across the ranks of the process group (one process per
    GPU of one host): each rank builds and holds its share, and a step gathers each sample's rows from whichever GPU
    holds them, with the same numbers as the replicated cache."""

    def __init__(
        self,
        memory_size,
        opts,
        model_type,
        distillation_modality_weighing_strategy="equal",
        distillation_layer_weighing_strategy="single",
        distillation_coeff=1.0,
        replay_coeff=1.0,
        distillation_layer=-1,
        cls_distillation=False,
        distillation_loss="mse",
        gamma: float = 0.8,
        num_hidden_layers: int = 11,
        **kwargs,
    ):
        super().__init__(opts=opts)
        self.opts = opts
        self.model_type = model_type
        # ---- episodic memory bookkeeping (reference :36-46)
        self.memory_size = memory_size
        self.memory_per_task = int(memory_size / (len(opts.tasks) - 1))
        self.batch_size = opts.batch_size
        self.num_workers = 2
        self.seed = 1
        self.datasets = []
        self.rng = np.random.default_rng(opts.seed)
        self.pin_mem = opts.pin_mem
        self.step = 0
        # ---- loss configuration (reference :49-73)
        self.past_model = None
        self.replay_coeff = replay_coeff
        self.distillation_coeff = distillation_coeff
        self.weighing_strategy = distillation_modality_weighing_strategy
        self._cls_distillation = cls_distillation
        self.distillation_loss = "cosine" if distillation_loss == "cosine" else "mse"
        self._loss_kind = cabi.LOSS_COSINE if self.distillation_loss == "cosine" else cabi.LOSS_MSE
        self._compute_distillation_loss = (
            self._compute_cosine_distillation_loss if self._loss_kind == cabi.LOSS_COSINE
            else self._compute_mse_distillation_loss)
        in_range = distillation_layer is not None and 0 <= distillation_layer < num_hidden_layers
        self.loss_weights = DistillationWeights(
            distillation_modality_weighing_strategy=distillation_modality_weighing_strategy,
            distillation_layer_weighing_strategy=distillation_layer_weighing_strategy,
            gamma=gamma,
            num_hidden_layers=num_hidden_layers,
            distillation_layer=distillation_layer if in_range else None,
        )
        self.num_vision_tokens = 256
        # ---- B200 path state
        self.process_group = kwargs.get("process_group")   # None: default group when initialised
        self.populate_batch_masks = True                    # keep the reference's side effect on `batch`
        # one-pass step (loss sums and gradients from a single read of student and teacher); the upstream
        # gradient it bakes in is Lightning's 1/accumulate_grad_batches, checked on the device in backward
        self.single_pass = bool(kwargs.get("single_pass", True))
        self.assumed_grad_out = 1.0 / float(self.update_freq)
        # The backward gate leaves the upstream gradient it really saw in a pinned word; distill() reads it (a plain
        # host read, possibly a step old) and re-aims `assumed_grad_out`, so a trainer that scales the loss
        # differently (a static loss scale, another accumulation factor) pays the exact backward once, not per step.
        # An upstream gradient that keeps changing (dynamic loss scaling) switches the strategy to the two-pass form.
        self.adapt_assumed_grad_out = bool(kwargs.get("adapt_assumed_grad_out", True))
        self._gout_seen = self._gout_seen_np = None
        self._gout_changes = 0
        # Batch-sharded runs return the GLOBAL-batch loss on every rank, so each rank's hidden-state gradient is its
        # share of dL_global/dh.  DistributedDataParallel then AVERAGES parameter gradients over the ranks, which
        # would leave the distillation term world_size times too small next to the (per-rank mean) LM losses.
        # None: multiply by world_size whenever the sharded path is active (right under DDP); pass 1.0 when the
        # gradients are summed, not averaged, across ranks.
        self.grad_multiplier = kwargs.get("grad_multiplier")
        # record only the distilled hidden states with forward hooks instead of output_hidden_states=True
        self.selective_capture = bool(kwargs.get("selective_capture", False))
        # walk one memory-loader iterator instead of spawning a fresh one per replay step
        self.persistent_memory_iterator = bool(kwargs.get("persistent_memory_iterator", False))
        # hold the frozen teacher snapshot in bf16 / fp16 (None: the model's own dtype, as the reference does).  Its
        # forward runs under an autocast of that dtype and every teacher hidden state is handed over in it (see
        # _teacher_forward), so the step reads them as they are next to fp32 student states; the teacher's weights and
        # states are rounded to it, so the numbers differ from the reference's
        self.teacher_dtype = kwargs.get("teacher_dtype")
        if self.teacher_dtype not in (None, torch.bfloat16, torch.float16):
            raise ValueError(f"teacher_dtype must be None, torch.bfloat16 or torch.float16, not {self.teacher_dtype!r}")
        # stop the teacher forward after the last distilled hidden state (and the student's too when no replay loss is
        # taken): the layers after it, the final layer norm and the LM head compute nothing the step reads.  Eager only:
        # under torch.compile the forwards run in full (see _stop_early)
        self.early_exit = bool(kwargs.get("early_exit", False))
        # `adaptive` weights of a batch-sharded run: compute the importances over the union of the ranks' task loaders,
        # the same on every rank (one exchange per task), instead of each rank's own shard.  Off by default: each rank
        # then keeps its own importances, as naive DDP over the reference does
        self.global_importances = bool(kwargs.get("global_importances", False))
        # serve replay steps' teacher states from a per-task cache of the episodic memory (mafed_b200.teacher_cache)
        # instead of a teacher forward: built in update(), gathered by one kernel per step.  Eager only, as early_exit
        self.teacher_cache = bool(kwargs.get("teacher_cache", False))
        # split the cache across the ranks of the process group (teacher_cache.build_sharded) instead of a whole copy
        # per rank: HBM held for the task traded against NVLink reads per step.  On one rank the cache is replicated
        self.shard_teacher_cache = bool(kwargs.get("shard_teacher_cache", False))
        if self.shard_teacher_cache and not self.teacher_cache:
            raise ValueError("shard_teacher_cache=True needs teacher_cache=True")
        self._teacher_cache = None          # the TeacherCache of the current task (None: built on the next replay)
        self._retired_cache = None          # a sharded cache load_state_dict dropped: released by the next build
        self._memory_index = None           # memory indices of the batch replay() drew, for _past_states
        self._mem_iter = self._mem_iter_source = None
        self._mem_epoch = 0
        self._plan_cache = None
        self.last_layer_losses: Optional[torch.Tensor] = None   # device [3L]: layer, then (text, vision)
        self.last_layers: List[int] = []
        self._pending_logs = deque()
        self._tickets = {}                                   # id(attention_mask) -> (mask, its version, ticket)

    # ------------------------------------------------------------------ trainer hooks
    def update(self, dataset, model, dataloader, mask=None, **kwargs):
        self._update_model(model)
        self._update_memory(dataset)
        if self.teacher_cache:
            self._build_teacher_cache()
        if self.global_importances:
            self.loss_weights.update_weights(model, dataloader, self.task_id, process_group=self.process_group)
            self.check_importances()
        else:
            self.loss_weights.update_weights(model, dataloader, self.task_id)
        self.task_id += 1

    def check_importances(self):
        """``global_importances``: raise unless every rank of the group holds rank 0's ``adaptive`` language weights
        (compared bit for bit, one all-gather of the L-float host table).  Ranks whose kernels read different weights
        would each compute a different "global" loss, and DDP would average gradients of no single computation."""
        distributed, pg = resolve_group(self.process_group)
        if not distributed or self.loss_weights._modality_weighing_strategy != "adaptive":
            return
        dist = torch.distributed
        bits = torch.tensor(self.loss_weights._adaptive_host_table(), dtype=torch.float32).view(torch.int32).tolist()
        every = [None] * dist.get_world_size(pg)
        dist.all_gather_object(every, bits, group=pg)
        differ = [r if pg is None else dist.get_global_rank(pg, r) for r, b in enumerate(every) if b != every[0]]
        if differ:
            raise cabi.MafedDistillError(
                f"the adaptive language weights of rank(s) {differ} differ from rank 0's after the importance exchange: "
                "every rank must compute them over the same process group")

    def compute_loss(self, model, loss, batch, **kwargs):
        return loss

    def update_after_new_task(self, model, dataset):
        if self.weighing_strategy != "loss_based":
            return
        self.lang_coeff = self.loss_based_distill.update(
            new_model=model, new_dataset=dataset, memory_dataloader=self.mem_dataloader)

    def update_after_step(self, model, batch_idx=0, on_train_start=False):
        if self.task_id == 0 or self.weighing_strategy != "dynamic":
            return
        if self._is_batch_after_step(batch_idx):
            model.vqa_output_distill_loss_params.update()

    def update_mask(self, mask=None):
        pass

    # ------------------------------------------------------------------ the replay / distillation step
    def replay(self, model):
        """Memory batch -> student forward (hidden states kept) -> replay LM loss + distillation loss.
        Returns ``(loss, n_examples)`` like ``distillation.py:84-103``."""
        batch = self._next_memory_batch()
        if self.teacher_cache:
            self._memory_index = batch.pop("memory_index", None)
        n_ex = batch["input_ids"].size(0)
        do_replay = self.replay_coeff > 0 and self.task_id > 0
        loss = None
        if self.distillation_coeff != 0 and not self._cls_distillation:
            # batch-sharded: this rank's token counts leave for the peers now, behind the student forward
            self.prefetch_counts(batch)
        # without a replay loss nothing reads the student's output past the last distilled hidden state
        stop_student = not do_replay and self._stop_early()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if (self.selective_capture or stop_student) and self.distillation_coeff != 0:
                # keep only the distilled entries of the hidden-state tuple alive (SURVEY 8f rank 2)
                output = None       # stays None when the capture stops the forward: no logits, no loss
                with HiddenStateCapture(model, self.loss_weights.get_distillation_layers(),
                                        stop_after_last=stop_student) as cap:
                    output = model(**batch, compute_loss=do_replay, output_hidden_states=False, return_dict=True)
                output = _CapturedOutput(output, cap.hidden_states)
            else:
                output = model(**batch, compute_loss=do_replay, output_hidden_states=True, return_dict=True)
            if do_replay:
                loss = self.replay_coeff * output.loss
            if self.distillation_coeff == 0:
                return loss, n_ex
            dloss = self.distill(output=output, batch=batch)
            loss = dloss if loss is None else loss + dloss
        return loss, n_ex

    def _next_memory_batch(self):
        """The reference builds a NEW DataLoader iterator for every replay step
        (``next(iter(self.mem_dataloader))``, ``distillation.py:85``), i.e. the first batch of a fresh
        shuffle -- and a respawn of the loader's worker processes each time.  That stays the default;
        ``persistent_memory_iterator=True`` walks one iterator and re-creates it only when an epoch over
        the memory ends (SURVEY 8f rank 4)."""
        if not self.persistent_memory_iterator:
            return next(iter(self.mem_dataloader))
        if self._mem_iter is None or self._mem_iter_source is not self.mem_dataloader:
            self._mem_iter, self._mem_iter_source, self._mem_epoch = iter(self.mem_dataloader), self.mem_dataloader, 0
        try:
            return next(self._mem_iter)
        except StopIteration:
            self._mem_epoch += 1
            sampler = getattr(self, "mem_sampler", None)
            if hasattr(sampler, "set_epoch"):
                sampler.set_epoch(self._mem_epoch)
            self._mem_iter = iter(self.mem_dataloader)
            return next(self._mem_iter)

    def prefetch_counts(self, batch, force: bool = False):
        """Send this rank's token counts to the peers ahead of the step (batch-sharded runs).  The counts depend
        only on ``attention_mask``, which is known as soon as the memory batch is drawn -- before the student
        forward (``distillation.py:85-91``) -- so the step's kernel later finds the global counts in its own
        mailbox instead of exchanging them at its start.  The 1-CTA launch goes to a side stream (ordered behind the
        producer of the mask), so it does not sit between kernels of the compute stream.  ``replay`` calls this itself;
        a trainer that draws batches ahead may call it up to two steps early (every rank alike: the call is part of
        the exchange sequence).  No-op on a single rank unless ``force``."""
        attn = batch.get("attention_mask") if hasattr(batch, "get") else None
        if attn is None or not attn.is_cuda or attn.dtype != torch.int64 or not attn.is_contiguous():
            return None
        peer = self._peer()
        if peer is None and not force:
            return None
        from mafed_b200 import node
        ticket = node.load().prefetch_counts(attn, self.num_vision_tokens, peer.handle.value if peer is not None else 0,
                                             cabi.active_tuning_address())
        if len(self._tickets) >= 3:          # at most 3 batches ahead (the mailbox keeps 4 generations of counts)
            self._tickets.pop(next(iter(self._tickets)))
        self._tickets[id(attn)] = (attn, attn._version, ticket)
        return ticket

    def capture(self, hidden_states, past_hidden_states, attention_mask, grad_out=None, warmup: int = 3):
        """``distill`` + ``backward`` over static hidden-state buffers as a replayable CUDA graph
        (``mafed_b200.graphed.GraphedDistillStep``): every launch of the step is capture-safe, and a replay costs the
        host ~4 us instead of the ~150 us of Python and autograd-engine time of the eager calls.  ``hidden_states`` /
        ``past_hidden_states``: the student's and the teacher's full tuples; fill them (or let the producing kernels
        write there), ``step.replay()``, read ``step.loss`` / ``step.grads``."""
        from mafed_b200.graphed import GraphedDistillStep
        return GraphedDistillStep(self, hidden_states, past_hidden_states, attention_mask, grad_out=grad_out,
                                  warmup=warmup)

    def _peer(self):
        """The peer-memory communicator of a batch-sharded run (None: single rank, or the NCCL sequence)."""
        distributed, pg = resolve_group(self.process_group)
        if not distributed:
            return None
        from mafed_b200.comm import get_peer_comm
        return get_peer_comm(pg)

    def distill(self, output, batch):
        """Sum over the selected layers of ``layer_coeff * distillation_coeff * layer_loss``
        (``distillation.py:105-122``) -- as one fused launch instead of a Python loop."""
        layers = self.loss_weights.get_distillation_layers()
        # Under torch.compile the host-only bookkeeping is skipped, so the step traces without a graph break: no
        # re-aiming of `assumed_grad_out` (the gate still keeps the gradients exact), no counts ticket (the kernel
        # exchanges the counts itself), no exchange check and no W&B queue -- `record_step()` does the last two eagerly.
        compiling = torch.compiler.is_compiling()
        cached = None
        if self.teacher_cache and not compiling:
            # the cached teacher rows of this batch: read straight from the cache by the step where it takes them,
            # otherwise gathered (as _past_states does)
            batch.pop("labels", None)
            cached = self._cache_step(batch, layers)
            past_hidden_states = None
        else:
            # the teacher's states come out of a no_grad forward and the node never differentiates them: the
            # per-tensor `.detach()` of the reference (`_get_past_hidden_states`, distillation.py:223) is only paid for
            # the distilled layers, and only if a tensor carries a graph at all
            past_hidden_states = self._past_states(batch, layers)
        if self.adapt_assumed_grad_out and self._gout_seen_np is not None and not compiling:
            self._adapt_assumed()
        plan = self._step_plan(layers)
        hidden = output.hidden_states
        students = [hidden[l] for l in layers]
        result = None
        if cached is not None:
            result = self._launch_cached(plan, batch, students, *cached)
            if result is None:
                cache, idx, T = cached
                past_hidden_states = cache.gather(idx, T, layers)
        total, aux = result if result is not None else self._launch(plan, batch, students, past_hidden_states,
                                                                    teachers_detached=True)
        if compiling:
            # `self.step` is advanced by record_step(): an int attribute changed inside the trace would be guarded on,
            # and every step would retrace (or feed a new int to the graph, which CUDA-graph trees re-record for)
            self.last_layer_losses = aux
            self.last_layers = list(layers)
        else:
            self._record(aux, layers)
            self.step += 1
        return total

    def record_step(self):
        """The host side of a step that ran under ``torch.compile``: queue its per-layer losses for W&B (one
        ``wandb.log`` per layer per step, in order, as ``distill`` does eagerly) and check the in-kernel exchange of a
        batch-sharded run, and advance ``step``.  Call it once after every compiled step, outside the compiled region (with
        ``mode="reduce-overhead"``, before the next replay overwrites ``last_layer_losses``)."""
        if self.last_layer_losses is not None:
            self._record(self.last_layer_losses, self.last_layers)
        self.step += 1

    def _step_plan(self, layers) -> DistillPlan:
        """The plan of the all-layer step, rebuilt only when something it depends on changes (the host
        tables cost ~50 us of Python per step otherwise)."""
        lw = self.loss_weights
        coeff = getattr(lw, "lang_coeff", None)
        key = (tuple(layers), self.distillation_coeff, self._cls_distillation, self._loss_kind, self.num_vision_tokens,
               self.single_pass, self.assumed_grad_out, lw._modality_weighing_strategy, _identity(coeff),
               getattr(coeff, "_version", None), _identity(lw.layer_coeffs), self.grad_multiplier, self.process_group)
        if self._plan_cache is None or self._plan_cache[0] != key:
            coeffs, modality_kind, lang_weights = self._tables(layers)
            plan = self._plan(layers, coeffs, self.distillation_coeff, modality_kind, lang_weights)
            if len(layers) <= cabi.MAX_LAYERS and not torch.compiler.is_compiling():
                plan.weights()      # the ctypes tables of the eager path (the compiled ops take plain values)
            self._plan_cache = (key, plan)
        return self._plan_cache[1]

    def feature_distillation(self, batch, hidden_states, past_hidden_states, layer: int):
        """Layer loss ``w_text * loss_text + w_vision * loss_vision`` of one layer, without the layer
        coefficient (``distillation.py:124-166``)."""
        coeffs, modality_kind, lang_weights = self._tables([layer])
        plan = self._plan([layer], [1.0], 1.0, modality_kind, lang_weights)
        total, aux = self._launch(plan, batch, [hidden_states], [past_hidden_states])
        if not self._cls_distillation:
            self._record(aux, [layer])
        return total

    # ------------------------------------------------------------------ internals
    def _tables(self, layers):
        if self._cls_distillation:
            coeffs = [float(self.loss_weights.get_layer_loss_weight(l)) for l in layers]
            return coeffs, cabi.MODW_CLS, None
        return self.loss_weights.kernel_tables(layers)

    def _plan(self, layers, coeffs, distill_coeff, modality_kind, lang_weights) -> DistillPlan:
        if self._cls_distillation and self._loss_kind != cabi.LOSS_COSINE:
            # quirk kept from the reference: MSELoss takes two arguments, the CLS branch passes three
            raise TypeError("cls_distillation requires distillation_loss='cosine' "
                            "(MSELoss.forward() takes 3 positional arguments but 4 were given)")
        mul = self.grad_multiplier
        if mul is None:
            distributed, pg = resolve_group(self.process_group)
            mul = float(torch.distributed.get_world_size(pg)) if distributed else 1.0
        return DistillPlan(layers=list(layers), layer_coeffs=list(coeffs), distill_coeff=float(distill_coeff),
                           modality_kind=modality_kind, lang_weights=lang_weights, loss_kind=self._loss_kind,
                           cls=bool(self._cls_distillation), n_vis=self.num_vision_tokens,
                           single_pass=self.single_pass, assumed_grad_out=self.assumed_grad_out,
                           grad_multiplier=float(mul))

    def _adapt_assumed(self):
        """Re-aim the one-pass step at the upstream gradient the gate last saw (see ``__init__``)."""
        seen = float(self._gout_seen_np[0])
        if seen == 0.0 or seen != seen or seen in (float("inf"), float("-inf")):
            return
        mul = self._plan_cache[1].grad_multiplier if self._plan_cache is not None else 1.0
        want = seen / mul
        if abs(want - self.assumed_grad_out) <= 1e-7 * abs(want):
            return
        self.assumed_grad_out = want
        self._gout_changes += 1
        if self._gout_changes > 8 and self.single_pass:
            # the upstream gradient is not a constant of this run: stop guessing
            self.single_pass = False

    def _launch(self, plan: DistillPlan, batch, students, teachers, teachers_detached=False):
        attn, mask_out, ticket = None, None, None
        if not plan.cls:
            attn = batch["attention_mask"]
            if self.populate_batch_masks:
                if attn.is_cuda and attn.dtype == torch.int64 and attn.is_contiguous():
                    # the masks the reference leaves in `batch` are allocated and written by the step itself
                    mask_out = True
                else:
                    batch["lang_masks"], batch["image_masks"] = modality_masks(attn, self.num_vision_tokens)
            if self._tickets and not torch.compiler.is_compiling():
                tk = self._tickets.pop(id(attn), None)
                if tk is not None and tk[0] is attn and tk[1] == attn._version:
                    ticket = tk[2]
        if plan.single_pass and self._gout_seen is None and not torch.compiler.is_compiling():
            self._gout_seen = seen_slot()
            self._gout_seen_np = self._gout_seen.numpy()
        total, aux, masks = distill_loss(students, teachers, attn, plan, group=self.process_group,
                                         teachers_detached=teachers_detached, mask_out=mask_out, ticket=ticket,
                                         seen=self._gout_seen if plan.single_pass else None, return_masks=True)
        if masks is not None:
            batch["lang_masks"], batch["image_masks"] = masks
        return total, aux

    def _launch_cached(self, plan: DistillPlan, batch, students, cache, idx, T):
        """The step with the teacher rows read straight from a replicated teacher cache (``cached_distill_loss``), or
        ``None`` (nothing launched) where the gather + step takes it: a sharded cache, a step across ranks, the
        two-pass form, CLS, or a launch ``libmafed_cached_step.so`` does not take."""
        from mafed_b200 import teacher_cache
        if (not isinstance(cache, teacher_cache.TeacherCache) or resolve_group(self.process_group)[0] or
                not plan.single_pass or plan.cls):
            return None
        states, idx, T, T_c = cache.step_inputs(idx, T, plan.layers)
        attn, mask_out = batch["attention_mask"], None
        if self.populate_batch_masks and attn.is_cuda and attn.dtype == torch.int64 and attn.is_contiguous():
            mask_out = True
        if self._gout_seen is None:
            self._gout_seen = seen_slot()
            self._gout_seen_np = self._gout_seen.numpy()
        res = cached_distill_loss(students, states, idx, T_c, attn, plan, mask_out=mask_out, seen=self._gout_seen,
                                  return_masks=True)
        if res is None:
            return None
        total, aux, masks = res
        if masks is not None:
            batch["lang_masks"], batch["image_masks"] = masks
        elif self.populate_batch_masks:
            batch["lang_masks"], batch["image_masks"] = modality_masks(attn, self.num_vision_tokens)
        return total, aux

    def _teacher_forward(self, batch):
        """Autocast region of the teacher forward.  A snapshot held in ``teacher_dtype`` runs under an autocast of that
        dtype: inside replay's bf16 region an fp16 snapshot would otherwise get bf16 out of its linears next to fp16 out
        of its embeddings, and its hidden states would come out in mixed dtypes."""
        if self.teacher_dtype is None:
            return contextlib.nullcontext()
        am = batch.get("attention_mask")
        return torch.autocast(am.device.type if torch.is_tensor(am) else "cuda", dtype=self.teacher_dtype)

    def _as_teacher_dtype(self, h):
        """A teacher hidden state in ``teacher_dtype`` (if set).  Autocast leaves some of them in fp32 (the output of the
        final layer norm: layer_norm is an fp32 op under autocast); rounding that one too keeps every distilled teacher
        state in one dtype, so the step reads them natively instead of up-casting every layer."""
        return h if self.teacher_dtype is None or h.dtype == self.teacher_dtype else h.to(self.teacher_dtype)

    def _stop_early(self) -> bool:
        """``early_exit`` in effect: eager calls only.  A compiled step keeps the full forwards, which trace into one
        graph; the capture's hooks and the exception that stops the forward would not."""
        return self.early_exit and not torch.compiler.is_compiling()

    def _past_states(self, batch, layers):
        """Teacher hidden states of the distilled layers only (same forward and side effects as
        ``_get_past_hidden_states``; with ``early_exit`` the forward stops after the last of them)."""
        if self.teacher_cache and not torch.compiler.is_compiling():
            batch.pop("labels", None)
            return self._cached_past_states(batch, layers)
        stop = self._stop_early()
        with torch.no_grad(), self._teacher_forward(batch):
            batch.pop("labels", None)
            if self.selective_capture or stop:
                with HiddenStateCapture(self.past_model, layers, detach=True, stop_after_last=stop) as cap:
                    self.past_model(**batch, output_hidden_states=False, return_dict=True)
                states = cap.hidden_states
            else:
                states = self.past_model(**batch, output_hidden_states=True, return_dict=True).hidden_states
        # no per-tensor `.detach()` (distillation.py:223): these come out of a no_grad forward, and the node never builds
        # a graph edge to a teacher tensor whatever its flags are
        return [self._as_teacher_dtype(states[l]) for l in layers]

    def _cached_past_states(self, batch, layers):
        """``teacher_cache``: the distilled layers' teacher states of the batch ``replay()`` drew, gathered from the cache
        (built here if ``load_state_dict`` left none) -- no teacher forward."""
        cache, idx, T = self._cache_step(batch, layers)
        return cache.gather(idx, T, layers)

    def _cache_step(self, batch, layers):
        """``(cache, memory indices, T)`` of the batch ``replay()`` drew: takes its ``memory_index`` and builds the cache
        if ``load_state_dict`` left none."""
        idx, self._memory_index = self._memory_index, None
        if idx is None:
            raise cabi.MafedDistillError(
                "teacher_cache: the batch has no memory_index (replay() takes it from the memory loader, which yields it "
                "with teacher_cache=True)")
        if self._teacher_cache is None:
            if self.past_model is None:
                raise cabi.MafedDistillError("teacher_cache: there is no teacher (past_model) to build the cache from")
            self._build_teacher_cache()
        return self._teacher_cache, idx, batch["attention_mask"].shape[1] + self.num_vision_tokens

    def _build_teacher_cache(self):
        from mafed_b200 import teacher_cache
        if self.shard_teacher_cache:
            self._build_sharded_teacher_cache()
            return
        self._teacher_cache = None              # the previous task's cache goes before the new one is allocated
        self._teacher_cache = teacher_cache.build(self)

    def _build_sharded_teacher_cache(self):
        """``shard_teacher_cache``: release the previous shards (collective: a peer's gather may still read this rank's
        shard until every rank has synchronised), then build this task's across the group, or the replicated cache
        when there is no group to shard over."""
        from mafed_b200 import teacher_cache
        old, self._teacher_cache, self._retired_cache = self._teacher_cache or self._retired_cache, None, None
        if isinstance(old, teacher_cache.ShardedTeacherCache):
            old.release()
        del old
        distributed, group = resolve_group(self.process_group)
        self._teacher_cache = teacher_cache.build_sharded(self, group) if distributed else teacher_cache.build(self)

    def _get_past_hidden_states(self, batch):
        with torch.no_grad(), self._teacher_forward(batch):
            batch.pop("labels", None)
            if self.selective_capture:
                layers = self.loss_weights.get_distillation_layers()
                with HiddenStateCapture(self.past_model, layers, detach=True) as cap:
                    self.past_model(**batch, output_hidden_states=False, return_dict=True)
                hs = cap.hidden_states
                if self.teacher_dtype is None:
                    return hs
                return HiddenStateTuple(len(hs), {l: self._as_teacher_dtype(hs[l]) for l in layers})
            states = self.past_model(**batch, output_hidden_states=True, return_dict=True).hidden_states
        return [self._as_teacher_dtype(h.detach()) for h in states]

    # ---- single-tensor token losses, kept for API compatibility (distillation.py:226-257)
    def _masked_token_loss(self, hidden_states, past_hidden_states, mask, loss_kind):
        dim = hidden_states.shape[-1]
        h = hidden_states.reshape(1, -1, dim)
        p = past_hidden_states.reshape(1, -1, dim)
        plan = DistillPlan(layers=[0], layer_coeffs=[1.0], distill_coeff=1.0, modality_kind=cabi.MODW_TEXT_ONLY,
                           loss_kind=loss_kind, n_vis=0)
        total, _ = distill_loss([h], [p.detach()], mask.reshape(1, -1), plan, group=False)
        return total

    def _compute_cosine_distillation_loss(self, hidden_states, past_hidden_states, mask):
        return self._masked_token_loss(hidden_states, past_hidden_states, mask, cabi.LOSS_COSINE)

    def _compute_mse_distillation_loss(self, hidden_states, past_hidden_states, mask):
        return self._masked_token_loss(hidden_states, past_hidden_states, mask, cabi.LOSS_MSE)

    def _compute_cls_distillation_loss(self, hidden_states, past_hidden_states):
        if self._loss_kind != cabi.LOSS_COSINE:
            raise TypeError("MSELoss.forward() takes 3 positional arguments but 4 were given")
        plan = DistillPlan(layers=[0], layer_coeffs=[1.0], distill_coeff=1.0, modality_kind=cabi.MODW_CLS,
                           loss_kind=self._loss_kind, cls=True, n_vis=self.num_vision_tokens)
        total, _ = distill_loss([hidden_states], [past_hidden_states.detach()], None, plan, group=False)
        return total

    # ------------------------------------------------------------------ logging without host syncs
    def _record(self, aux: torch.Tensor, layers: List[int]):
        """Keep the per-layer losses on the device; hand earlier steps' values to W&B once they have landed in
        pinned memory (the reference calls ``.item()`` per layer, ``distillation.py:165``).  Every step's values
        are logged, in order: a step whose copy has not completed yet stays queued."""
        self.last_layer_losses = aux
        self.last_layers = list(layers)
        if self.process_group is not False and _comm._cache:
            self.check_exchange(sync=False)
        if _wandb is None or getattr(_wandb, "run", None) is None:
            return
        if torch.cuda.is_current_stream_capturing():
            return      # inside a CUDA-graph capture: the values stay in `last_layer_losses` (static per replay)
        self.flush_logs(wait=False)
        host = torch.empty(len(layers), dtype=torch.float32, pin_memory=True)
        host.copy_(aux[: len(layers)], non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(aux.device))
        self._pending_logs.append((host, done, list(layers), self.task_id))
        while len(self._pending_logs) > 64:     # the host is far ahead of the device: wait for the oldest step
            self._flush_one(wait=True)

    def _flush_one(self, wait: bool) -> bool:
        host, done, layers, task_id = self._pending_logs[0]
        if not wait and not done.query():
            return False
        done.synchronize()
        self._pending_logs.popleft()
        if _wandb is not None and getattr(_wandb, "run", None) is not None:
            # one `wandb.log` per layer, like the reference (distillation.py:165): W&B's step axis advances L times
            # per replay step either way
            for l, v in zip(layers, host.tolist()):
                _wandb.log({f"task_{task_id}/distill_loss_{l}": float(v)})
        return True

    def flush_logs(self, wait: bool = True):
        """Send the queued per-layer values to W&B (``task_{id}/distill_loss_{layer}``), oldest first."""
        while self._pending_logs and self._flush_one(wait):
            pass

    def check_exchange(self, sync: bool = True):
        """Batch-sharded runs: raise if a peer missed an in-kernel exchange (that step's loss and gradients are NaN;
        every rank must run the same number of distillation steps).  The status word lives in mapped pinned host
        memory, so reading it costs nothing: ``distill`` does it every step (``sync=False``: it sees every step
        that has FINISHED, i.e. a missed exchange raises one step late at the latest, before the poisoned
        gradients can survive an optimizer step unnoticed); ``sync=True`` waits for the queued steps first."""
        group = self.process_group
        if group is False:
            return
        peer = _comm.peek_peer_comm(None if group is None or group is True else group)
        if peer is not None:
            if sync:
                torch.cuda.synchronize()
            peer.check()

    def layer_loss_dict(self) -> Dict[str, float]:
        """The reference's W&B payload for the last step (synchronises the host)."""
        if self.last_layer_losses is None:
            return {}
        vals = self.last_layer_losses[: len(self.last_layers)].tolist()
        self.check_exchange()
        return {f"task_{self.task_id}/distill_loss_{l}": v for l, v in zip(self.last_layers, vals)}

    # ------------------------------------------------------------------ checkpoint / resume
    def state_dict(self) -> Dict[str, object]:
        """Strategy state that the reference keeps only in the live Python object across the task loop
        (``train.py:207``; SURVEY 5 "checkpoint / resume"): task counter, step counter, the sampled memory
        indices per task, the sampling RNG, and the adaptive language coefficients."""
        coeff = getattr(self.loss_weights, "lang_coeff", None)
        return {
            "task_id": self.task_id,
            "step": self.step,
            "memory_indices": [np.asarray(ds.indices).tolist() for ds in self.datasets],
            "rng_state": self.rng.bit_generator.state,
            "lang_coeff": coeff.detach().cpu() if torch.is_tensor(coeff) else coeff,
        }

    def load_state_dict(self, state: Dict[str, object], datasets=None):
        """Restore ``state_dict()``.  ``datasets`` (one per finished task, in order) lets the episodic memory be
        rebuilt from the saved indices; the teacher snapshot itself comes from the model checkpoint
        (``_update_model``)."""
        self.task_id = int(state["task_id"])
        self.step = int(state["step"])
        self.rng.bit_generator.state = state["rng_state"]
        coeff = state.get("lang_coeff")
        if coeff is not None:
            if torch.is_tensor(coeff) and torch.cuda.is_available():
                coeff = coeff.cuda()     # `update_weights` averages it with importances computed on the device
            self.loss_weights.lang_coeff = coeff
            self.loss_weights._lang_coeff_host = None
        self._plan_cache = None
        if self.shard_teacher_cache:     # its shards are released collectively, by the rebuild
            self._retired_cache = self._teacher_cache or self._retired_cache
        self._teacher_cache = None      # not saved: rebuilt on the first replay, from the restored memory and teacher
        if datasets is not None:
            from torch.utils.data import Subset
            self.datasets = [Subset(ds, idx) for ds, idx in zip(datasets, state["memory_indices"])]
            if self.datasets:
                self._rebuild_loader()

    # ------------------------------------------------------------------ between tasks
    def _update_model(self, model):
        """Freeze a copy of the just-trained model as the next task's teacher (in ``teacher_dtype`` if set)."""
        self.past_model = deepcopy(model)
        if self.teacher_dtype is not None:
            self.past_model.to(self.teacher_dtype)
        self.past_model.eval()

    def _update_memory(self, dataset):
        """Add ``memory_per_task`` random samples of the finished task to the episodic memory and
        rebuild its loader (``distillation.py:182-209``).  Data loading itself is the reference's
        (``mafed.data``); it is imported lazily because it is outside this package's scope."""
        from torch.utils.data import Subset
        if hasattr(self, "mem_dataloader"):
            del self.mem_dataloader
        picked = self.rng.choice(np.arange(len(dataset)), self.memory_per_task, replace=False)
        assert len(set(picked)) == self.memory_per_task
        self.seed = 1
        self.datasets.append(Subset(dataset, picked))
        self._rebuild_loader()

    def _rebuild_loader(self):
        """(Re)create the memory loader over ``self.datasets`` (``distillation.py:192-209``)."""
        from torch.utils.data import ConcatDataset, DataLoader, RandomSampler
        from torch.utils.data.distributed import DistributedSampler
        import torch.distributed as dist

        memory = ConcatDataset(self.datasets)
        distributed = dist.is_available() and dist.is_initialized()
        sampler = DistributedSampler(memory) if distributed else RandomSampler(memory)
        collate, prefetch = self._data_hooks()
        data = memory
        if self.teacher_cache:
            # each batch also carries its samples' memory indices (a host list), which select their cached teacher rows
            from mafed_b200.teacher_cache import IndexedCollate, IndexedDataset
            data, collate = IndexedDataset(memory), IndexedCollate(collate)
        loader = DataLoader(data, sampler=sampler, num_workers=self.num_workers, batch_size=self.batch_size,
                            collate_fn=collate)
        self.mem_dataloader = prefetch(loader)
        self.mem_sampler = sampler

    def _data_hooks(self):
        hooks = getattr(self, "data_hooks", None)
        if hooks is not None:
            return hooks
        try:
            from mafed.data import PrefetchLoader, collate_fn
        except ImportError as exc:  # pragma: no cover - depends on the host installation
            raise ImportError(
                "FeatureDistillation._update_memory needs the reference's `mafed.data` (collate_fn, "
                "PrefetchLoader) or `self.data_hooks = (collate_fn, loader_wrapper)`") from exc
        return collate_fn["train"][self.model_type], PrefetchLoader
