"""Layer selection, layer coefficients and modality weights for the distillation loss.

Mirror of ``mafed/methods/distillation_loss_weights.py:9-174`` (same constructor, attributes and
getters).  The difference is where the numbers go: instead of being multiplied into per-layer
torch scalars, they are exported as small host tables (``kernel_tables``) that ride in the kernel
parameters of the fused epilogue -- no device tensors, no ``.item()`` per layer.
"""
from __future__ import annotations

import logging
from typing import List, Optional, Tuple

import torch

from mafed_b200 import cabi

LOGGER = logging.getLogger("mafed_b200")

_MODALITY_STRATEGIES = ("equal", "balanced", "adaptive")


class DistillationWeights:
    def __init__(
        self,
        distillation_modality_weighing_strategy="equal",
        distillation_layer_weighing_strategy="single",
        gamma: float = 0.9,
        num_hidden_layers: int = 11,
        distillation_layer: Optional[int] = -1,
        num_vision_tokens: int = 256,
    ) -> None:
        self._layer_coeff_method = "equal"
        self.gamma = gamma  # discount: the closer to 1, the flatter the per-layer weights
        self.num_vision_tokens = num_vision_tokens
        self._hidden_state_layer = distillation_layer
        self._modality_weighing_strategy = distillation_modality_weighing_strategy
        if distillation_modality_weighing_strategy == "balanced":
            self.lang_coeff = 0.5
        self._lang_coeff_host: Optional[List[float]] = None  # cached host copy for "adaptive"

        strategy = distillation_layer_weighing_strategy
        # reference :33-36 -- these two combinations are constructor errors
        if distillation_layer is None and strategy in ("single", "cumulative"):
            hint = "Use 'equal' or 'discounted' instead!" if strategy == "single" else \
                "Please pass the distillation layer!"
            raise AssertionError(f"Invalid layer weighting strategy '{strategy}'. {hint}")
        # reference :37-43 -- "cumulative" distils layers [0, layer); any other strategy given an
        # explicit layer collapses to "single"
        self.num_hidden_layers = distillation_layer if strategy == "cumulative" else num_hidden_layers
        if distillation_layer is not None and strategy != "cumulative":
            strategy = "single"
        self._layer_weighing_strategy = strategy
        self.prepare_layer_coeffs()
        LOGGER.info("Distillation layer weighting strategy: %s layer(s): %s", strategy,
                    self.get_distillation_layers())

    # ------------------------------------------------------------------ layers
    def prepare_layer_coeffs(self):
        """Per-layer loss coefficients (reference :49-60): ``None`` for single, uniform for equal,
        ``gamma ** (L - i)`` normalised for discounted / cumulative (last layer heaviest)."""
        n = self.num_hidden_layers
        if self._layer_weighing_strategy == "single":
            self.layer_coeffs = None
        elif self._layer_weighing_strategy == "equal":
            self.layer_coeffs = torch.full((n,), 1.0) / n
        else:
            # fp32 throughout, element by element as the reference does (`gamma ** 0-dim int64 tensor`)
            raw = torch.stack([torch.pow(self.gamma, d) for d in torch.arange(n, 0, -1)])
            self.layer_coeffs = raw / raw.sum()

    def get_distillation_layers(self) -> List[int]:
        if self._layer_weighing_strategy == "single":
            return [self._hidden_state_layer]
        return list(range(self.num_hidden_layers))

    def get_layer_loss_weight(self, layer: int):
        if self.layer_coeffs is None or self._layer_weighing_strategy == "single":
            return 1.0
        return self.layer_coeffs[layer]

    # ------------------------------------------------------------------ modalities
    def get_modality_loss_weights(self, batch, layer: int):
        """(language weight, vision weight) for one layer -- reference :71-79."""
        kind = self._modality_weighing_strategy
        if kind == "equal":
            return self._get_equal_loss_weights(batch)
        if kind == "balanced":
            return self._get_balanced_loss_weights()
        if kind == "adaptive":
            return self._get_adaptive_layer_loss_weights(layer)
        raise NotImplementedError

    def _get_equal_loss_weights(self, batch):
        n_text = batch["lang_masks"].sum()
        n_vis = batch["image_masks"].sum()
        n_all = n_text + n_vis
        return n_text / n_all, n_vis / n_all

    def _get_dynamic_loss_weights(self, loss_weights):
        if loss_weights is None:
            raise ValueError("Did not get loss weights from model")
        return loss_weights[0], 1 - loss_weights[0]

    def _get_balanced_loss_weights(self):
        return self.lang_coeff, (1 - self.lang_coeff)

    def _get_adaptive_layer_loss_weights(self, layer):
        coeff = self.lang_coeff
        lang = coeff.item() if coeff.shape[0] == 1 else coeff[layer].item()
        return lang, 1 - lang

    # ------------------------------------------------------------------ kernel tables
    def kernel_tables(self, layers: Optional[List[int]] = None) -> Tuple[List[float], int, Optional[List[float]]]:
        """Host tables for the fused epilogue: (layer coefficients, modality kind, language weights).

        ``adaptive`` reads ``lang_coeff`` once per change (one device->host copy per task, cached),
        not once per layer per step as ``_get_adaptive_layer_loss_weights`` does.
        """
        layers = self.get_distillation_layers() if layers is None else layers
        coeffs = [float(self.get_layer_loss_weight(l)) for l in layers]
        kind = self._modality_weighing_strategy
        if kind == "equal":
            return coeffs, cabi.MODW_EQUAL, None
        if kind == "balanced":
            return coeffs, cabi.MODW_TABLE, [float(self.lang_coeff)] * len(layers)
        if kind == "adaptive":
            host = self._adaptive_host_table()
            lang = [host[0] if len(host) == 1 else host[l] for l in layers]
            return coeffs, cabi.MODW_TABLE, lang
        raise NotImplementedError

    def _adaptive_host_table(self) -> List[float]:
        coeff = self.lang_coeff
        key = (id(coeff), getattr(coeff, "_version", 0))
        if self._lang_coeff_host is None or self._lang_coeff_key != key:
            self._lang_coeff_host = [float(x) for x in torch.as_tensor(coeff).detach().float().reshape(-1).cpu()]
            self._lang_coeff_key = key
        return self._lang_coeff_host

    # ------------------------------------------------------------------ adaptive importances
    def update_weights(self, model, dataloader, task_id, process_group=False):
        """Running average over tasks of the gradient-based language importance (reference :62-69).
        ``process_group``: see ``gradient_norm_sums``."""
        if self._modality_weighing_strategy != "adaptive":
            return
        fresh = self.compute_adaptive_weights(model, dataloader, process_group=process_group)
        if task_id < 1:
            self.lang_coeff = fresh
        else:
            self.lang_coeff = (fresh + task_id * self.lang_coeff) / (task_id + 1)
        self._lang_coeff_host = None

    def compute_adaptive_weights(self, model, dataloader, process_group=False):
        """Per-layer share of the LM-loss gradient norm that falls on text tokens (reference :91-146).

        For every batch: gradient of the LM loss w.r.t. each selected hidden state, per-token L2
        norm, masked sums per modality; finally ``lang / (lang + image)`` of the per-token means.
        ``process_group``: see ``gradient_norm_sums``.
        """
        L = len(self.get_distillation_layers())
        running = self.gradient_norm_sums(model, dataloader, process_group=process_group)
        sums = running[: 2 * L].reshape(L, 2)
        lang_imp = (sums[:, 0] / running[2 * L]).float()
        image_imp = (sums[:, 1] / running[2 * L + 1]).float()
        return lang_imp / (lang_imp + image_imp)

    def gradient_norm_sums(self, model, dataloader, process_group=False):
        """The totals behind ``compute_adaptive_weights``: device fp64 ``[2L + 2]``, per selected layer the sums of the
        per-token L2 norms of the LM-loss gradient over text and over vision tokens, then the two token counts, added
        over the batches of ``dataloader``.

        ``process_group``: ``False`` (the default) keeps them this process's own.  Otherwise (``None``: the default
        group, when one is initialised with more than one rank) the ranks' loaders are taken as the shards of one
        dataset: each rank adds its own batches, then the totals are exchanged once (an fp64 SUM-allreduce, the same
        on every rank), so every rank gets those of the union of the shards.  Every rank of the group must make the
        call (the exchange is a collective).  A ``DistributedSampler`` pads the last shard with repeated samples: the totals are then those of the
        padded union, which is what the ranks' loaders yield.
        """
        from mafed_b200.distill_op import allreduce_sums, modality_masks as device_masks, resolve_group, token_norm_sums

        model.eval()
        layers = self.get_distillation_layers()
        n_vis = self.num_vision_tokens
        running = None  # device fp64 [2L + 2]: per layer (text, vision) norm sums, then token counts
        for batch in dataloader:
            model.zero_grad()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                outputs = model(**batch, compute_loss=True, output_hidden_states=True,
                                allow_input_gradients=True, return_dict=True)
            attn = batch["attention_mask"]
            batch["lang_masks"], batch["image_masks"] = device_masks(attn, n_vis)
            states = [outputs.hidden_states[l] for l in layers]
            grads = torch.autograd.grad(outputs.loss, states, retain_graph=False, create_graph=False)
            # one fused pass over all L gradients instead of L x (norm, 2 masked sums)
            now = token_norm_sums(grads, attn, n_vis)
            running = now if running is None else running + now
        model.zero_grad()
        # the pass is additive over batches: one exchange of the totals, not one per batch
        distributed, pg = resolve_group(process_group)
        if distributed:
            allreduce_sums(running, pg)
        return running


def modality_masks(attention_mask: torch.Tensor, num_vision_tokens: int):
    """``[B, n_vis + txt]`` language / image masks on the mask's own device, without a host round trip
    (the reference builds both on the CPU and copies them over for every layer,
    ``distillation.py:134-144``)."""
    bsz = attention_mask.shape[0]
    pad = attention_mask.new_zeros((bsz, num_vision_tokens))
    lang = torch.cat([pad, attention_mask], dim=1)
    image = torch.cat([pad + 1, torch.zeros_like(attention_mask)], dim=1)
    return lang, image
