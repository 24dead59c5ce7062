"""Selective hidden-state capture (SURVEY.md 8f rank 2).

The reference asks the decoder for *all* hidden states (``output_hidden_states=True``,
``mafed/model/vl_pythia.py:298-308``; ``mafed/methods/distillation.py:91,222``) and keeps the whole
``L+1`` tuple alive for student and teacher even when one layer is distilled.  ``HiddenStateCapture``
records only the selected entries of that tuple with forward hooks, with the exact indexing of HF's
``GPTNeoXModel``: entry ``i < L`` is the input of decoder layer ``i`` (= output of layer ``i-1``; entry 0 is
the embedding output after dropout), entry ``L`` is the output of ``final_layer_norm``.

The captured student tensors are the graph's own tensors, so gradients of the distillation loss flow into
the model exactly as with ``output.hidden_states``.

With ``stop_after_last=True`` the forward ends as soon as the highest captured entry is stored: the decoder layers
after it, ``final_layer_norm`` (unless entry ``L`` is captured) and whatever the model computes from the decoder's output
(the LM head and its logits) never run, and the model call returns nothing.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence

import torch
from torch import nn


def find_decoder(model: nn.Module):
    """Locate (layers, final_norm) of a VL-Pythia style model: ``model.gpt_neox.layers`` and
    ``model.gpt_neox.final_layer_norm`` (``vl_pythia.py:204-237``), or a bare ``GPTNeoXModel``."""
    for root in (getattr(model, "gpt_neox", None), model, getattr(model, "model", None)):
        if root is None:
            continue
        layers = getattr(root, "layers", None)
        if isinstance(layers, nn.ModuleList):
            return layers, getattr(root, "final_layer_norm", None)
    raise AttributeError("cannot find decoder layers: pass `layer_modules=` explicitly")


class HiddenStateTuple(Sequence):
    """Read-only stand-in for ``output.hidden_states`` holding only the captured entries."""

    def __init__(self, length: int, states: Dict[int, torch.Tensor]):
        self._length = length
        self._states = states

    def __len__(self):
        return self._length

    def __getitem__(self, index):
        if isinstance(index, slice):
            return [self[i] for i in range(*index.indices(self._length))]
        if index < 0:
            index += self._length
        if index not in self._states:
            raise KeyError(f"hidden state {index} was not captured (captured: {sorted(self._states)})")
        return self._states[index]


class _StopForward(Exception):
    """Raised by the hook of the highest captured entry to end the forward there; ``args[0]`` is the capture that
    raised it, so that only its own ``__exit__`` suppresses it."""


class HiddenStateCapture:
    """Context manager: ``with HiddenStateCapture(model, layers) as cap: model(**batch)`` then
    ``cap.hidden_states[layer]``.

    ``stop_after_last=True``: the hook of the highest captured entry stores it and then stops the forward (for an entry
    ``i < L`` before decoder layer ``i`` runs, for entry ``L`` after ``final_layer_norm``).  ``__exit__`` suppresses only
    that stop; any other exception propagates.  The model call then returns nothing, so read the states from ``cap``."""

    def __init__(self, model: nn.Module, layers: Iterable[int], layer_modules: Optional[nn.ModuleList] = None,
                 final_norm: Optional[nn.Module] = None, detach: bool = False, stop_after_last: bool = False):
        if layer_modules is None:
            layer_modules, found_norm = find_decoder(model)
            final_norm = final_norm if final_norm is not None else found_norm
        self.layer_modules = layer_modules
        self.final_norm = final_norm
        self.n_states = len(layer_modules) + 1
        self.layers: List[int] = sorted({l if l >= 0 else l + self.n_states for l in layers})
        for l in self.layers:
            if not 0 <= l < self.n_states:
                raise IndexError(f"hidden state {l} out of range for a {len(layer_modules)}-layer decoder")
        if self.n_states - 1 in self.layers and final_norm is None:
            raise AttributeError("the last hidden state needs `final_norm=`")
        self.detach = detach
        self._stop_at = self.layers[-1] if stop_after_last and self.layers else None
        self.states: Dict[int, torch.Tensor] = {}
        self._handles = []

    def _store(self, index: int, tensor: torch.Tensor):
        self.states[index] = tensor.detach() if self.detach else tensor
        if index == self._stop_at:
            raise _StopForward(self)

    def __enter__(self):
        self.states.clear()
        last = self.n_states - 1
        for index in self.layers:
            if index == last:
                def post_hook(module, args, output, index=index):
                    self._store(index, output[0] if isinstance(output, tuple) else output)
                self._handles.append(self.final_norm.register_forward_hook(post_hook))
            else:
                def pre_hook(module, args, kwargs, index=index):
                    hidden = args[0] if args else kwargs["hidden_states"]
                    self._store(index, hidden)
                self._handles.append(self.layer_modules[index].register_forward_pre_hook(pre_hook, with_kwargs=True))
        return self

    def __exit__(self, exc_type, exc, tb):
        for h in self._handles:
            h.remove()
        self._handles.clear()
        return exc_type is _StopForward and exc.args[0] is self

    @property
    def hidden_states(self) -> HiddenStateTuple:
        return HiddenStateTuple(self.n_states, self.states)
