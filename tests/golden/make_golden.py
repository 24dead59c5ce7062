"""Generate golden vectors from the UNMODIFIED reference class.

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    python tests/golden/make_golden.py

Imports ``/root/reference/mafed/methods/distillation.py`` with ``sys.modules`` stubs for the
third-party packages that are absent here (``toolz``, ``pytorch_lightning``; SURVEY.md 8c) and a
recording ``wandb.log``; drives ``FeatureDistillation.distill`` + ``.backward()`` on CPU tensors;
writes ``tests/golden/distill_cases.npz`` (inputs + reference outputs) and
``tests/golden/layer_plans.json`` (layer lists / coefficients / constructor errors).
"""
import itertools
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def _install_stubs():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    mod("toolz")
    mod("toolz.sandbox", unzip=lambda s: zip(*s))

    class _WandbLogger:  # pragma: no cover - placeholder base class
        def __init__(self, *a, **k):
            pass

    def _identity(fn):
        return fn

    mod("pytorch_lightning")
    mod("pytorch_lightning.loggers", WandbLogger=_WandbLogger)
    mod("pytorch_lightning.utilities")
    mod("pytorch_lightning.utilities.rank_zero", rank_zero_only=_identity, rank_zero_warn=lambda *a, **k: None)
    sys.path.insert(0, REF)


class _Opts:
    tasks = ["a", "b", "c"]
    batch_size = 4
    seed = 42
    pin_mem = False
    accumulate_grad_batches = 1


class _Out:
    def __init__(self, hs):
        self.hidden_states = hs


def run_reference(case, students, teachers, am):
    import wandb
    from mafed.methods import CLMethod

    logged = {}
    wandb.log = lambda d, *a, **k: logged.update(d)
    fd = CLMethod["featdistill"](
        memory_size=8,
        opts=_Opts(),
        model_type="vlpythia",
        distillation_modality_weighing_strategy=case["modality"],
        distillation_layer_weighing_strategy=case["layer_strategy"],
        distillation_coeff=case["coeff"],
        distillation_layer=case["layer"],
        cls_distillation=case["cls"],
        distillation_loss=case["loss"],
        gamma=case["gamma"],
        num_hidden_layers=case["num_hidden_layers"],
    )
    fd.num_vision_tokens = case["n_vis"]  # public attribute (distillation.py:73)
    if case["modality"] == "adaptive":
        fd.loss_weights.lang_coeff = torch.tensor(case["lang_coeff"], dtype=torch.float32)
    fd.past_model = lambda **kw: _Out(tuple(teachers))
    st = [s.detach().clone().requires_grad_(True) for s in students]
    batch = {"attention_mask": am.clone(), "labels": torch.zeros(1)}
    import contextlib

    ctx = torch.autocast("cpu", dtype=torch.bfloat16) if case["dtype"] == "bf16" else contextlib.nullcontext()
    with ctx:
        loss = fd.distill(_Out(tuple(st)), batch)
    (loss * case["grad_out"]).backward()
    assert "labels" not in batch and ("lang_masks" in batch or case["cls"])
    return loss.detach(), logged, [s.grad for s in st]


def main():
    _install_stubs()
    sys.path.insert(0, os.path.join(HERE, "..", ".."))
    sys.path.insert(0, os.path.join(HERE, ".."))
    from golden_util import digest
    from oracle.distill_oracle import make_inputs

    cases = []
    base = dict(coeff=1.0, cls=False, gamma=0.5, num_hidden_layers=4, n_tuple=6, layer=None, grad_out=1.0,
                n_vis=8, txt=5, bsz=3, dim=32, dtype="fp32", teacher="close", lang_coeff=None)
    for modality, ls, loss in itertools.product(["equal", "balanced", "adaptive"],
                                                ["equal", "discounted"], ["mse", "cosine"]):
        c = dict(base, modality=modality, layer_strategy=ls, loss=loss)
        if modality == "adaptive":
            c["lang_coeff"] = [0.3, 0.6, 0.45, 0.8]
        cases.append(c)
    cases.append(dict(base, modality="balanced", layer_strategy="single", layer=2, loss="mse"))
    cases.append(dict(base, modality="equal", layer_strategy="cumulative", layer=3, loss="mse", coeff=0.7))
    cases.append(dict(base, modality="adaptive", layer_strategy="discounted", loss="mse", lang_coeff=[0.35]))
    cases.append(dict(base, modality="balanced", layer_strategy="discounted", loss="mse", grad_out=0.25,
                      teacher="independent"))
    cases.append(dict(base, modality="balanced", layer_strategy="discounted", loss="cosine", cls=True))
    # the real layout: 256 visual tokens
    cases.append(dict(base, modality="balanced", layer_strategy="discounted", loss="mse", n_vis=256, txt=7,
                      bsz=2, dim=16))
    cases.append(dict(base, modality="equal", layer_strategy="discounted", loss="cosine", n_vis=256, txt=7,
                      bsz=2, dim=16))
    # bf16 under autocast (distillation.py:90)
    for loss in ["mse", "cosine"]:
        cases.append(dict(base, modality="balanced", layer_strategy="discounted", loss=loss, dtype="bf16"))
        cases.append(dict(base, modality="equal", layer_strategy="equal", loss=loss, dtype="bf16",
                          grad_out=0.25, teacher="independent"))

    blob = {}
    meta = []
    for i, c in enumerate(cases):
        dtype = torch.bfloat16 if c["dtype"] == "bf16" else torch.float32
        st, te, am = make_inputs(c["n_tuple"], c["bsz"], c["txt"], c["dim"], n_vis=c["n_vis"], dtype=dtype,
                                 seed=1000 + i, teacher=c["teacher"], mask="ragged")
        loss, logged, grads = run_reference(c, st, te, am)
        # the inputs are regenerated from their seed when the file is read (golden_util.case_inputs): stored as a digest
        blob[f"c{i}_inputs_sha256"] = np.array(digest([s.float().numpy() for s in st] + [t.float().numpy() for t in te]))
        blob[f"c{i}_mask"] = am.numpy()
        blob[f"c{i}_loss"] = loss.float().numpy()
        sel = [j for j, g in enumerate(grads) if g is not None]
        blob[f"c{i}_grad_layers"] = np.array(sel, dtype=np.int64)
        blob[f"c{i}_grads"] = np.stack([grads[j].float().numpy() for j in sel])
        assert all(g.dtype == dtype for g in grads if g is not None)
        keys = sorted(logged, key=lambda k: int(k.rsplit("_", 1)[1]))
        blob[f"c{i}_logged_layers"] = np.array([int(k.rsplit("_", 1)[1]) for k in keys], dtype=np.int64)
        blob[f"c{i}_logged"] = np.array([logged[k] for k in keys], dtype=np.float64)
        meta.append(c)
        print(i, c["modality"], c["layer_strategy"], c["loss"], c["dtype"], float(loss), sel)
    blob["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(HERE, "distill_cases.npz"), **blob)

    # ---- layer plans / constructor behaviour (distillation_loss_weights.py:33-60,81-89)
    from mafed.methods.distillation_loss_weights import DistillationWeights

    plans = []
    for strat, layer, nh, gamma in [
        ("single", 2, 4, 0.5), ("equal", None, 4, 0.5), ("discounted", None, 4, 0.5), ("cumulative", 3, 4, 0.5),
        ("equal", 1, 4, 0.5), ("discounted", 0, 4, 0.9), ("single", None, 4, 0.5), ("cumulative", None, 4, 0.5),
        ("discounted", None, 11, 0.5), ("discounted", None, 15, 0.8), ("equal", None, 23, 0.9),
        ("cumulative", 7, 11, 0.7),
    ]:
        rec = dict(strategy=strat, layer=layer, num_hidden_layers=nh, gamma=gamma)
        try:
            dw = DistillationWeights("balanced", strat, gamma=gamma, num_hidden_layers=nh, distillation_layer=layer)
            ls = dw.get_distillation_layers()
            rec["layers"] = ls
            rec["coeffs"] = [float(dw.get_layer_loss_weight(l)) for l in ls]
            rec["effective"] = dw._layer_weighing_strategy
        except AssertionError:
            rec["error"] = "AssertionError"
        plans.append(rec)
    # distillation.py:61-64 resolution of the CLI's distillation_layer
    resolves = []
    for dl, nh in [(-1, 11), (None, 11), (0, 11), (10, 11), (11, 11), (5, 4)]:
        try:
            fd_kwargs = dict(memory_size=8, opts=_Opts(), model_type="x", distillation_layer=dl,
                             distillation_layer_weighing_strategy="equal", num_hidden_layers=nh)
            from mafed.methods import CLMethod

            fd = CLMethod["featdistill"](**fd_kwargs)
            resolves.append(dict(distillation_layer=dl, num_hidden_layers=nh,
                                 layers=fd.loss_weights.get_distillation_layers(),
                                 memory_per_task=fd.memory_per_task, update_freq=fd.update_freq))
        except AssertionError:
            resolves.append(dict(distillation_layer=dl, num_hidden_layers=nh, error="AssertionError"))
    with open(os.path.join(HERE, "layer_plans.json"), "w") as f:
        json.dump({"plans": plans, "resolves": resolves}, f, indent=1)
    print("wrote", len(cases), "cases,", len(plans), "plans")


if __name__ == "__main__":
    main()
