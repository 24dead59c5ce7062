"""Helpers for the -m gpu parity tests: drive the product API exactly as the reference's callers do."""
import torch

from mafed_b200 import cabi
from mafed_b200.methods import CLMethod


class Opts:
    tasks = ["a", "b", "c"]
    batch_size = 4
    seed = 42
    pin_mem = False
    accumulate_grad_batches = 1


class Out:
    def __init__(self, hs):
        self.hidden_states = hs
        self.loss = None


def make_method(meta, **extra):
    fd = CLMethod["featdistill"](
        memory_size=8, opts=Opts(), model_type="vlpythia",
        distillation_modality_weighing_strategy=meta["modality"],
        distillation_layer_weighing_strategy=meta["layer_strategy"],
        distillation_coeff=meta.get("coeff", 1.0), distillation_layer=meta.get("layer"),
        cls_distillation=meta.get("cls", False), distillation_loss=meta["loss"], gamma=meta.get("gamma", 0.5),
        num_hidden_layers=meta["num_hidden_layers"], **extra)
    fd.num_vision_tokens = meta.get("n_vis", 256)
    if meta["modality"] == "adaptive":
        fd.loss_weights.lang_coeff = torch.tensor(meta["lang_coeff"], dtype=torch.float32, device="cuda")
    return fd


def run_product(meta, students, teachers, mask, grad_out=1.0, variant=cabi.VARIANT_DEFAULT, dev="cuda",
                single_pass=True, accumulate=1):
    """distill() + backward() on the GPU through the mirrored strategy API."""
    with cabi.tuning(variant=variant):
        fd = make_method(meta, single_pass=single_pass)
        fd.assumed_grad_out = 1.0 / accumulate
        st = [s.to(dev).detach().clone().requires_grad_(True) for s in students]
        te = [t.to(dev) for t in teachers]
        fd.past_model = lambda **kw: Out(tuple(te))
        batch = {"attention_mask": mask.to(dev), "labels": torch.zeros(1)}
        loss = fd.distill(Out(tuple(st)), batch)
        (loss * grad_out).backward()
        torch.cuda.synchronize()
        return dict(loss=loss.detach().float().cpu(), grads=[None if s.grad is None else s.grad.cpu() for s in st],
                    layer_dict=fd.layer_loss_dict(), batch=batch, fd=fd, students=st)


def reference_forward_backward(meta, students, teachers, mask, grad_out=1.0, autocast_bf16=False):
    """``distill()`` + ``backward()`` as the reference computes them, on the tensors' own device and under
    ``torch.autocast(bfloat16)`` if asked (as ``replay()`` runs it, ``distillation.py:90``).  This is the unmodified
    reference where its files are present (``oracle/_ref``, or the tree ``MAFED_REFERENCE`` names).  Elsewhere it is the
    oracle restatement, which runs the reference's torch ops in the same order and is held to vectors the reference
    produced by ``test_oracle_golden``.  Returns loss, the per-layer values sent to W&B, the gradients and the batch
    the step leaves behind."""
    from oracle import distill_oracle as O
    from oracle import ref_harness as R
    if R.available():
        fd = R.make_reference_method(modality=meta["modality"], layer_strategy=meta["layer_strategy"], loss=meta["loss"],
                                     gamma=meta["gamma"], num_hidden_layers=meta["num_hidden_layers"],
                                     layer=meta.get("layer"), coeff=meta.get("coeff", 1.0), n_vis=meta.get("n_vis", 256),
                                     lang_coeff=meta.get("lang_coeff"))
        if meta.get("lang_coeff") is not None:
            fd.loss_weights.lang_coeff = fd.loss_weights.lang_coeff.to(students[0].device)
        return R.reference_forward_backward(fd, students, teachers, mask, grad_out=grad_out, autocast_bf16=autocast_bf16)
    cfg = O.OracleConfig(modality_strategy=meta["modality"], layer_strategy=meta["layer_strategy"], gamma=meta["gamma"],
                         num_hidden_layers=meta["num_hidden_layers"], distillation_layer=meta.get("layer"),
                         distillation_coeff=meta.get("coeff", 1.0), loss=meta["loss"],
                         num_vision_tokens=meta.get("n_vis", 256), lang_coeff=meta.get("lang_coeff"))
    ref = O.forward_backward(students, teachers, mask, cfg, grad_out=grad_out, autocast_bf16=autocast_bf16)
    lang, image = O.build_masks(mask, cfg.num_vision_tokens)
    # the strategy's first task logs under task_0 (base.py; distillation.py:165 logs one value per layer)
    logged = {f"task_0/distill_loss_{l}": float(v) for l, v in ref["layer_losses"].items()}
    return {"loss": ref["loss"], "logged": logged, "grads": ref["grads"],
            "batch": {"attention_mask": mask, "lang_masks": lang, "image_masks": image}}


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def tolerances(dtype):
    """north_star: 1e-5 relative for fp32 inputs, 2e-3 for bf16 inputs (norm-wise for gradients)."""
    return (1e-5, 1e-5) if dtype == torch.float32 else (2e-3, 2e-3)
