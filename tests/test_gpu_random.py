"""Seeded random sweep of shapes / dtypes / masks / strategies against the CPU oracle (both kernel families,
one-pass and two-pass)."""
import random

import pytest
import torch

from golden_util import oracle_cfg
from gpu_util import reference_forward_backward, rel_err, run_product, tolerances
from mafed_b200 import cabi
from oracle import distill_oracle as O

pytestmark = pytest.mark.gpu

DIMS = [8, 16, 24, 40, 64, 96, 100, 128, 200, 256, 384, 520, 768, 1000, 1024, 2048, 4104, 8192]


def _case(seed):
    r = random.Random(seed)
    dim = r.choice(DIMS)
    n_vis = r.choice([1, 5, 64, 256])
    cfg = dict(
        dim=dim, n_vis=n_vis, bsz=r.randint(1, 6 if dim <= 2048 else 2), txt=r.randint(1, 40),
        dtype=r.choice([torch.float32, torch.bfloat16, torch.float16]), loss=r.choice(["mse", "cosine"]),
        modality=r.choice(["equal", "balanced", "adaptive"]), nh=r.randint(1, 5),
        layer_strategy=r.choice(["equal", "discounted", "single", "cumulative"]), gamma=r.choice([0.5, 0.8, 0.9]),
        coeff=r.choice([1.0, 0.3, 2.0]), grad_out=r.choice([1.0, 1.0, 0.25, 3.0]), accumulate=r.choice([1, 1, 4]),
        single_pass=r.choice([True, True, False]), variant=r.choice([cabi.VARIANT_LDG, cabi.VARIANT_TMA]),
        mask=r.choice(["ragged", "full", "random", "sparse"]), teacher=r.choice(["close", "independent"]), seed=seed)
    cfg["layer"] = r.randint(0, cfg["nh"] - 1) if cfg["layer_strategy"] in ("single", "cumulative") else None
    if cfg["layer_strategy"] == "cumulative" and cfg["layer"] == 0:
        cfg["layer"] = 1 if cfg["nh"] > 1 else None
        if cfg["layer"] is None:
            cfg["layer_strategy"] = "equal"
    cfg["lang_coeff"] = [round(r.uniform(0.1, 0.9), 3) for _ in range(cfg["nh"])] if cfg["modality"] == "adaptive" else None
    return cfg


@pytest.mark.parametrize("seed", range(60))
def test_random_configuration(seed):
    c = _case(seed)
    st, te, am = O.make_inputs(c["nh"] + 1, c["bsz"], c["txt"], c["dim"], n_vis=c["n_vis"], dtype=c["dtype"],
                               seed=c["seed"], teacher=c["teacher"], mask="ragged" if c["mask"] == "ragged" else "full")
    g = torch.Generator().manual_seed(seed)
    if c["mask"] == "random":
        am = (torch.rand(am.shape, generator=g) > 0.4).long()
    elif c["mask"] == "sparse":
        am = torch.zeros_like(am)
        am[0, -1] = 1
    if int(am.sum()) == 0:
        am[0, -1] = 1                                               # keep the text loss finite
    meta = dict(modality=c["modality"], layer_strategy=c["layer_strategy"], loss=c["loss"], gamma=c["gamma"],
                num_hidden_layers=c["nh"], layer=c["layer"], n_vis=c["n_vis"], coeff=c["coeff"], cls=False,
                lang_coeff=c["lang_coeff"])
    ref = O.forward_backward(st, te, am, oracle_cfg(meta), grad_out=c["grad_out"])
    out = run_product(meta, st, te, am, grad_out=c["grad_out"], variant=c["variant"], single_pass=c["single_pass"],
                      accumulate=c["accumulate"])
    ltol, gtol = tolerances(c["dtype"])
    if c["dtype"] == torch.float16:
        ltol = gtol = 2e-3
    assert float(out["loss"]) == pytest.approx(float(ref["loss"]), rel=ltol, abs=1e-12), c
    for i, r in enumerate(ref["grads"]):
        if r is None:
            assert out["grads"][i] is None, c
            continue
        gpu = out["grads"][i]
        assert gpu.dtype == c["dtype"]
        if float(r.float().norm()) == 0.0:
            assert float(gpu.float().norm()) == 0.0
        else:
            assert rel_err(gpu.float(), r.float()) <= gtol, (c, i)
        zero_rows = r.float().abs().amax(-1) == 0
        assert bool((gpu.float().abs().amax(-1)[zero_rows] == 0).all()), c


@pytest.mark.parametrize("seed", range(100, 132))
def test_random_configuration_against_the_reference_on_this_gpu(seed):
    """The same sweep against the reference's computation run on this GPU on the same tensors -- under
    ``torch.autocast("cuda", bfloat16)`` for bf16 inputs, as ``replay()`` runs it (``distillation.py:90``): the
    like-for-like check of SURVEY 8(c).  The unmodified reference where its files are present, otherwise its op-for-op
    restatement (``gpu_util.reference_forward_backward``)."""
    c = _case(seed)
    if c["dtype"] == torch.float16:
        c["dtype"] = torch.bfloat16                                 # (the reference never feeds fp16)
    st, te, am = O.make_inputs(c["nh"] + 1, c["bsz"], c["txt"], c["dim"], n_vis=c["n_vis"], dtype=c["dtype"],
                               seed=c["seed"], teacher=c["teacher"], mask="ragged" if c["mask"] == "ragged" else "full")
    if c["mask"] in ("random", "sparse"):
        am = (torch.rand(am.shape, generator=torch.Generator().manual_seed(seed)) > 0.4).long()
    if int(am.sum()) == 0:
        am[0, -1] = 1
    meta = dict(modality=c["modality"], layer_strategy=c["layer_strategy"], loss=c["loss"], gamma=c["gamma"],
                num_hidden_layers=c["nh"], layer=c["layer"], n_vis=c["n_vis"], coeff=c["coeff"], cls=False,
                lang_coeff=c["lang_coeff"])
    ref = reference_forward_backward(meta, [s.cuda() for s in st], [t.cuda() for t in te], am.cuda(),
                                     grad_out=c["grad_out"], autocast_bf16=c["dtype"] != torch.float32)
    out = run_product(meta, st, te, am, grad_out=c["grad_out"], variant=c["variant"], single_pass=c["single_pass"],
                      accumulate=c["accumulate"])
    ltol, gtol = tolerances(c["dtype"])
    assert float(out["loss"]) == pytest.approx(float(ref["loss"]), rel=ltol, abs=1e-12), c
    # the masks the reference leaves in `batch` (distillation.py:139,144) and the values it sends to W&B (:165)
    assert torch.equal(out["batch"]["lang_masks"].cpu(), ref["batch"]["lang_masks"].cpu().long())
    assert torch.equal(out["batch"]["image_masks"].cpu(), ref["batch"]["image_masks"].cpu().long())
    assert "labels" not in out["batch"] and "labels" not in ref["batch"]
    mine = out["layer_dict"]
    assert sorted(mine) == sorted(ref["logged"]), c
    for k, v in ref["logged"].items():
        assert mine[k] == pytest.approx(v, rel=ltol, abs=1e-12), (c, k)
    for i, r in enumerate(ref["grads"]):
        if r is None:
            assert out["grads"][i] is None, c
            continue
        gpu = out["grads"][i]
        assert gpu.dtype == c["dtype"]
        assert rel_err(gpu.float(), r.float().cpu()) <= gtol, (c, i)
