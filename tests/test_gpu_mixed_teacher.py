"""fp32 student hidden states distilled against a bf16 / fp16 teacher, read by the kernels as they are: the oracle on
the teacher up-cast to fp32, the same step on ``teacher.float()``, CLS mode, CUDA-graph replay, reproducibility,
``FeatureDistillation(teacher_dtype=...)`` and the batch-sharded step."""
import os
import re
import subprocess
import sys

import pytest
import torch

from golden_util import oracle_cfg
from gpu_util import Out, make_method, rel_err, run_product
from mafed_b200 import cabi
from oracle import distill_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TEACHERS = {"bf16": torch.bfloat16, "fp16": torch.float16}
META = dict(modality="balanced", layer_strategy="equal", gamma=0.5, num_hidden_layers=2, layer=None, n_vis=256,
            coeff=1.0, cls=False, lang_coeff=None)
# hidden size -> samples: base and 1B widths take the TMA ring; 100 (D % 8 == 4) the LDG family; 50 the generic
# kernels; 9216 (36 KB fp32 rows, above the ring's 32 KB) the LDG multi-pass class
SHAPES = {"base": (768, 3), "1B": (2048, 2), "D100": (100, 3), "D50": (50, 3), "D9216": (9216, 2)}
VARIANTS = {"ldg": cabi.VARIANT_LDG, "tma": cabi.VARIANT_DEFAULT}


def _inputs(shape, teacher_dtype, teacher="close", seed=71):
    D, B = SHAPES[shape]
    st, te, am = O.make_inputs(3, B, 32, D, n_vis=256, seed=seed, teacher=teacher, mask="ragged")
    return st, [t.to(teacher_dtype) for t in te], am


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("single_pass", [True, False], ids=["one-pass", "two-pass"])
@pytest.mark.parametrize("loss", ["mse", "cosine"])
@pytest.mark.parametrize("teacher", list(TEACHERS))
def test_matches_oracle_on_the_upcast_teacher(teacher, loss, single_pass, shape):
    meta = dict(META, loss=loss)
    # close teacher with the assumed upstream gradient (the gate skips); independent teacher with 0.25 (the gate
    # starts the exact backward, or the two-pass backward scales by it)
    for kind, grad_out in (("close", 1.0), ("independent", 0.25)):
        st, te, am = _inputs(shape, TEACHERS[teacher], teacher=kind)
        ref = O.forward_backward(st, [t.float() for t in te], am, oracle_cfg(meta), grad_out=grad_out)
        # a cosine loss is 1 - cos: with a close teacher (cos ~ 0.995) the subtraction cancels, and two fp32 sums of
        # 9216 products in different orders can differ by a few 1e-5 of the loss itself.  The tolerance is then 1e-5
        # relative to the loss at cos = 0, i.e. to cos
        scale = abs(float(ref["loss"])) if loss == "mse" else max(abs(float(ref["loss"])), 1.0)
        for variant in VARIANTS.values():
            out = run_product(meta, st, te, am, grad_out=grad_out, variant=variant, single_pass=single_pass)
            assert out["loss"].dtype == torch.float32
            assert abs(float(out["loss"]) - float(ref["loss"])) <= 1e-5 * scale, (kind, variant)
            for g, r in zip(out["grads"], ref["grads"]):
                assert (g is None) == (r is None)
                if r is not None:
                    assert g.dtype == torch.float32
                    assert rel_err(g, r) < 1e-5, (kind, variant)


# (shape, variant): pairs where the fp32 step and the paired step take the same kernel family
FAMILY_CASES = [("base", "tma"), ("base", "ldg"), ("1B", "tma"), ("D100", "ldg"), ("D50", "tma"), ("D9216", "tma")]


@pytest.mark.parametrize("shape,variant", FAMILY_CASES, ids=[f"{s}-{v}" for s, v in FAMILY_CASES])
@pytest.mark.parametrize("single_pass", [True, False], ids=["one-pass", "two-pass"])
@pytest.mark.parametrize("loss", ["mse", "cosine"])
@pytest.mark.parametrize("teacher", list(TEACHERS))
def test_same_results_as_the_step_on_teacher_float(teacher, loss, single_pass, shape, variant):
    """Widening a teacher value is exact and every per-element expression is the same: mse gradients are bit for bit
    those of the step on ``teacher.float()``.  The cosine row statistics and the loss sums come from another tile
    geometry, so their last bits may differ."""
    meta = dict(META, loss=loss)
    st, te, am = _inputs(shape, TEACHERS[teacher], teacher="independent")
    kw = dict(grad_out=0.25, variant=VARIANTS[variant], single_pass=single_pass)
    pair = run_product(meta, st, te, am, **kw)
    wide = run_product(meta, st, [t.float() for t in te], am, **kw)
    assert float(pair["loss"]) == pytest.approx(float(wide["loss"]), rel=1e-6)
    for g, w in zip(pair["grads"], wide["grads"]):
        if w is None:
            assert g is None
        elif loss == "mse":
            assert torch.equal(g, w)
        else:
            assert rel_err(g, w) < 1e-6


@pytest.mark.parametrize("teacher", list(TEACHERS))
def test_cls_mode(teacher):
    meta = dict(META, loss="cosine", cls=True)
    st, te, am = _inputs("base", TEACHERS[teacher], teacher="independent")
    ref = O.forward_backward(st, [t.float() for t in te], am, oracle_cfg(meta))
    for single_pass in (True, False):
        out = run_product(meta, st, te, am, single_pass=single_pass)
        assert float(out["loss"]) == pytest.approx(float(ref["loss"]), rel=1e-5)
        for g, r in zip(out["grads"], ref["grads"]):
            if r is not None:
                assert rel_err(g, r) < 1e-5


def test_bit_reproducible_run_to_run():
    for loss in ("mse", "cosine"):
        meta = dict(META, loss=loss)
        st, te, am = _inputs("base", torch.bfloat16, teacher="independent")
        a = run_product(meta, st, te, am, grad_out=0.25)
        b = run_product(meta, st, te, am, grad_out=0.25)
        assert torch.equal(a["loss"], b["loss"])
        for x, y in zip(a["grads"], b["grads"]):
            assert (x is None and y is None) or torch.equal(x, y)


def test_graphed_step_equals_eager_step():
    meta = dict(META, loss="mse", layer_strategy="discounted", num_hidden_layers=3)
    st, te, am = O.make_inputs(4, 3, 6, 768, n_vis=256, seed=31)
    te = [t.bfloat16() for t in te]
    fd = make_method(meta)
    step = fd.capture([s.cuda() for s in st], [t.cuda() for t in te], am.cuda().clone())
    assert step.teachers[0].dtype == torch.bfloat16 and step.students[0].dtype == torch.float32
    for trial, seed in enumerate((32, 33)):
        st2, te2, am2 = O.make_inputs(4, 3, 6, 768, n_vis=256, seed=seed, teacher="close" if trial else "independent")
        te2 = [t.bfloat16() for t in te2]
        with torch.no_grad():
            for dst, src in zip(step.students, st2):
                dst.copy_(src)
            for dst, src in zip(step.teachers, te2):
                dst.copy_(src)
            step.attention_mask.copy_(am2)
        loss = step.replay()
        torch.cuda.synchronize()
        fd_e = make_method(meta)
        fd_e.past_model = lambda **kw: Out(tuple(t.cuda() for t in te2))
        leaves = [s.cuda().requires_grad_(True) for s in st2]
        e_loss = fd_e.distill(Out(tuple(leaves)), {"attention_mask": am2.cuda()})
        e_loss.backward()
        torch.cuda.synchronize()
        assert torch.equal(loss, e_loss.detach())
        for l, g in zip(step.layers, step.grads):
            assert torch.equal(g, leaves[l].grad)
        ref = O.forward_backward(st2, [t.float() for t in te2], am2, oracle_cfg(meta))
        assert float(loss) == pytest.approx(float(ref["loss"]), rel=1e-5)


def _kernel_names(fn):
    """Names of the CUDA kernels ``fn`` launches (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


# a kernel of this library instantiated for an fp32 student and a half-precision teacher, demangled or mangled
_PAIR_KERNEL = re.compile(r"k_\w+<float, [^>]*(__nv_bfloat16|__half)>|k_\w+If\w*(13__nv_bfloat16|6__half)EE")
_FP32_KERNEL = re.compile(r"k_\w+<float, [0-9, ]+>")


def _assert_native(names):
    assert any(_PAIR_KERNEL.search(n) for n in names), sorted(names)
    assert not any(_FP32_KERNEL.search(n) for n in names), sorted(names)


@pytest.mark.parametrize("teacher", list(TEACHERS))
@pytest.mark.parametrize("single_pass", [True, False], ids=["one-pass", "two-pass"])
def test_pair_kernels_run_through_the_node_and_the_ctypes_path(teacher, single_pass):
    """The pair is not up-cast on the way: the compiled node and the ctypes sequence (what the NCCL path runs) both
    launch the pair kernels, and they agree bit for bit."""
    from mafed_b200.distill_op import DistillPlan, _DistillFunction, distill_loss
    st, te, am = _inputs("base", TEACHERS[teacher], teacher="independent")
    s = [x.cuda() for x in st[:2]]
    t = [x.cuda() for x in te[:2]]
    mask = am.cuda()
    plan = DistillPlan(layers=[0, 1], layer_coeffs=[0.25, 0.75], modality_kind=cabi.MODW_EQUAL, single_pass=single_pass)
    results = {}

    def node():
        leaves = [x.clone().requires_grad_(True) for x in s]
        total, _ = distill_loss(leaves, t, mask, plan, group=False)
        (total * 0.5).backward()
        results["node"] = (total.detach(), [x.grad for x in leaves])

    def ctypes_path():
        leaves = [x.clone().requires_grad_(True) for x in s]
        total, _ = _DistillFunction.apply(plan, mask, False, tuple(t), None, *leaves)
        (total * 0.5).backward()
        results["ctypes"] = (total.detach(), [x.grad for x in leaves])

    _assert_native(_kernel_names(node))
    _assert_native(_kernel_names(ctypes_path))
    assert torch.equal(results["node"][0], results["ctypes"][0])
    for a, b in zip(results["node"][1], results["ctypes"][1]):
        assert torch.equal(a, b)
    ref = O.forward_backward(st[:2], [x.float() for x in te[:2]], am,
                             O.OracleConfig(modality_strategy="equal", layer_strategy="discounted",
                                            num_hidden_layers=2, distillation_layer=None), grad_out=0.5)
    # (the oracle's discounted coefficients for 2 layers are not 0.25 / 0.75: weigh its per-layer losses by hand)
    want = sum(c * float(ref["layer_losses"][l]) for l, c in zip((0, 1), (0.25, 0.75)))
    assert float(results["node"][0]) == pytest.approx(want, rel=1e-5)


class _Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 2


@pytest.mark.parametrize("teacher", list(TEACHERS))
def test_feature_distillation_teacher_dtype_on_tiny_vl(teacher):
    """replay() with a half-precision teacher snapshot: the teacher forward runs under an autocast of the snapshot's
    dtype (also inside replay's bf16 region), every distilled teacher state comes out in that dtype, the step reads it
    natively, and the result is the reference's op chain on the states that teacher produced."""
    import copy
    from mafed_b200.methods import CLMethod
    from test_gpu_replay_e2e import _torch_replay
    from tiny_vl import TinyVL, make_batch
    dt = TEACHERS[teacher]
    torch.manual_seed(0)
    model = TinyVL().cuda()
    teacher_model = copy.deepcopy(model)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.02 * torch.randn_like(p))
    batch = make_batch(device="cuda")

    def make(**kw):
        fd = CLMethod["featdistill"](memory_size=8, opts=_Opts(), model_type="vlpythia",
                                     distillation_modality_weighing_strategy="balanced",
                                     distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                     distillation_loss="mse", gamma=0.5, num_hidden_layers=3, replay_coeff=1.0,
                                     distillation_coeff=2.0, **kw)
        fd.num_vision_tokens = 8
        fd.task_id = 1
        fd._update_model(teacher_model)
        fd.mem_dataloader = [dict(batch)]
        return fd

    assert all(p.dtype == torch.float32 for p in make().past_model.parameters())
    fd = make(teacher_dtype=dt)
    assert all(p.dtype == dt for p in fd.past_model.parameters())
    layers = fd.loss_weights.get_distillation_layers()
    coeffs = [float(fd.loss_weights.get_layer_loss_weight(l)) for l in layers]
    # the snapshot's own forward under an autocast of its dtype, every state in that dtype
    inputs = {k: v for k, v in batch.items() if k != "labels"}
    with torch.no_grad(), torch.autocast("cuda", dtype=dt):
        states = [h.to(dt) for h in fd.past_model(**inputs, output_hidden_states=True, return_dict=True).hidden_states]
    with torch.autocast("cuda", dtype=torch.bfloat16):     # replay's region
        got = fd._past_states(dict(batch), layers)
    assert all(g.dtype == dt and torch.equal(g, states[l]) for g, l in zip(got, layers))

    class _Teacher:
        hidden_states = states

    ref_model = copy.deepcopy(model)
    ref_loss = _torch_replay(ref_model, lambda **kw: _Teacher, batch, layers, coeffs, 8, 1.0, 2.0)
    (ref_loss / 2).backward()
    res = {}

    def step():
        loss, _ = fd.replay(model)
        (loss / 2).backward()
        res["loss"] = loss.detach()

    _assert_native(_kernel_names(step))
    assert float(res["loss"]) == pytest.approx(float(ref_loss), rel=1e-5)
    checked = 0
    for (name, p), (_, q) in zip(model.named_parameters(), ref_model.named_parameters()):
        if q.grad is not None:
            err = float((p.grad - q.grad).norm() / q.grad.norm().clamp_min(1e-20))
            assert err < 2e-4, (name, err)
            checked += 1
    assert checked > 10


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("path", ["peer", "nccl"])
def test_sharded_equals_one_gpu_on_the_concatenated_batch(path):
    """Both batch-sharded forms: the compiled node over the peer-memory communicator, and the NCCL sequence of
    ctypes calls (``_DistillFunction``)."""
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29519", os.path.join(ROOT, "tools", "multirank_check.py"),
           "--teacher-dtype", "bf16"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, MAFED_B200_DIST=path))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
