"""A step over layers of several dtypes, one launch per dtype group: against the same step on all-``.float()`` inputs
(the up-cast it replaces), against the reference under bf16 autocast, against each group run alone, one-pass and
two-pass, CLS, more than MAFED_MAX_LAYERS layers, CUDA-graph replay, torch.compile, no state-sized cast or copy,
``replay()`` and the adaptive importances on a bf16 model whose final-layer-norm entry is fp32, and the batch-sharded
step."""
import copy
import os
import subprocess
import sys

import pytest
import torch
from torch.utils._python_dispatch import TorchDispatchMode

from gpu_util import Out, make_method, reference_forward_backward, rel_err, run_product, tolerances
from mafed_b200 import cabi, node
from mafed_b200.distill_op import DistillPlan, distill_loss, dtype_groups
from oracle import distill_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
# (student dtypes, teacher dtypes) per entry of a 4-entry hidden-state tuple
CASES = {
    "bf16-model": ([BF16] * 3 + [F32], [BF16] * 3 + [F32]),          # the fp32 final-layer-norm entry of a bf16 model
    "fp16-model": ([F16] * 3 + [F32], [F16] * 3 + [F32]),
    "fp32-in-the-middle": ([BF16, F32, BF16, BF16], [BF16, F32, BF16, BF16]),
    "fp32-bf16-teacher": ([F32] * 4, [BF16, BF16, F32, BF16]),       # one fp32 teacher layer among bf16 ones
}
LOSSES = {"mse": cabi.LOSS_MSE, "cosine": cabi.LOSS_COSINE}


def _data(case, seed, n=4, D=768, bsz=3, txt=32):
    s_types, t_types = CASES[case] if n == 4 else case
    st, te, am = O.make_inputs(n, bsz, txt, D, n_vis=256, seed=seed, teacher="independent", mask="ragged")
    return ([s.to(d).cuda() for s, d in zip(st, s_types)], [t.to(d).cuda() for t, d in zip(te, t_types)], am.cuda())


def _plan(L, loss_kind, cls=False, single_pass=True):
    return DistillPlan(layers=list(range(L)), layer_coeffs=[0.5 + 0.25 * i for i in range(L)], distill_coeff=0.7,
                       modality_kind=cabi.MODW_CLS if cls else cabi.MODW_TABLE,
                       lang_weights=None if cls else [0.3 + 0.1 * (i % 5) for i in range(L)], loss_kind=loss_kind,
                       cls=cls, n_vis=256, single_pass=single_pass)


def _run(plan, st, te, am, grad_out, upcast=False):
    """distill_loss + backward; ``upcast``: the caller hands ``.float()`` copies of every state (the old path)."""
    leaves = [s.detach().clone().requires_grad_(True) for s in st]
    ins = [l.float() for l in leaves] if upcast else leaves
    teach = [t.float() for t in te] if upcast else te
    total, aux = distill_loss(ins, teach, am, plan, group=False)
    (total * grad_out).backward()
    torch.cuda.synchronize()
    return total.detach().clone(), aux.detach().clone(), [l.grad for l in leaves]


def _close(a, b, rel):
    return abs(float(a) - float(b)) <= rel * abs(float(b))


@pytest.mark.parametrize("grad_out", [1.0, 0.25], ids=["gate-skips", "gate-runs"])
@pytest.mark.parametrize("single_pass", [True, False], ids=["one-pass", "two-pass"])
@pytest.mark.parametrize("loss", list(LOSSES))
@pytest.mark.parametrize("case", list(CASES))
def test_same_results_as_the_upcast_step(case, loss, single_pass, grad_out):
    """mse: every gradient element is the same fp32 expression, rounded once to the student dtype either way, so the
    gradients are bit for bit those of the up-cast step; the loss sums come from other launches and tile geometries.
    cosine: the row statistics too, so within the dtype's tolerance."""
    st, te, am = _data(case, seed=81)
    plan = _plan(4, LOSSES[loss], single_pass=single_pass)
    got = _run(plan, st, te, am, grad_out)
    want = _run(plan, st, te, am, grad_out, upcast=True)
    assert got[0].dtype == F32 and got[1].shape == (12,)
    for g, w, s in zip(got[2], want[2], st):
        assert g.dtype == s.dtype == w.dtype
        if loss == "mse":
            assert torch.equal(g, w)
        else:
            assert rel_err(g, w) < tolerances(s.dtype)[1]
    rel = 1e-6 if loss == "mse" else 1e-5
    assert _close(got[0], want[0], rel)
    for a, b in zip(got[1].tolist(), want[1].tolist()):
        assert abs(a - b) <= rel * max(abs(b), 1e-3)


@pytest.mark.parametrize("loss", list(LOSSES))
@pytest.mark.parametrize("case", list(CASES))
def test_matches_the_reference_under_bf16_autocast(case, loss):
    meta = dict(modality="balanced", layer_strategy="discounted", loss=loss, gamma=0.5, num_hidden_layers=4,
                layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
    st, te, am = _data(case, seed=82)
    ref = reference_forward_backward(meta, st, te, am, grad_out=0.5, autocast_bf16=True)
    out = run_product(meta, st, te, am, grad_out=0.5)
    tol = tolerances(BF16)
    assert _close(out["loss"], ref["loss"], tol[0])
    for g, r in zip(out["grads"], ref["grads"]):
        assert g.dtype == r.dtype
        assert rel_err(g.float(), r.float().cpu()) < tol[1]


@pytest.mark.parametrize("single_pass", [True, False], ids=["one-pass", "two-pass"])
@pytest.mark.parametrize("loss", list(LOSSES))
@pytest.mark.parametrize("case", list(CASES))
def test_each_group_alone_gives_the_same_gradients_and_losses(case, loss, single_pass):
    st, te, am = _data(case, seed=83)
    plan = _plan(4, LOSSES[loss], single_pass=single_pass)
    total, aux, grads = _run(plan, st, te, am, 0.25)
    groups = dtype_groups([(s.dtype, t.dtype) for s, t in zip(st, te)])
    assert groups is not None and sorted(i for g in groups for i in g) == [0, 1, 2, 3]
    want_total = None
    for idx in groups:
        sub = DistillPlan(layers=idx, layer_coeffs=[plan.layer_coeffs[i] for i in idx], distill_coeff=plan.distill_coeff,
                          modality_kind=plan.modality_kind, lang_weights=[plan.lang_weights[i] for i in idx],
                          loss_kind=plan.loss_kind, n_vis=256, single_pass=single_pass)
        t_g, aux_g, grads_g = _run(sub, [st[i] for i in idx], [te[i] for i in idx], am, 0.25)
        want_total = t_g if want_total is None else want_total + t_g
        m = len(idx)
        for j, i in enumerate(idx):
            assert torch.equal(grads[i], grads_g[j])
            assert torch.equal(aux[i], aux_g[j])
            assert torch.equal(aux[4 + 2 * i:6 + 2 * i], aux_g[m + 2 * j:m + 2 * j + 2])
    assert torch.equal(total, want_total)


@pytest.mark.parametrize("case", ["bf16-model", "fp32-bf16-teacher"])
def test_cls_mode(case):
    st, te, am = _data(case, seed=84)
    for single_pass in (True, False):
        plan = _plan(4, cabi.LOSS_COSINE, cls=True, single_pass=single_pass)
        got = _run(plan, st, te, am, 0.25)
        want = _run(plan, st, te, am, 0.25, upcast=True)
        assert _close(got[0], want[0], 1e-5)
        for g, w, s in zip(got[2], want[2], st):
            assert g.dtype == s.dtype and rel_err(g, w) < tolerances(s.dtype)[1]


def test_more_layers_than_one_launch_carries():
    n = cabi.MAX_LAYERS + 6
    s_types = [BF16] * n
    s_types[3] = s_types[cabi.MAX_LAYERS + 2] = F32
    st, te, am = _data((s_types, s_types), seed=85, n=n, bsz=2, txt=4)
    for single_pass in (True, False):
        plan = _plan(n, cabi.LOSS_MSE, single_pass=single_pass)
        got = _run(plan, st, te, am, 0.25)
        want = _run(plan, st, te, am, 0.25, upcast=True)
        assert got[1].shape == (3 * n,)
        assert _close(got[0], want[0], 1e-6)
        for a, b in zip(got[1].tolist(), want[1].tolist()):
            assert abs(a - b) <= 1e-6 * max(abs(b), 1e-3)
        for g, w in zip(got[2], want[2]):
            assert torch.equal(g, w)


def test_graphed_step_equals_eager_step():
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=4,
                layer=None, n_vis=256, coeff=1.0, cls=False, lang_coeff=None)
    st, te, am = _data("fp32-in-the-middle", seed=86)
    fd = make_method(meta)
    step = fd.capture(st, te, am.clone(), grad_out=0.5)
    assert [s.dtype for s in step.students] == CASES["fp32-in-the-middle"][0]
    for seed in (87, 88):
        st2, te2, am2 = _data("fp32-in-the-middle", seed=seed)
        with torch.no_grad():
            for dst, src in zip(step.students + step.teachers, st2 + te2):
                dst.copy_(src)
            step.attention_mask.copy_(am2)
        loss = step.replay()
        torch.cuda.synchronize()
        fd_e = make_method(meta)
        fd_e.past_model = lambda **kw: Out(tuple(te2))
        leaves = [s.clone().requires_grad_(True) for s in st2]
        e_loss = fd_e.distill(Out(tuple(leaves)), {"attention_mask": am2})
        (e_loss * 0.5).backward()
        torch.cuda.synchronize()
        assert torch.equal(loss, e_loss.detach())
        assert torch.equal(step.layer_losses, fd_e.last_layer_losses)
        for l, g in zip(step.layers, step.grads):
            assert torch.equal(g, leaves[l].grad)


@pytest.mark.parametrize("grad_out", [1.0, 0.25], ids=["gate-skips", "gate-runs"])
@pytest.mark.parametrize("single_pass", [True, False], ids=["one-pass", "two-pass"])
@pytest.mark.parametrize("case", ["bf16-model", "fp32-bf16-teacher"])
def test_compiled_equals_eager_bit_for_bit(case, single_pass, grad_out):
    node.load()
    torch._dynamo.reset()
    plan = _plan(4, cabi.LOSS_MSE, single_pass=single_pass)

    def step(students, teachers, am):
        return distill_loss(students, teachers, am, plan, group=False, mask_out=True, return_masks=True)

    def run(fn, st, te, am):
        leaves = [s.detach().clone().requires_grad_(True) for s in st]
        total, aux, masks = fn(leaves, te, am)
        (total * grad_out).backward()
        torch.cuda.synchronize()
        return total.detach().clone(), aux.detach().clone(), masks, [l.grad for l in leaves]

    compiled = torch.compile(step, fullgraph=True)
    try:
        for seed in (89, 90):               # new data, same graph
            st, te, am = _data(case, seed=seed)
            b = run(step, st, te, am)           # (as FeatureDistillation does, an eager step comes first)
            a = run(compiled, st, te, am)
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
            assert torch.equal(a[2][0], b[2][0]) and torch.equal(a[2][1], b[2][1])
            for ga, gb in zip(a[3], b[3]):
                assert ga.dtype == gb.dtype and torch.equal(ga, gb)
    finally:
        torch._dynamo.reset()


class _StateSizedCopies(TorchDispatchMode):
    """Records every cast or copy op that takes a tensor of ``shape`` (the backward's ops included: autograd's worker
    thread runs under the caller's dispatch modes)."""

    def __init__(self, shape):
        super().__init__()
        self.shape, self.seen = tuple(shape), []

    def __torch_dispatch__(self, func, types, args=(), kwargs=None):
        if func.overloadpacket in (torch.ops.aten._to_copy, torch.ops.aten.copy_, torch.ops.aten.clone):
            if any(isinstance(a, torch.Tensor) and tuple(a.shape) == self.shape for a in args):
                self.seen.append(str(func))
        return func(*args, **(kwargs or {}))


def test_no_state_sized_cast_or_copy_and_less_memory_than_one_fp32_copy():
    """The groups read the states as they are: no cast or copy op takes a [B, T, D] tensor, and the step (gradients
    included) allocates less than one fp32 copy of the student states.  The old path did both."""
    st, te, am = _data("bf16-model", seed=91, D=2048, bsz=8, txt=32)
    fp32_copy = sum(s.numel() for s in st) * 4
    plan = _plan(4, cabi.LOSS_MSE)
    leaves = [s.detach().clone().requires_grad_(True) for s in st]
    for upcast in (False, True):
        for grad_out in (1.0, 0.25):
            for l in leaves:
                l.grad = None
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            with _StateSizedCopies(st[0].shape) as mode:
                ins = [l.float() for l in leaves] if upcast else leaves
                total, _ = distill_loss(ins, [t.float() for t in te] if upcast else te, am, plan, group=False)
                (total * grad_out).backward()
                del ins, total
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            if upcast:
                assert mode.seen and peak > fp32_copy, (mode.seen, peak)
            else:
                assert not mode.seen and peak < fp32_copy, (mode.seen, peak, fp32_copy)


# ---------------------------------------------------------------- a bf16 model: its final-layer-norm entry is fp32
class _Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 2


def _bf16_tiny_vl():
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    model = TinyVL().cuda().to(BF16)
    teacher = copy.deepcopy(model)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.02 * torch.randn_like(p))
    batch = make_batch(device="cuda")
    with torch.no_grad(), torch.autocast("cuda", dtype=BF16):
        hs = model(**batch, output_hidden_states=True).hidden_states
    assert [h.dtype for h in hs] == [BF16, BF16, BF16, F32]     # the mixed set this file is about
    return model, teacher, batch


@pytest.mark.parametrize("selective", [False, True], ids=["full-tuple", "selective-capture"])
def test_replay_on_a_bf16_model_with_the_final_layer_norm_entry(selective):
    from mafed_b200.methods import CLMethod
    from test_gpu_replay_e2e import _torch_replay
    model, teacher, batch = _bf16_tiny_vl()
    fd = CLMethod["featdistill"](memory_size=8, opts=_Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy="balanced",
                                 distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                 distillation_loss="mse", gamma=0.5, num_hidden_layers=4, replay_coeff=1.0,
                                 distillation_coeff=2.0, selective_capture=selective)
    fd.num_vision_tokens = 8
    fd.task_id = 1
    fd._update_model(teacher)
    fd.mem_dataloader = [dict(batch)]
    layers = fd.loss_weights.get_distillation_layers()
    assert layers == [0, 1, 2, 3]
    coeffs = [float(fd.loss_weights.get_layer_loss_weight(l)) for l in layers]
    ref_model = copy.deepcopy(model)
    ref_loss = _torch_replay(ref_model, teacher, batch, layers, coeffs, 8, 1.0, 2.0)
    (ref_loss / 2).backward()
    loss, n_ex = fd.replay(model)
    (loss / 2).backward()
    torch.cuda.synchronize()
    assert n_ex == 4
    assert float(loss) == pytest.approx(float(ref_loss), rel=1e-4)
    checked = 0
    for (name, p), (_, q) in zip(model.named_parameters(), ref_model.named_parameters()):
        if q.grad is None:
            assert p.grad is None, name
            continue
        err = float((p.grad.float() - q.grad.float()).norm() / q.grad.float().norm().clamp_min(1e-20))
        assert err < 1e-2, (name, err)
        checked += 1
    assert checked > 10
    assert fd.layer_loss_dict().keys() == {f"task_1/distill_loss_{l}" for l in layers}


def test_adaptive_importances_on_a_bf16_model():
    """compute_adaptive_weights over gradients of several dtypes, against the oracle's adaptive loop
    (``oracle.distill_oracle.adaptive_importances``) restated on the device under the same autocast."""
    from mafed_b200.methods import DistillationWeights
    from tiny_vl import make_batch
    model, _, _ = _bf16_tiny_vl()
    batches = [make_batch(seed=s, device="cuda") for s in (1, 2)]
    dw = DistillationWeights("adaptive", "equal", num_hidden_layers=4, distillation_layer=None, num_vision_tokens=8)
    imp = dw.compute_adaptive_weights(model, [dict(b) for b in batches])
    lang = image = None
    n_lang = n_image = 0.0
    for batch in batches:
        model.zero_grad()
        with torch.autocast("cuda", dtype=BF16):
            out = model(**dict(batch), compute_loss=True, output_hidden_states=True, allow_input_gradients=True)
        lang_mask, image_mask = O.build_masks(batch["attention_mask"], 8)
        la, ia = [], []
        for l in range(4):
            g = torch.autograd.grad(out.loss, out.hidden_states[l], retain_graph=True)[0]
            assert g.dtype == (F32 if l == 3 else BF16)
            norm = torch.linalg.norm(g.float(), dim=-1)
            la.append((norm * lang_mask).sum())
            ia.append((norm * image_mask).sum())
        la, ia = torch.stack(la), torch.stack(ia)
        lang = la if lang is None else lang + la
        image = ia if image is None else image + ia
        n_lang, n_image = n_lang + lang_mask.sum(), n_image + image_mask.sum()
    lang, image = lang / n_lang, image / n_image
    want = lang / (lang + image)
    torch.testing.assert_close(imp.cpu(), want.float().cpu(), rtol=1e-4, atol=0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("path", ["peer", "nccl"])
def test_sharded_equals_one_gpu_on_the_concatenated_batch(path):
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29523", os.path.join(ROOT, "tools", "multirank_check.py"),
           "--mixed-layers"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, MAFED_B200_DIST=path))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
