"""The step under torch.compile (the ``mafed::`` ops): opcheck, bit-identical results against the eager node, no graph
break, CUDA-graph replay, the same kernels as eager without a gradient-sized copy, bounded recompiles, the eager
bookkeeping call, and the sharded step on 2 GPUs."""
import os
import re
import subprocess
import sys

import pytest
import torch

from gpu_util import Out, make_method
from oracle import distill_oracle as O

from mafed_b200 import cabi, node
from mafed_b200.distill_op import DistillPlan, distill_loss

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(autouse=True)
def _fresh_dynamo():
    node.load()
    torch._dynamo.reset()
    yield
    torch._dynamo.reset()


def _plan(L, loss_kind, cls=False, single_pass=True, assumed=1.0):
    return DistillPlan(layers=list(range(L)), layer_coeffs=[0.5 + 0.25 * i for i in range(L)], distill_coeff=0.7,
                       modality_kind=cabi.MODW_CLS if cls else cabi.MODW_TABLE,
                       lang_weights=None if cls else [0.3 + 0.1 * i for i in range(L)], loss_kind=loss_kind, cls=cls,
                       n_vis=256, single_pass=single_pass, assumed_grad_out=assumed)


def _data(L, dtype, t_dtype, seed, D=768, bsz=4, txt=9):
    st, te, am = O.make_inputs(L, bsz, txt, D, n_vis=256, dtype=torch.float32, seed=seed)
    return ([s.to(dtype).cuda() for s in st], [t.to(t_dtype).cuda() for t in te], am.cuda())


def _run(fn, st, te, am, grad_out):
    leaves = [s.detach().clone().requires_grad_(i != 1) for i, s in enumerate(st)]     # layer 1 needs no gradient
    total, aux, masks = fn(leaves, te, am)
    (total * grad_out).backward()
    torch.cuda.synchronize()
    return total.detach().clone(), aux.detach().clone(), masks, [l.grad for l in leaves]


def _step_fn(plan):
    def f(students, teachers, am):
        return distill_loss(students, teachers, am, plan, group=False, mask_out=True, return_masks=True)
    return f


def _assert_same(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    if a[2] is not None or b[2] is not None:
        assert torch.equal(a[2][0], b[2][0]) and torch.equal(a[2][1], b[2][1])
    for ga, gb in zip(a[3], b[3]):
        assert (ga is None) == (gb is None)
        if ga is not None:
            assert ga.dtype == gb.dtype and torch.equal(ga, gb)


# ---------------------------------------------------------------- opcheck
def test_opcheck_each_op():
    L = 2
    st, te, am = _data(L, torch.float32, torch.float32, seed=5, D=256)
    plan = (cabi.MODW_TABLE, 1.0, cabi.LOSS_MSE, False, 256)
    args = ([1.0, 0.5], [0.4, 0.6]) + plan
    leaves = [s.clone().requires_grad_(True) for s in st]
    # (the AOT-dispatch check calls the backward of an op with Tensor[] inputs directly, which torch does not
    # support; the compiled-step tests below run that path through torch.compile instead)
    utils = ("test_schema", "test_autograd_registration", "test_faketensor")
    torch.library.opcheck(torch.ops.mafed.step.default,
                          (leaves, te, am, *args, 1.0, 1.0, [True, True], 0, True, 0), test_utils=utils)
    torch.library.opcheck(torch.ops.mafed.fwd_step.default,
                          (leaves, te, am, *args, 1.0, [True, True], 0, True, 0), test_utils=utils)
    out, grads, scale, _ = torch.ops.mafed.step(st, te, am, *args, 1.0, 1.0, [True, True], 0, False, 0)
    gout = torch.full((), 0.5, device="cuda")
    torch.library.opcheck(torch.ops.mafed.bwd.default,
                          (st, te, am, grads.clone(), scale, gout, 1.0, 1.0, [True, True], cabi.LOSS_MSE, False, 256, 0))
    torch.library.opcheck(torch.ops.mafed.bwd.default,
                          (st, te, am, torch.empty_like(grads), scale, gout, 1.0, None, [True, True], cabi.LOSS_MSE,
                           False, 256, 0))


# ---------------------------------------------------------------- compiled == eager, bit for bit
PAIRS = [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16), (torch.float32, torch.bfloat16)]


@pytest.mark.parametrize("grad_out", [1.0, 0.25])
@pytest.mark.parametrize("single_pass", [True, False])
@pytest.mark.parametrize("pair", PAIRS, ids=["fp32", "bf16", "fp32-bf16"])
@pytest.mark.parametrize("loss_kind", [cabi.LOSS_MSE, cabi.LOSS_COSINE], ids=["mse", "cosine"])
def test_compiled_equals_eager_bit_for_bit(loss_kind, pair, single_pass, grad_out):
    L = 3
    plan = _plan(L, loss_kind, single_pass=single_pass)
    st, te, am = _data(L, *pair, seed=11)
    eager = _run(_step_fn(plan), st, te, am, grad_out)
    compiled = _run(torch.compile(_step_fn(plan), fullgraph=True), st, te, am, grad_out)
    _assert_same(compiled, eager)
    st, te, am = _data(L, *pair, seed=12)          # new data, same graph
    _assert_same(_run(torch.compile(_step_fn(plan), fullgraph=True), st, te, am, grad_out),
                 _run(_step_fn(plan), st, te, am, grad_out))


@pytest.mark.parametrize("grad_out", [1.0, 0.25])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_compiled_cls_equals_eager(dtype, grad_out):
    L = 2
    plan = _plan(L, cabi.LOSS_COSINE, cls=True)
    st, te, am = _data(L, dtype, dtype, seed=13)
    _assert_same(_run(torch.compile(_step_fn(plan), fullgraph=True), st, te, am, grad_out),
                 _run(_step_fn(plan), st, te, am, grad_out))


def test_compiled_chunked_step_above_the_layer_limit_equals_eager():
    L = cabi.MAX_LAYERS + 2
    plan = _plan(L, cabi.LOSS_MSE)
    st, te, am = _data(L, torch.bfloat16, torch.bfloat16, seed=14, D=64, bsz=2, txt=4)
    _assert_same(_run(torch.compile(_step_fn(plan), fullgraph=True), st, te, am, 1.0),
                 _run(_step_fn(plan), st, te, am, 1.0))


# ---------------------------------------------------------------- no graph break
def test_explain_reports_no_graph_break_for_distill_loss():
    plan = _plan(3, cabi.LOSS_MSE)
    st, te, am = _data(3, torch.bfloat16, torch.bfloat16, seed=15)
    leaves = [s.requires_grad_(True) for s in st]
    exp = torch._dynamo.explain(_step_fn(plan))(leaves, te, am)
    assert exp.graph_break_count == 0 and exp.graph_count == 1, exp.break_reasons


def _tiny_vl_setup():
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    model = TinyVL(n_vis=256, dim=256, layers=3).cuda()
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=4,
                layer=None, n_vis=256)
    fd = make_method(meta)
    fd.past_model = TinyVL(n_vis=256, dim=256, layers=3).cuda().eval()
    fd.past_model.load_state_dict(model.state_dict())
    with torch.no_grad():
        for p in fd.past_model.parameters():
            p.add_(0.01 * torch.randn_like(p))
    return model, fd, make_batch


def test_explain_reports_no_graph_break_for_feature_distillation_on_the_tiny_vl_model():
    model, fd, make_batch = _tiny_vl_setup()
    batch = make_batch(bsz=4, txt=6, n_vis=256, device="cuda")
    batch.pop("labels")

    out = model(**batch, output_hidden_states=True)
    fd.distill(out, dict(batch))                     # eager first: plan cache
    exp = torch._dynamo.explain(fd.distill)(out, dict(batch))     # the teacher forward runs inside distill
    assert exp.graph_break_count == 0, exp.break_reasons


def test_feature_distillation_compiled_with_the_model_equals_eager():
    model, fd, make_batch = _tiny_vl_setup()
    fd.adapt_assumed_grad_out = False

    def step(batch):
        out = model(**batch, output_hidden_states=True)
        return fd.distill(out, batch)

    compiled = torch.compile(step)
    for seed in (1, 2):
        batch = make_batch(bsz=4, txt=6, n_vis=256, seed=seed, device="cuda")
        batch.pop("labels")
        model.zero_grad(set_to_none=True)
        e_batch = dict(batch)
        e_loss = step(e_batch)
        e_loss.backward()
        e_loss = e_loss.detach().clone()
        e_grads = [None if p.grad is None else p.grad.clone() for p in model.parameters()]
        model.zero_grad(set_to_none=True)
        c_batch = dict(batch)
        c_loss = compiled(c_batch)
        c_loss.backward()
        torch.cuda.synchronize()
        # the model's own kernels may differ between eager and Inductor; the distillation term's inputs are the same
        assert float(c_loss) == pytest.approx(float(e_loss), rel=1e-4)
        for p, g in zip(model.parameters(), e_grads):
            assert (p.grad is None) == (g is None)
            assert g is None or torch.allclose(p.grad, g, rtol=1e-3, atol=1e-5)
        assert torch.equal(c_batch["lang_masks"], e_batch["lang_masks"])
        assert torch.equal(c_batch["image_masks"], e_batch["image_masks"])
        assert fd.last_layer_losses.shape == (3 * len(fd.last_layers),)


# ---------------------------------------------------------------- CUDA-graph replay
class _GraphCount:
    """Counts CUDA-graph captures and replays (the CUDA-graph trees of reduce-overhead use torch.cuda.CUDAGraph)."""

    def __init__(self, monkeypatch):
        self.captures = self.replays = 0
        cls = torch.cuda.graphs.CUDAGraph
        capture_begin, replay = cls.capture_begin, cls.replay

        def counted_capture(graph, *args, **kwargs):
            self.captures += 1
            return capture_begin(graph, *args, **kwargs)

        def counted_replay(graph):
            self.replays += 1
            return replay(graph)

        monkeypatch.setattr(cls, "capture_begin", counted_capture)
        monkeypatch.setattr(cls, "replay", counted_replay)


def _assert_replayed(history, settle=3):
    """history: (captures, replays) after each step.  After `settle` steps nothing is captured any more, and every
    later step replays the forward and the backward graph."""
    settled = history[settle - 1][0]
    assert settled >= 1, history
    for (c0, r0), (c1, r1) in zip(history[settle - 1:], history[settle:]):
        assert c1 == settled and r1 >= r0 + 2, history


@pytest.mark.parametrize("single_pass", [True, False])
def test_reduce_overhead_replays_over_fresh_inputs_and_matches_eager(single_pass, monkeypatch):
    from torch._dynamo.utils import counters
    L = 3
    plan = _plan(L, cabi.LOSS_MSE, single_pass=single_pass)

    def f(students, teachers, am):
        return distill_loss(students, teachers, am, plan, group=False)

    compiled = torch.compile(f, mode="reduce-overhead", fullgraph=True)
    counters.clear()
    count = _GraphCount(monkeypatch)
    history = []
    for seed in range(20, 30):
        st, te, am = _data(L, torch.bfloat16, torch.bfloat16, seed=seed)
        leaves = [s.detach().clone().requires_grad_(True) for s in st]
        total, aux = compiled(leaves, te, am)
        c_total, c_aux = total.detach().clone(), aux.clone()
        total.backward()
        c = (c_total, c_aux, [l.grad.clone() for l in leaves])
        history.append((count.captures, count.replays))
        eleaves = [s.detach().clone().requires_grad_(True) for s in st]
        et, ea = distill_loss(eleaves, te, am, plan, group=False)
        et.backward()
        torch.cuda.synchronize()
        assert torch.equal(c[0], et.detach()) and torch.equal(c[1], ea)
        for g, l in zip(c[2], eleaves):
            assert torch.equal(g, l.grad)
    assert counters["inductor"]["cudagraph_skips"] == 0
    _assert_replayed(history)


_FD = None      # the strategy as a module-level global, as a training script holds it


def _global_step(students, batch):
    return _FD.distill(Out(tuple(students)), batch)


@pytest.mark.parametrize("mode", [None, "reduce-overhead"])
@pytest.mark.parametrize("holder", ["global", "closure"])
def test_compiled_feature_distillation_neither_recompiles_nor_rerecords_per_step(holder, mode, monkeypatch):
    """fd.distill compiled with fullgraph=True over more steps than Dynamo's recompile limit: one graph, no per-step
    guard on the strategy's state, and with reduce-overhead a CUDA graph that is replayed, not re-recorded."""
    global _FD
    from torch._dynamo.utils import counters
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256)
    fd = make_method(meta)
    fd.adapt_assumed_grad_out = False
    st, te, am = _data(3, torch.bfloat16, torch.bfloat16, seed=60)
    fd.past_model = lambda **kw: Out(tuple(te))
    fd.distill(Out(tuple(s.clone().requires_grad_(True) for s in st)), {"attention_mask": am})   # eager: plan tables
    if holder == "global":
        _FD = fd
        step = _global_step
    else:
        def step(students, batch):
            return fd.distill(Out(tuple(students)), batch)
    compiled = torch.compile(step, fullgraph=True, mode=mode)
    counters.clear()
    count = _GraphCount(monkeypatch)
    history = []
    steps = torch._dynamo.config.recompile_limit + 4
    try:
        for i in range(steps):
            s_i = [(s * (1 + 0.01 * i)).requires_grad_(True) for s in st]
            loss = compiled(s_i, {"attention_mask": am})
            value = loss.detach().clone()
            loss.backward()
            grads = [s.grad.clone() for s in s_i]
            fd.record_step()
            history.append((count.captures, count.replays))
        # the last step against an eager step of a fresh strategy on the same inputs
        ref = make_method(meta)
        ref.past_model = fd.past_model
        e_i = [(s * (1 + 0.01 * (steps - 1))).requires_grad_(True) for s in st]
        e_loss = ref.distill(Out(tuple(e_i)), {"attention_mask": am})
        e_loss.backward()
        torch.cuda.synchronize()
        assert torch.equal(value, e_loss.detach())
        for g, e in zip(grads, e_i):
            assert torch.equal(g, e.grad)
    finally:
        _FD = None
    assert counters["stats"]["unique_graphs"] == 1, dict(counters["stats"])
    assert fd.step == 1 + steps                      # advanced by record_step(), outside the graph
    if mode == "reduce-overhead":
        assert counters["inductor"]["cudagraph_skips"] == 0
        _assert_replayed(history)


# ---------------------------------------------------------------- same kernels, no gradient-sized copy
def _kernels(fn, *args):
    from torch.profiler import ProfilerActivity, profile
    fn(*args)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        fn(*args)
        torch.cuda.synchronize()
    return [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("single_pass", [True, False])
def test_profile_lists_the_eager_kernels_and_no_gradient_sized_copy(single_pass):
    L = 3
    plan = _plan(L, cabi.LOSS_MSE, single_pass=single_pass)
    st, te, am = _data(L, torch.bfloat16, torch.bfloat16, seed=30)
    leaves = [s.requires_grad_(True) for s in st]

    def step(students):
        return distill_loss(students, te, am, plan, group=False)[0]

    def run(fn):
        for l in leaves:
            l.grad = None
        fn(leaves).backward()

    eager = _kernels(run, step)
    compiled = _kernels(run, torch.compile(step, fullgraph=True))
    ours = lambda evs: sorted(e.name for e in evs if re.search(r"\bk_(fwd|bwd|gate|epilogue|modality)", e.name))
    assert ours(eager) and ours(compiled) == ours(eager), (ours(compiled), ours(eager))
    copies = [e.name for e in compiled if re.search(r"clone|memcpy|copy_kernel|_copy", e.name, re.IGNORECASE)]
    assert not copies, copies


# ---------------------------------------------------------------- recompiles
def test_a_changed_assumed_gradient_recompiles_a_bounded_number_of_times():
    from torch._dynamo.utils import counters
    L = 2
    st, te, am = _data(L, torch.float32, torch.float32, seed=40, D=256)
    plans = {a: _plan(L, cabi.LOSS_MSE, assumed=a) for a in (1.0, 0.5, 0.25)}

    def f(students, plan):
        return distill_loss(students, te, am, plan, group=False)[0]

    compiled = torch.compile(f, fullgraph=True)
    counters.clear()
    for _ in range(3):
        for a, plan in plans.items():
            leaves = [s.clone().requires_grad_(True) for s in st]
            compiled(leaves, plan).backward()
    frames = counters["stats"]["unique_graphs"]
    assert frames <= len(plans), dict(counters["stats"])


def test_a_step_traced_inside_a_tuning_block_is_retraced_after_it():
    """The tuning address is guarded on: leaving the `cabi.tuning` block retraces instead of handing the library the
    address of a freed table."""
    from torch._dynamo.utils import counters
    plan = _plan(2, cabi.LOSS_MSE)
    st, te, am = _data(2, torch.bfloat16, torch.bfloat16, seed=45, D=512)
    compiled = torch.compile(_step_fn(plan), fullgraph=True)
    counters.clear()
    with cabi.tuning(variant=cabi.VARIANT_LDG):
        inside = _run(compiled, st, te, am, 1.0)
        assert _run(compiled, st, te, am, 1.0)[0].equal(inside[0])
    assert counters["stats"]["unique_graphs"] == 1
    outside = _run(compiled, st, te, am, 1.0)
    assert counters["stats"]["unique_graphs"] == 2
    _assert_same(outside, _run(_step_fn(plan), st, te, am, 1.0))


# ---------------------------------------------------------------- the eager bookkeeping call
def test_record_step_keeps_the_logging_contract(monkeypatch):
    import mafed_b200.methods.distillation as D
    logged = []

    class FakeWandb:
        run = object()

        @staticmethod
        def log(d):
            logged.append(d)

    monkeypatch.setattr(D, "_wandb", FakeWandb)
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256)
    fd = make_method(meta)
    st, te, am = _data(3, torch.float32, torch.float32, seed=50, D=256)
    fd.past_model = lambda **kw: Out(tuple(te))

    @torch.compile(fullgraph=True)
    def step(students, batch):
        return fd.distill(Out(tuple(students)), batch)

    fd.distill(Out(tuple(s.detach().requires_grad_(True) for s in st)), {"attention_mask": am})   # plan
    fd.flush_logs(wait=True)
    logged.clear()
    values = []
    for i in range(3):
        leaves = [(s * (1 + i)).detach().requires_grad_(True) for s in st]
        step(leaves, {"attention_mask": am}).backward()
        values.append(fd.last_layer_losses[:3].tolist())
        assert not logged or len(logged) % 3 == 0
        fd.record_step()
    fd.flush_logs(wait=True)
    keys = [f"task_0/distill_loss_{l}" for l in (0, 1, 2)]
    assert [list(d) for d in logged] == [[k] for k in keys] * 3
    got = [[d[k] for d, k in zip(logged[3 * i:3 * i + 3], keys)] for i in range(3)]
    assert got == values


# ---------------------------------------------------------------- 2 GPUs, peer communicator
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_compiled_sharded_step_equals_eager_sharded_step():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29531", os.path.join(ROOT, "tools", "compiled_multirank_check.py")]
    env = dict(os.environ, MAFED_B200_DIST="peer")
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
