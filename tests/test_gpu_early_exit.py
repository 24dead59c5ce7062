"""``FeatureDistillation(early_exit=True)`` on the GPU: replay() stops the teacher forward after the last distilled
hidden state (and the student's when no replay loss is taken) and gives bit-identical results to the full forwards --
loss, n_ex, every parameter gradient, the masks left in the batch, the `labels` pop and the W&B calls.  Under
torch.compile the option does not apply and fd.distill keeps its one graph."""
import copy
import types

import pytest
import torch
from torch.nn.attention import SDPBackend, sdpa_kernel

from gpu_util import Out

pytestmark = pytest.mark.gpu


class Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 2


# TinyVL has L = 3 decoder layers; num_hidden_layers=4 distils entry L (the final layer norm's output) as well
CASES = {
    "equal-single": dict(modality="equal", strategy="single", layer=1),
    "equal-discounted": dict(modality="equal", strategy="discounted"),
    "balanced-single": dict(modality="balanced", strategy="single", layer=2),
    "balanced-discounted": dict(modality="balanced", strategy="discounted"),
    "balanced-discounted-with-entry-L": dict(modality="balanced", strategy="discounted", num_hidden_layers=4),
    "cosine-discounted": dict(modality="balanced", strategy="discounted", loss="cosine"),
    "cosine-single": dict(modality="equal", strategy="single", layer=0, loss="cosine"),
    "cls": dict(modality="equal", strategy="discounted", loss="cosine", cls=True),
    "bf16-teacher": dict(modality="balanced", strategy="discounted", teacher_dtype=torch.bfloat16),
    "bf16-teacher-with-entry-L": dict(modality="balanced", strategy="discounted", num_hidden_layers=4,
                                      teacher_dtype=torch.bfloat16),
    "no-replay-loss-discounted": dict(modality="balanced", strategy="discounted", replay_coeff=0.0),
    "no-replay-loss-single": dict(modality="equal", strategy="single", layer=1, replay_coeff=0.0),
    "no-replay-loss-with-entry-L": dict(modality="balanced", strategy="discounted", num_hidden_layers=4,
                                        replay_coeff=0.0),
    "no-replay-loss-cls": dict(modality="equal", strategy="single", layer=1, loss="cosine", cls=True,
                               replay_coeff=0.0),
}


def _make(teacher, batch, early_exit, modality, strategy, layer=None, loss="mse", cls=False, num_hidden_layers=3,
          replay_coeff=1.0, teacher_dtype=None):
    from mafed_b200.methods import CLMethod
    fd = CLMethod["featdistill"](memory_size=8, opts=Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy=modality,
                                 distillation_layer_weighing_strategy=strategy, distillation_layer=layer,
                                 distillation_loss=loss, cls_distillation=cls, gamma=0.5,
                                 num_hidden_layers=num_hidden_layers, replay_coeff=replay_coeff, distillation_coeff=2.0,
                                 teacher_dtype=teacher_dtype, early_exit=early_exit)
    fd.num_vision_tokens = 8
    fd.task_id = 1
    fd._update_model(teacher)
    fd.mem_dataloader = [{k: v.clone() for k, v in batch.items()}]
    return fd


def _heads_run(*models):
    """Counts the completed forwards of each model's LM head."""
    counts = [0] * len(models)
    handles = []
    for i, m in enumerate(models):
        def hook(mod, args, out, i=i):
            counts[i] += 1
        handles.append(m.embed_out.register_forward_hook(hook))
    return counts, handles


def _replay(student, teacher, batch, early_exit, cfg, logged):
    model = copy.deepcopy(student)
    fd = _make(teacher, batch, early_exit, **cfg)
    mem = fd.mem_dataloader[0]
    logged.clear()
    heads, handles = _heads_run(model, fd.past_model)
    # the math attention backend: the memory-efficient one's backward accumulates with atomics, so two runs of the
    # same graph could differ in the last bits
    with sdpa_kernel([SDPBackend.MATH]):
        loss, n_ex = fd.replay(model)
        (loss / Opts.accumulate_grad_batches).backward()
    fd.flush_logs()
    torch.cuda.synchronize()
    for h in handles:
        h.remove()
    grads = {n: None if p.grad is None else p.grad.clone() for n, p in model.named_parameters()}
    assert not any(p.grad is not None for p in fd.past_model.parameters())
    return dict(loss=loss.detach().clone(), n_ex=n_ex, grads=grads, batch=mem, logged=list(logged), heads=heads,
                step=fd.step, layers=fd.loss_weights.get_distillation_layers())


@pytest.mark.parametrize("name", list(CASES))
def test_early_exit_replay_is_bit_identical(name, monkeypatch):
    from mafed_b200.methods import distillation as D
    from tiny_vl import TinyVL, make_batch
    cfg = CASES[name]
    logged = []
    monkeypatch.setattr(D, "_wandb", types.SimpleNamespace(run=object(), log=lambda d, *a, **k: logged.append(dict(d))))
    torch.manual_seed(0)
    student = TinyVL().cuda()
    teacher = copy.deepcopy(student)
    with torch.no_grad():
        for p in student.parameters():
            p.add_(0.02 * torch.randn_like(p))                       # the student has moved away from the teacher
    batch = make_batch(device="cuda")

    full = _replay(student, teacher, batch, False, cfg, logged)
    early = _replay(student, teacher, batch, True, cfg, logged)

    replay_loss = cfg.get("replay_coeff", 1.0) > 0
    assert full["heads"] == [1, 1]                                   # student, teacher: both forwards ran to the end
    assert early["heads"] == [1 if replay_loss else 0, 0]            # the teacher's never reached its LM head
    assert torch.equal(early["loss"], full["loss"]) and early["n_ex"] == full["n_ex"] == 4
    assert early["step"] == full["step"] == 1
    assert early["grads"].keys() == full["grads"].keys()
    checked = 0
    for n, g in full["grads"].items():
        e = early["grads"][n]
        assert (e is None) == (g is None), n
        if g is not None:
            assert torch.equal(e, g), n
            checked += 1
    assert checked > 5
    assert sorted(early["batch"]) == sorted(full["batch"])          # `labels` popped (and the masks added) alike
    assert "labels" not in early["batch"]
    for k in ("lang_masks", "image_masks"):
        if k in full["batch"]:
            assert torch.equal(early["batch"][k], full["batch"][k]), k
    assert early["logged"] == full["logged"] and len(full["logged"]) == len(full["layers"])   # one call per layer


def test_stopped_student_output_has_no_logits_or_loss():
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    student = TinyVL().cuda()
    fd = _make(student, make_batch(device="cuda"), True, "balanced", "single", layer=1, replay_coeff=0.0)
    seen = {}
    distill = fd.distill

    def spy(output, batch):
        seen["output"] = output
        return distill(output, batch)

    fd.distill = spy
    loss, n_ex = fd.replay(student)
    out = seen["output"]
    assert len(out.hidden_states) == 4 and out.hidden_states[1].requires_grad
    for attr in ("logits", "loss"):
        with pytest.raises(AttributeError):
            getattr(out, attr)
    assert loss.requires_grad and n_ex == 4


@pytest.fixture
def _fresh_dynamo():
    from mafed_b200 import node
    node.load()
    torch._dynamo.reset()
    yield
    torch._dynamo.reset()


def test_compiled_distill_with_early_exit_keeps_one_graph(_fresh_dynamo):
    """Under torch.compile the teacher forward runs in full inside fd.distill: with ``fullgraph=True`` any graph break
    would raise, and over more steps than the recompile limit Dynamo builds one graph."""
    from torch._dynamo.utils import counters
    from gpu_util import make_method
    from tiny_vl import TinyVL, make_batch
    torch.manual_seed(0)
    model = TinyVL(n_vis=256, dim=256, layers=3).cuda()
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=3,
                layer=None, n_vis=256)
    fd, ref = make_method(meta, early_exit=True), make_method(meta, early_exit=True)
    fd.adapt_assumed_grad_out = ref.adapt_assumed_grad_out = False
    batch = make_batch(bsz=4, txt=6, n_vis=256, device="cuda")
    batch.pop("labels")
    # the student has run eagerly with output_hidden_states=True before it becomes the teacher, as in training: HF
    # installs its hidden-state hooks on that first call, under a lock Dynamo cannot trace, and the snapshot
    # (`_update_model`, a deep copy) inherits them
    with torch.no_grad():
        states = [h.detach() for h in model(**batch, output_hidden_states=True).hidden_states]
    fd._update_model(model)
    with torch.no_grad():
        for p in fd.past_model.parameters():
            p.add_(0.01 * torch.randn_like(p))
    ref.past_model = fd.past_model
    head_runs, handles = _heads_run(fd.past_model)
    fd.distill(Out(tuple(s.clone().requires_grad_(True) for s in states)), dict(batch))   # eager: plan tables
    for h in handles:
        h.remove()
    assert head_runs == [0]                                          # the eager step stopped the teacher

    def step(students, b):
        return fd.distill(Out(tuple(students)), b)

    compiled = torch.compile(step, fullgraph=True)
    counters.clear()
    steps = torch._dynamo.config.recompile_limit + 2
    for i in range(steps):
        s_i = [(s * (1 + 0.01 * i)).requires_grad_(True) for s in states]
        loss = compiled(s_i, dict(batch))
        loss.backward()
        fd.record_step()
    e_i = [(s * (1 + 0.01 * (steps - 1))).requires_grad_(True) for s in states]
    e_loss = ref.distill(Out(tuple(e_i)), dict(batch))
    e_loss.backward()
    torch.cuda.synchronize()
    assert counters["stats"]["unique_graphs"] == 1, dict(counters["stats"])
    # the teacher forward inside the graph is Inductor's, the eager one stops early: same states up to kernel rounding
    assert float(loss) == pytest.approx(float(e_loss), rel=1e-4)
    for s, e in zip(s_i, e_i):
        assert (s.grad is None) == (e.grad is None)
        assert s.grad is None or float((s.grad - e.grad).norm() / e.grad.norm()) < 1e-3
