"""``replay()`` and the reference's own caller against outputs of the UNMODIFIED reference
(tests/golden/replay_cases.npz, made by tests/golden/make_golden_replay.py on the CPU):

* the mirror's ``replay(model)`` on the GPU -- loss, ``n_ex``, every parameter gradient, what it leaves in the batch,
  what it sends to W&B -- for five configurations (SURVEY 8a row a3);
* the unmodified ``VLPythiaVQACLearner.training_step`` (oracle/_ref, Lightning stubbed) with the registry entry
  ``CLMethod["featdistill"]`` swapped to the mirror, over two tasks x four batches (row a12).
"""
import copy
import json
import os
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 2e-4          # fp32 model on CPU (golden) vs fp32 model on the GPU (cuBLAS / different reduction orders)


def _golden():
    z = np.load(os.path.join(HERE, "golden", "replay_cases.npz"))
    return z, json.loads(str(z["meta"]))


def _generator():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_replay", os.path.join(HERE, "golden", "make_golden_replay.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    return gen


def _models(z, device):
    """The two models the goldens were made with, regenerated from their seeds and checked against the stored digests."""
    gen = _generator()
    student, teacher = gen.models()
    assert gen.weights_digest(student) == str(z["student_sha256"]), "regenerated student weights differ from the goldens'"
    assert gen.weights_digest(teacher) == str(z["teacher_sha256"]), "regenerated teacher weights differ from the goldens'"
    return student.to(device), teacher.to(device).eval()


def _batch(z, prefix, device):
    return {k[len(prefix) + 1:]: torch.from_numpy(z[k]).to(device) for k in z.files if k.startswith(prefix + "/")}


def _sample_positions(numel, k=64):
    rng = np.random.default_rng(11)
    return np.sort(rng.choice(numel, size=min(k, numel), replace=False)).astype(np.int64)


def _check_grads(model, z, prefix, names):
    have = [n for n, p in model.named_parameters() if p.grad is not None]
    assert have == names, (have, names)
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.detach().double().cpu()
        want_norm = float(z[f"{prefix}/gnorm/{name}"])
        if want_norm == 0.0:
            assert float(g.norm()) == 0.0
            continue
        assert float(g.norm()) == pytest.approx(want_norm, rel=TOL), name
        want = torch.from_numpy(z[f"{prefix}/gsamp/{name}"])
        got = g.reshape(-1)[_sample_positions(g.numel())]
        assert float((got - want).norm()) <= TOL * max(float(want.norm()), 1e-3 * want_norm), name


class _Opts:
    tasks = ["a", "b", "c"]
    batch_size = 4
    seed = 42
    pin_mem = False
    accumulate_grad_batches = 1


def _mirror(case, registry=None):
    from mafed_b200.methods import CLMethod
    registry = registry or CLMethod
    opts = _Opts()
    opts.accumulate_grad_batches = case["accumulate"]
    fd = registry["featdistill"](memory_size=8, opts=opts, model_type="vlpythia",
                                 distillation_modality_weighing_strategy=case["modality"],
                                 distillation_layer_weighing_strategy=case["layer_strategy"],
                                 distillation_coeff=case["coeff"], distillation_layer=case["layer"],
                                 distillation_loss=case["loss"], gamma=0.5, num_hidden_layers=3,
                                 replay_coeff=case["replay_coeff"])
    fd.num_vision_tokens = 8
    fd.task_id = case["task_id"]
    return fd


@pytest.mark.gpu
@pytest.mark.parametrize("selective", [False, True], ids=["full-tuple", "selective-capture"])
@pytest.mark.parametrize("name", ["discounted", "single2", "equal_cosine", "no_distill", "first_task"])
def test_replay_matches_the_reference(name, selective, monkeypatch):
    import types as _types

    from mafed_b200.methods import distillation as D
    z, meta = _golden()
    case = [c for c in meta["replay"] if c["name"] == name][0]
    logged = []
    monkeypatch.setattr(D, "_wandb", _types.SimpleNamespace(run=object(), log=lambda d, *a, **k: logged.append(dict(d))))
    student, teacher = _models(z, "cuda")
    fd = _mirror(case)
    fd.selective_capture = selective
    fd.past_model = teacher
    batch = _batch(z, "batch", "cuda")
    fd.mem_dataloader = [batch]
    loss, n_ex = fd.replay(student)
    assert n_ex == case["n_ex"] and fd.step == case["step"]
    assert (loss is None) == case["loss_is_none"]
    assert sorted(batch.keys()) == case["batch_keys"]          # `labels` popped, the two masks added (or neither)
    if "lang_sum" in case:
        assert list(batch["lang_masks"].shape) == case["mask_shape"] == list(batch["image_masks"].shape)
        assert int(batch["lang_masks"].sum()) == case["lang_sum"] and int(batch["image_masks"].sum()) == case["image_sum"]
    (loss / case["accumulate"]).backward()                      # Lightning: loss / accumulate_grad_batches
    torch.cuda.synchronize()
    assert float(loss) == pytest.approx(float(z[f"replay/{name}/loss"]), rel=TOL)
    _check_grads(student, z, f"replay/{name}", case["grad_names"])
    assert not any(p.grad is not None for p in teacher.parameters())
    fd.flush_logs()
    got = {}
    for d in logged:
        got.update(d)
    assert got.keys() == case["logged"].keys()
    for k, v in case["logged"].items():
        assert got[k] == pytest.approx(v, rel=TOL)
    if case["coeff"] != 0:
        assert len(logged) == len(case["logged"])               # one wandb.log per layer, like distillation.py:165


@pytest.mark.gpu
def test_unmodified_training_step_drives_the_mirror():
    """mafed/model/vqa_cont_learner.py:213-236 as shipped (oracle/_ref), its `cl_method` built from the registry
    with "featdistill" swapped to the B200 strategy (INTEGRATION.md's one-line swap)."""
    from oracle import ref_harness as R
    if not R.available():
        pytest.skip("oracle/_ref is absent: run `python oracle/make_ref.py` in the build container")
    import mafed_b200.methods as mirror
    methods = R.load()
    Learner = R.learner_class()
    z, meta = _golden()
    ts = meta["training_step"]
    original = methods.CLMethod["featdistill"]
    methods.CLMethod["featdistill"] = mirror.FeatureDistillation      # the swap
    try:
        fd = _mirror(ts["case"], registry=methods.CLMethod)
        assert type(fd) is mirror.FeatureDistillation
        student, teacher = _models(z, "cuda")
        fd.past_model = teacher
        mem, task_batch = _batch(z, "ts_mem", "cuda"), _batch(z, "ts_task", "cuda")

        class FreshBatches:
            def __iter__(self):
                yield {k: v.clone() for k, v in mem.items()}

        fd.mem_dataloader = FreshBatches()
        learner = Learner.__new__(Learner)
        learner.model, learner.cl_method = student, fd
        learner.config = types.SimpleNamespace(replay_interval=2)
        for step in ts["steps"]:
            learner.task_id = fd.task_id = step["task_id"]
            learner.logged = []
            student.zero_grad(set_to_none=True)
            loss = learner.training_step({k: v.clone() for k, v in task_batch.items()}, step["batch_idx"])
            (loss / ts["case"]["accumulate"]).backward()
            torch.cuda.synchronize()
            tag = f"ts/{step['task_id']}_{step['batch_idx']}"
            assert float(loss) == pytest.approx(float(z[f"{tag}/loss"]), rel=TOL), tag
            assert len(learner.logged) == 1 and learner.logged[0][0] == step["log_name"] and learner.logged[0][1] is loss
            assert {k: v for k, v in learner.logged[0][2].items()} == step["log_kwargs"]
            assert fd.step == step["fd_step"]
            _check_grads(student, z, tag, step["grad_names"])
    finally:
        methods.CLMethod["featdistill"] = original


def test_replay_goldens_are_what_the_reference_produces_here():
    """Re-run the unmodified reference on the CPU (oracle/_ref or /root/reference) and compare with the committed
    file: the goldens are reproducible, not hand-made."""
    from oracle import ref_harness as R
    if not R.available():
        pytest.skip("the reference is not available on this machine")
    gen = _generator()
    z, meta = _golden()
    student, teacher = gen.models()
    assert gen.weights_digest(student) == str(z["student_sha256"])
    batch = gen.make_batch(seed=0)
    for case in gen.REPLAY_CASES[:3]:
        fd = gen.make_method(case)
        model = copy.deepcopy(student)
        fd.past_model = copy.deepcopy(teacher).eval()
        fd.mem_dataloader = [{k: v.clone() for k, v in batch.items()}]
        loss, n_ex = fd.replay(model)
        assert float(loss) == pytest.approx(float(z[f"replay/{case['name']}/loss"]), rel=1e-6)
        (loss / case["accumulate"]).backward()
        for name, p in model.named_parameters():
            if p.grad is not None:
                assert float(p.grad.double().norm()) == pytest.approx(float(z[f"replay/{case['name']}/gnorm/{name}"]), rel=1e-6)


def test_oracle_ref_is_byte_identical_to_the_reference():
    """oracle/_ref holds unmodified copies: every file matches its recorded sha256, and -- where the reference's
    tree is present -- the tree itself."""
    import hashlib

    from oracle import make_ref
    if not os.path.exists(os.path.join(make_ref.OUT, "MANIFEST.json")):
        pytest.skip("oracle/_ref has not been made on this machine")
    assert make_ref.verify()
    with open(os.path.join(make_ref.OUT, "MANIFEST.json")) as f:
        manifest = json.load(f)
    assert sorted(manifest["files"]) == sorted(make_ref.FILES)
    if os.path.isdir(os.path.join(make_ref.REFERENCE, "mafed")):
        for rel, digest in manifest["files"].items():
            with open(os.path.join(make_ref.REFERENCE, rel), "rb") as f:
                assert hashlib.sha256(f.read()).hexdigest() == digest, rel
