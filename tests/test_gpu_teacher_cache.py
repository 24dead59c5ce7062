"""``FeatureDistillation(teacher_cache=True)`` on the GPU: the gather kernel against the torch reference gather, a cached
replay step against the same step fed the reference gather of the same cache (bit-identical), and against the uncached
teacher forward where the cache computes the same thing (every sample at the same text length)."""
import copy
import types

import pytest
import torch
from torch.nn.attention import SDPBackend, sdpa_kernel

from gpu_util import rel_err, tolerances
from mafed_b200 import teacher_cache as TC

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------- the kernel
def _cache(L, M, T_c, D, dtype, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn((M, T_c, D), generator=g, device="cuda").to(dtype) for _ in range(L)]


def _bitwise(a, b):
    bits = {4: torch.int32, 2: torch.int16}[a.element_size()]
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(bits), b.view(bits))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("L,M,T_c,D", [(1, 9, 21, 64), (3, 9, 21, 37), (70, 5, 14, 24), (2, 7, 300, 2048)])
@pytest.mark.parametrize("short", [0, 5])
def test_gather_matches_reference(dtype, L, M, T_c, D, short):
    n_vis = 8
    cache = _cache(L, M, T_c, D, dtype)
    idx = [3, 0, M - 1, 3, 1, 2 % M]
    T = T_c - short
    got = TC.gather(cache, idx, T, n_vis)
    want = TC.reference_gather(cache, idx, T, n_vis)
    torch.cuda.synchronize()
    assert len(got) == L
    for g, w in zip(got, want):
        assert _bitwise(g, w)


def test_gather_unaligned_views_many_samples_and_no_visual_prefix():
    base = _cache(2, 2200, 10, 9, torch.bfloat16, seed=1)
    cache = [c.view(-1)[1:].view(-1)[: 2199 * 10 * 9].view(2199, 10, 9) for c in base]   # 2-byte aligned pointers
    idx = [(7 * b) % 2199 for b in range(2100)]                                              # two sample chunks
    for n_vis, T in ((0, 6), (4, 10), (4, 4)):
        got, want = TC.gather(cache, idx, T, n_vis), TC.reference_gather(cache, idx, T, n_vis)
        for g, w in zip(got, want):
            assert _bitwise(g, w)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_out_of_range_index_writes_nan_rows(dtype):
    M, T_c, D, T, n_vis = 6, 20, 64, 16, 8
    cache = _cache(3, M, T_c, D, dtype)
    idx = [2, M, 5, -4]
    out = [torch.zeros((4, T, D), dtype=dtype, device="cuda") for _ in cache]
    TC.gather_raw([o.data_ptr() for o in out], [c.data_ptr() for c in cache], idx, 4, M, T, T_c, n_vis, D,
                  TC._DTYPES[dtype], torch.cuda.current_stream().cuda_stream)
    want = TC.reference_gather(cache, idx, T, n_vis)
    torch.cuda.synchronize()
    for o, w in zip(out, want):
        assert o[[1, 3]].isnan().all()
        assert _bitwise(o[[0, 2]], w[[0, 2]])


# ---------------------------------------------------------------- the replay step
class Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 2


def _to_cuda(loader):
    class Prefetch:                     # PrefetchLoader's contract: tensors to the device, other values as they are
        dataset = loader.dataset

        def __iter__(self):
            for b in loader:
                yield {k: v.cuda() if torch.is_tensor(v) else v for k, v in b.items()}
    return Prefetch()


CASES = {
    "mse-discounted": dict(modality="balanced", strategy="discounted"),
    "mse-single-equal": dict(modality="equal", strategy="single", layer=1),
    "cosine-discounted": dict(modality="balanced", strategy="discounted", loss="cosine"),
    "with-entry-L": dict(modality="balanced", strategy="discounted", num_hidden_layers=4),
    "early-exit": dict(modality="balanced", strategy="discounted", early_exit=True),
    "bf16-teacher": dict(modality="balanced", strategy="discounted", teacher_dtype=torch.bfloat16, num_hidden_layers=4),
    "fp16-teacher-early-exit": dict(modality="balanced", strategy="discounted", teacher_dtype=torch.float16,
                                    early_exit=True),
    "selective-capture": dict(modality="balanced", strategy="discounted", selective_capture=True),
    "no-replay-loss": dict(modality="balanced", strategy="discounted", replay_coeff=0.0, early_exit=True),
}


def _strategy(cache, modality, strategy, layer=None, loss="mse", num_hidden_layers=3, replay_coeff=1.0, **kw):
    from mafed_b200.methods import CLMethod
    from vl_memory import collate
    fd = CLMethod["featdistill"](memory_size=16, opts=Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy=modality,
                                 distillation_layer_weighing_strategy=strategy, distillation_layer=layer,
                                 distillation_loss=loss, gamma=0.5, num_hidden_layers=num_hidden_layers,
                                 replay_coeff=replay_coeff, distillation_coeff=2.0, teacher_cache=cache, **kw)
    fd.num_vision_tokens = 8
    fd.num_workers = 0
    fd.data_hooks = (collate, _to_cuda)
    return fd


def _models(fp32_island=False):
    from tiny_vl import TinyVL
    torch.manual_seed(0)
    teacher = TinyVL(fp32_island=fp32_island).cuda()
    student = copy.deepcopy(teacher)
    with torch.no_grad():
        for p in student.parameters():
            p.add_(0.02 * torch.randn_like(p))
    return student, teacher


def _step(fd, student, batch, logged):
    model = copy.deepcopy(student)
    fd.mem_dataloader = [batch]
    logged.clear()
    calls = []
    handle = fd.past_model.register_forward_hook(lambda *a: calls.append(1)) if fd.past_model is not None else None
    with sdpa_kernel([SDPBackend.MATH]):
        loss, n_ex = fd.replay(model)
        (loss / Opts.accumulate_grad_batches).backward()
    fd.flush_logs()
    torch.cuda.synchronize()
    if handle is not None:
        handle.remove()
    grads = {n: None if p.grad is None else p.grad.clone() for n, p in model.named_parameters()}
    return dict(loss=loss.detach().clone(), n_ex=n_ex, grads=grads, batch=batch, logged=list(logged),
                teacher_calls=len(calls))


def _wandb(monkeypatch):
    from mafed_b200.methods import distillation as D
    logged = []
    monkeypatch.setattr(D, "_wandb", types.SimpleNamespace(run=object(), log=lambda d, *a, **k: logged.append(dict(d))))
    return logged


@pytest.mark.parametrize("name", list(CASES))
def test_cached_replay_is_bit_identical_to_the_reference_gather(name, monkeypatch):
    from vl_memory import VLSamples
    cfg = CASES[name]
    logged = _wandb(monkeypatch)
    student, teacher = _models()
    fd = _strategy(True, **cfg)
    fd.update(dataset=VLSamples(40, seed=1, max_txt=9), model=teacher, dataloader=None)
    cache = fd._teacher_cache
    assert cache is not None and cache.T_c == 8 + max(len(fd.mem_dataloader.dataset[i][1]["input_ids"])
                                                      for i in range(len(fd.mem_dataloader.dataset)))
    if cfg.get("teacher_dtype") is not None:
        assert all(s.dtype == cfg["teacher_dtype"] for s in cache.states)
    ref = _strategy(False, **cfg)
    ref.task_id, ref.past_model = fd.task_id, fd.past_model
    ref.loss_weights = fd.loss_weights

    def gathered(batch, layers):
        batch.pop("labels", None)
        return TC.reference_gather(cache.states, idx, batch["attention_mask"].shape[1] + 8, 8)

    ref._past_states = gathered
    steps = 0
    for drawn in fd.mem_dataloader:                                   # every batch of an epoch: ragged text lengths
        idx = drawn["memory_index"]
        plain = {k: v for k, v in drawn.items() if k != "memory_index"}
        a = _step(fd, student, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in drawn.items()}, logged)
        b = _step(ref, student, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in plain.items()}, logged)
        assert a["teacher_calls"] == 0
        assert torch.equal(a["loss"], b["loss"]) and a["n_ex"] == b["n_ex"] == len(idx)
        checked = 0
        for n, g in b["grads"].items():
            e = a["grads"][n]
            assert (e is None) == (g is None), n
            if g is not None:
                assert torch.equal(e, g), n
                checked += 1
        assert checked > 5
        assert sorted(a["batch"]) == sorted(b["batch"]) and "labels" not in a["batch"]
        assert "memory_index" not in a["batch"]
        for k in ("lang_masks", "image_masks"):
            assert torch.equal(a["batch"][k], b["batch"][k]), k
        assert a["logged"] == b["logged"] and len(a["logged"]) == len(fd.loss_weights.get_distillation_layers())
        steps += 1
    assert steps == 2                                                # 8 memory samples, batches of 4


@pytest.mark.parametrize("fp32", [True, False])
def test_cached_replay_matches_the_teacher_forward_at_one_text_length(fp32, monkeypatch):
    """Every memory sample has the same text length, so T == T_c and the cache computes what the teacher forward of
    the step computes, up to GEMM-shape rounding (fp32 under the fp32 island, bf16 under replay's autocast)."""
    from vl_memory import VLSamples
    logged = _wandb(monkeypatch)
    student, teacher = _models(fp32_island=fp32)
    cfg = dict(modality="balanced", strategy="discounted", num_hidden_layers=4)
    fd = _strategy(True, **cfg)
    fd.update(dataset=VLSamples(40, seed=2, min_txt=7, max_txt=7), model=teacher, dataloader=None)
    assert fd._teacher_cache.T_c == 15
    plain = _strategy(False, **cfg)
    plain.task_id, plain.past_model, plain.loss_weights = fd.task_id, fd.past_model, fd.loss_weights
    tol = tolerances(torch.float32 if fp32 else torch.bfloat16)[0]
    for drawn in fd.mem_dataloader:
        a = _step(fd, student, dict(drawn), logged)
        b = _step(plain, student, {k: v for k, v in drawn.items() if k != "memory_index"}, logged)
        assert a["teacher_calls"] == 0 and b["teacher_calls"] == 1
        assert rel_err(a["loss"], b["loss"]) < tol
        for n, g in b["grads"].items():
            if g is not None and g.norm() > 0:
                assert rel_err(a["grads"][n], g) < (tol if fp32 else 2e-2), n


def test_missing_memory_index_raises():
    from mafed_b200.cabi import MafedDistillError
    from vl_memory import VLSamples
    student, teacher = _models()
    fd = _strategy(True, modality="balanced", strategy="discounted")
    fd.update(dataset=VLSamples(40, seed=1), model=teacher, dataloader=None)
    drawn = next(iter(fd.mem_dataloader))
    drawn.pop("memory_index")
    fd.mem_dataloader = [drawn]
    with pytest.raises(MafedDistillError, match="memory_index"):
        fd.replay(copy.deepcopy(student))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_cached_replay_equals_one_gpu():
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.join(root, "tools", "multirank_check.py"),
           "--teacher-cache"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
