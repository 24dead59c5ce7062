"""Host side of ``FeatureDistillation(teacher_cache=True)`` (no GPU): the memory loader's sample indices, the cache's
length and left re-padding, when it is (re)built, the gather's row mapping (torch reference) and the argument checks of
``mafed_teacher_gather``."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from torch.utils.data import ConcatDataset, RandomSampler

from mafed_b200 import teacher_cache as TC
from mafed_b200.cabi import MafedDistillError
from mafed_b200.methods import FeatureDistillation
from vl_memory import PAD_ID, VLSamples, collate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 42; pin_mem = False; accumulate_grad_batches = 1


def _make(teacher_cache, memory_size=12, **kw):
    fd = FeatureDistillation(memory_size, Opts(), "vlpythia", distillation_modality_weighing_strategy="balanced",
                             distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                             num_hidden_layers=3, teacher_cache=teacher_cache, **kw)
    fd.num_workers = 0
    fd.num_vision_tokens = 8
    fd.data_hooks = (collate, lambda loader: loader)
    return fd


def _check_indices(fd, batches):
    memory = ConcatDataset(fd.datasets)
    seen = []
    for batch in batches:
        idx = batch["memory_index"]
        assert isinstance(idx, list) and all(type(i) is int for i in idx)
        assert [memory[i]["id"] for i in idx] == batch["ids"]
        seen += idx
    return seen


def test_loader_yields_memory_indices():
    fd = _make(True)
    fd._update_memory(VLSamples(40, seed=1))
    fd._update_memory(VLSamples(30, seed=2))
    assert isinstance(fd.mem_sampler, RandomSampler) and fd.mem_sampler.data_source is fd.mem_dataloader.dataset.dataset
    seen = _check_indices(fd, fd.mem_dataloader)
    assert sorted(seen) == list(range(12))                 # one epoch: every memory sample once
    fd.persistent_memory_iterator = True
    for _ in range(4):
        _check_indices(fd, [fd._next_memory_batch()])


def test_option_off_leaves_the_loader_as_it_was(monkeypatch):
    monkeypatch.setattr(TC, "build", lambda strategy: pytest.fail("no cache without the option"))
    fd = _make(False)
    fd.loss_weights.update_weights = lambda *a, **k: None
    fd.update(dataset=VLSamples(40, seed=1), model=torch.nn.Linear(2, 2), dataloader=None)
    loader = fd.mem_dataloader
    assert type(loader.dataset) is ConcatDataset and loader.collate_fn is collate
    assert fd._teacher_cache is None and fd._memory_index is None
    batch = fd._next_memory_batch()
    assert sorted(batch) == ["attention_mask", "ids", "input_ids", "labels", "pixel_values"]


def test_past_states_without_the_option_runs_the_teacher(monkeypatch):
    monkeypatch.setattr(TC, "gather", lambda *a, **k: pytest.fail("no gather without the option"))
    fd = _make(False)
    calls = []

    class Teacher:
        def __call__(self, **kw):
            calls.append(sorted(kw))
            return type("O", (), {"hidden_states": [torch.zeros(1)] * 4})()

    fd.past_model = Teacher()
    batch = {"attention_mask": torch.ones(2, 3, dtype=torch.int64), "labels": torch.zeros(2, 3)}
    fd._past_states(batch, [0, 1, 2])
    assert calls == [["attention_mask", "output_hidden_states", "return_dict"]] and "labels" not in batch


def test_repad_left_pads_like_the_collate():
    batch = collate([VLSamples(6, seed=3)[i] for i in range(3)])
    txt = batch["input_ids"].shape[1]
    out = TC.repad_left(batch, txt + 4)
    assert out["input_ids"].shape == (3, txt + 4) and out["attention_mask"].shape == (3, txt + 4)
    assert torch.equal(out["input_ids"][:, 4:], batch["input_ids"]) and (out["input_ids"][:, :4] == PAD_ID).all()
    assert torch.equal(out["attention_mask"][:, 4:], batch["attention_mask"]) and (out["attention_mask"][:, :4] == 0).all()
    assert out["pixel_values"] is batch["pixel_values"]
    assert TC.repad_left(batch, txt) is batch
    with pytest.raises(ValueError):
        TC.repad_left(batch, txt - 1)
    full = {"input_ids": torch.full((2, 3), 7), "attention_mask": torch.ones(2, 3, dtype=torch.int64)}
    assert (TC.repad_left(full, 5)["input_ids"][:, :2] == 0).all()    # no pad to copy: id 0 under mask 0


def test_cache_build_on_cpu_matches_each_sample_at_T_c():
    """T_c = n_vis + the longest text; each cached sample equals the teacher run on it alone, left-padded to T_c (on
    every row the step weighs: the pad rows' own states depend on the pad id, which a batch without padding lacks)."""
    from tiny_vl import TinyVL
    torch.manual_seed(0)
    fd = _make(True, selective_capture=True)
    data = VLSamples(40, seed=1, min_txt=2, max_txt=9)
    fd._update_memory(data)
    fd.past_model = TinyVL(fp32_island=True).eval()
    cache = TC.build(fd)
    memory = ConcatDataset(fd.datasets)
    longest = max(len(memory[i]["input_ids"]) for i in range(len(memory)))
    assert cache.T_c == 8 + longest and cache.layers == [0, 1, 2]
    M = len(memory)
    assert [tuple(s.shape) for s in cache.states] == [(M, cache.T_c, 64)] * 3
    assert cache.nbytes == 3 * M * cache.T_c * 64 * 4
    for j in range(len(memory)):
        one = TC.repad_left(collate([memory[j]]), longest)
        one.pop("labels")
        with torch.no_grad():
            hs = fd.past_model(**one, output_hidden_states=True).hidden_states
        live = torch.cat([torch.ones(8, dtype=torch.bool), one["attention_mask"][0].bool()])
        assert int(live.sum()) == 8 + len(memory[j]["input_ids"])
        for s, l in zip(cache.states, cache.layers):
            torch.testing.assert_close(s[j][live], hs[l][0][live], rtol=1e-5, atol=1e-5)


def test_cache_is_rebuilt_on_update_and_lazily_after_load(monkeypatch):
    built = []

    class Fake:
        def __init__(self, strategy):
            self.task = strategy.task_id

        def gather(self, idx, T, layers):
            return ("gathered", list(idx), T, list(layers))

    monkeypatch.setattr(TC, "build", lambda strategy: built.append(Fake(strategy)) or built[-1])
    fd = _make(True)
    fd.loss_weights.update_weights = lambda *a, **k: None
    model = torch.nn.Linear(2, 2)
    fd.update(dataset=VLSamples(40, seed=1), model=model, dataloader=None)
    assert len(built) == 1 and fd._teacher_cache is built[0]
    fd.update(dataset=VLSamples(30, seed=2), model=model, dataloader=None)
    assert len(built) == 2 and fd._teacher_cache is built[1]
    state = fd.state_dict()
    assert not any("cache" in k for k in state)
    other = _make(True)
    other.load_state_dict(state, datasets=[VLSamples(40, seed=1), VLSamples(30, seed=2)])
    assert other._teacher_cache is None and len(built) == 2
    batch = {"attention_mask": torch.ones(2, 5, dtype=torch.int64), "labels": torch.zeros(2, 5)}
    other._memory_index = [3, 1]
    with pytest.raises(MafedDistillError, match="no teacher"):
        other._past_states(dict(batch), [0, 1, 2])
    other._update_model(model)
    other._memory_index = [3, 1]
    assert other._past_states(batch, [0, 1, 2]) == ("gathered", [3, 1], 13, [0, 1, 2])
    assert len(built) == 3 and "labels" not in batch and other._memory_index is None
    with pytest.raises(MafedDistillError, match="no memory_index"):
        other._past_states(batch, [0, 1, 2])          # the index of a batch is used once
    assert len(built) == 3


def test_reference_gather_row_mapping():
    M, T_c, D, n_vis = 5, 11, 3, 4
    code = torch.arange(M * T_c, dtype=torch.float32).view(M, T_c, 1).expand(M, T_c, D).contiguous()
    idx = [4, 0, 2, 2]
    for T in (T_c, 7, n_vis):
        out = TC.reference_gather([code], idx, T, n_vis)[0]
        assert out.shape == (4, T, D)
        for b, s in enumerate(idx):
            for t in range(T):
                row = t if t < n_vis else t + (T_c - T)
                assert (out[b, t] == s * T_c + row).all()
    out = TC.reference_gather([code], [1, M, -1], 7, n_vis)[0]
    assert out[1:].isnan().all() and not out[0].isnan().any()


def test_gather_entry_point_rejects_bad_arguments_without_a_gpu():
    p = 1 << 20                                             # never dereferenced: every check runs before CUDA
    ok = dict(out_ptrs=[p], cache_ptrs=[p], idx=[0], B=1, M=4, T=10, T_c=12, n_vis=8, D=64, dtype_code=1, stream=None)
    bad = [dict(out_ptrs=[], cache_ptrs=[]), dict(idx=None), dict(B=0), dict(M=0), dict(M=1 << 31), dict(T=13),
           dict(n_vis=11), dict(n_vis=-1), dict(D=0), dict(dtype_code=3), dict(out_ptrs=[0]), dict(cache_ptrs=[p + 1]),
           dict(out_ptrs=[p + 2], dtype_code=0)]
    for change in bad:
        with pytest.raises(MafedDistillError, match="invalid argument"):
            TC.gather_raw(**{**ok, **change})
    assert TC.load().mafed_teacher_gather_abi_version() == TC.ABI_VERSION


def test_gather_rejects_python_indices_out_of_range_before_the_launch():
    cache = [torch.zeros(3, 10, 4)]
    with pytest.raises(MafedDistillError, match="memory index 3 out of range"):
        TC.gather(cache, [0, 3], 10, 8)
    with pytest.raises(MafedDistillError, match="memory index -1"):
        TC.gather(cache, [-1], 10, 8)
    with pytest.raises(MafedDistillError, match="does not fit"):
        TC.gather(cache, [0], 11, 8)


def _gloo_worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from torch.utils.data.distributed import DistributedSampler
    fd = _make(True, process_group=False)
    fd._update_memory(VLSamples(40, seed=1))
    fd._update_memory(VLSamples(30, seed=2))
    assert isinstance(fd.mem_sampler, DistributedSampler)
    seen = []
    for epoch in range(2):
        fd.mem_sampler.set_epoch(epoch)
        seen.append(_check_indices(fd, fd.mem_dataloader))
    ret[rank] = seen
    dist.destroy_process_group()


def test_loader_yields_memory_indices_under_a_distributed_sampler():
    ret = mp.Manager().dict()
    port = 29900 + os.getpid() % 90
    mp.spawn(_gloo_worker, args=(2, port, ret), nprocs=2, join=True)
    for epoch in range(2):
        assert sorted(ret[0][epoch] + ret[1][epoch]) == list(range(12))   # the ranks' shards cover the memory
    assert ret[0][0] != ret[0][1]                                          # reshuffled per epoch
