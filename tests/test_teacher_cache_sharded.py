"""Host side of ``FeatureDistillation(teacher_cache=True, shard_teacher_cache=True)`` (no GPU): the owner map and shard
layout, the argument checks of the sharded exports, the option's validation, its single-rank fall-back to the replicated
cache, the collective release of the previous shards, and the build's one-host and failed-allocation checks, which raise
on every rank together."""
import os
import re
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mafed_b200 import teacher_cache as TC
from mafed_b200.cabi import MafedDistillError
from mafed_b200.methods import FeatureDistillation
from vl_memory import VLSamples, collate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 42; pin_mem = False; accumulate_grad_batches = 1


def _make(memory_size=12, **kw):
    fd = FeatureDistillation(memory_size, Opts(), "vlpythia", distillation_modality_weighing_strategy="balanced",
                             distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                             num_hidden_layers=3, **kw)
    fd.num_workers = 0
    fd.num_vision_tokens = 8
    fd.data_hooks = (collate, lambda loader: loader)
    return fd


@pytest.mark.parametrize("M,bs,N", [(500, 64, 8), (500, 64, 2), (12, 4, 3), (13, 4, 2), (10, 4, 8), (1, 64, 8),
                                    (64, 64, 2), (7, 1, 3), (0, 4, 2)])
def test_owner_map_follows_the_build_batches(M, bs, N):
    rank, slot, count = TC.shard_owners(M, bs, N)
    assert len(rank) == len(slot) == M and len(count) == N and sum(count) == M
    # restate it: build batch k goes to rank k % N, whose batches fill its slots in order
    want = {}
    filled = [0] * N
    for k, lo in enumerate(range(0, M, bs)):
        for i in range(lo, min(lo + bs, M)):
            want[i] = (k % N, filled[k % N])
            filled[k % N] += 1
    assert [(rank[i], slot[i]) for i in range(M)] == [want[i] for i in range(M)]
    assert count == filled
    assert len(set(zip(rank, slot))) == M
    assert all(0 <= s < count[r] for r, s in zip(rank, slot))
    n_batches = -(-M // bs)
    assert [c == 0 for c in count] == [r >= n_batches for r in range(N)]      # fewer batches than ranks: empty shards
    with pytest.raises(ValueError):
        TC.shard_owners(M, 0, N)


def test_shard_layout_is_aligned_and_disjoint():
    for capacity, T_c, D, sizes in [(64, 288, 2048, [2] * 15 + [4]), (3, 7, 9, [2, 4, 2]), (1, 1, 1, [2])]:
        offsets, nbytes = TC.shard_layout(capacity, T_c, D, sizes)
        ends = [o + capacity * T_c * D * e for o, e in zip(offsets, sizes)]
        assert all(o % 256 == 0 for o in offsets) and offsets[0] == 0
        assert all(e <= o for e, o in zip(ends, offsets[1:])) and ends[-1] <= nbytes and nbytes % 256 == 0


def test_sharded_entry_points_reject_bad_arguments_without_a_gpu():
    p = 1 << 20                                             # never dereferenced: every check runs before CUDA
    ok = dict(out_ptrs=[p, p], bases=[p, p + 256], layer_off=[0, 512], src_rank=[0, 1], slot=[0, 0], B=2, slots=4,
              T=10, T_c=12, n_vis=8, D=64, dtype_code=1, stream=None)
    bad = [dict(bases=[]), dict(bases=[p] * 17), dict(out_ptrs=None), dict(bases=None), dict(layer_off=None),
           dict(src_rank=None), dict(slot=None), dict(bases=[p, 0]), dict(bases=[p, p + 1]),
           dict(bases=[p, p + 2], dtype_code=0), dict(layer_off=[0, 3]), dict(layer_off=[0, -2]), dict(out_ptrs=[p, 0]),
           dict(out_ptrs=[]), dict(B=0), dict(slots=0), dict(slots=1 << 31), dict(T=13), dict(n_vis=11),
           dict(n_vis=-1), dict(D=0), dict(dtype_code=3)]
    for change in bad:
        with pytest.raises(MafedDistillError, match="invalid argument"):
            TC.gather_sharded_raw(**{**ok, **change})
    lib = TC.load()
    assert lib.mafed_teacher_shard_handle_bytes() == 64
    import ctypes
    h, buf = ctypes.c_void_p(), ctypes.create_string_buffer(64)
    for world, rank, nbytes, out, handle in [(0, 0, 256, buf, h), (17, 0, 256, buf, h), (2, 2, 256, buf, h),
                                             (2, -1, 256, buf, h), (2, 0, 0, buf, h), (2, 0, 256, None, h),
                                             (2, 0, 256, buf, None)]:
        assert lib.mafed_teacher_shard_create(world, rank, nbytes, out,
                                              ctypes.byref(handle) if handle is not None else None) == 1
    assert lib.mafed_teacher_shard_connect(None, buf) == 1
    assert lib.mafed_teacher_shard_base(None, 0, ctypes.byref(h)) == 1
    assert lib.mafed_teacher_shard_destroy(None) == 0


def test_abi_version():
    assert TC.ABI_VERSION == 2 and TC.load().mafed_teacher_gather_abi_version() == 2
    with open(os.path.join(ROOT, "include", "mafed_teacher_gather.h")) as f:
        header = f.read()
    assert re.search(r"#define MAFED_GATHER_ABI_VERSION (\d+)", header).group(1) == "2"
    assert int(re.search(r"#define MAFED_GATHER_MAX_RANKS (\d+)", header).group(1)) == TC.MAX_RANKS


def test_option_needs_teacher_cache():
    with pytest.raises(ValueError, match="teacher_cache"):
        _make(shard_teacher_cache=True)
    assert _make(teacher_cache=True).shard_teacher_cache is False


def test_one_rank_builds_the_replicated_cache(monkeypatch):
    """No process group: nothing to shard; the option builds ``build``'s cache, with the same values."""
    from tiny_vl import TinyVL
    monkeypatch.setattr(TC, "build_sharded", lambda *a, **k: pytest.fail("no sharded build on one rank"))
    torch.manual_seed(0)
    teacher = TinyVL(fp32_island=True).eval()
    caches = []
    for shard in (True, False):
        fd = _make(teacher_cache=True, shard_teacher_cache=shard, process_group=False if shard else None)
        fd.loss_weights.update_weights = lambda *a, **k: None
        fd.update(dataset=VLSamples(40, seed=1, max_txt=9), model=teacher, dataloader=None)
        assert type(fd._teacher_cache) is TC.TeacherCache
        caches.append(fd._teacher_cache)
    assert all(torch.equal(a, b) for a, b in zip(caches[0].states, caches[1].states))


class _FakeShards(TC.ShardedTeacherCache):
    def __init__(self, log, task):
        self.log, self.task = log, task

    def release(self):
        self.log.append(("release", self.task))


def test_previous_shards_are_released_before_the_next_build(monkeypatch):
    from mafed_b200.methods import distillation as D
    log = []

    def build_sharded(strategy, group):
        log.append(("build", strategy.task_id))
        return _FakeShards(log, strategy.task_id)

    monkeypatch.setattr(TC, "build_sharded", build_sharded)
    monkeypatch.setattr(D, "resolve_group", lambda group: (True, None))
    fd = _make(teacher_cache=True, shard_teacher_cache=True)
    fd.loss_weights.update_weights = lambda *a, **k: None
    model = torch.nn.Linear(2, 2)
    fd.update(dataset=VLSamples(40, seed=1), model=model, dataloader=None)
    fd.update(dataset=VLSamples(30, seed=2), model=model, dataloader=None)
    assert log == [("build", 0), ("release", 0), ("build", 1)]
    # load_state_dict drops the cache from use; the rebuild on the first replay releases its shards first
    fd.load_state_dict(fd.state_dict(), datasets=[VLSamples(40, seed=1), VLSamples(30, seed=2)])
    assert fd._teacher_cache is None and log[-1] == ("build", 1)
    fd._memory_index = [0, 1]
    with pytest.raises(AttributeError):             # the fake cache has no gather: the rebuild is what is checked
        fd._past_states({"attention_mask": torch.ones(2, 3, dtype=torch.int64)}, [0, 1, 2])
    assert log[-2:] == [("release", 1), ("build", 2)]


def _gloo_worker(rank, world, port, ret, other_host):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from tiny_vl import TinyVL
    if other_host and rank == 1:
        socket.gethostname = lambda: "another-host"
    torch.manual_seed(0)
    fd = _make(teacher_cache=True)
    fd._update_memory(VLSamples(40, seed=1))
    fd._update_memory(VLSamples(30, seed=2))
    fd.past_model = TinyVL().eval()
    try:
        TC.build_sharded(fd)
        ret[rank] = "built"
    except MafedDistillError as exc:
        ret[rank] = str(exc)
    dist.destroy_process_group()


@pytest.mark.parametrize("other_host", [True, False])
def test_build_raises_on_every_rank_together(other_host):
    """Ranks on two hosts, or (on a machine without a GPU) a shard that cannot be allocated: every rank raises, none
    waits for the others in a later collective."""
    if other_host is False and torch.cuda.is_available():
        pytest.skip("the allocation succeeds with a GPU")
    ret = mp.Manager().dict()
    port = 29800 + os.getpid() % 90 + (0 if other_host else 5)
    mp.spawn(_gloo_worker, args=(2, port, ret, other_host), nprocs=2, join=True)
    want = "one host" if other_host else "could not allocate"
    assert want in ret[0] and want in ret[1], dict(ret)
