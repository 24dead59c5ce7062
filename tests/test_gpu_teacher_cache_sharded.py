"""``FeatureDistillation(teacher_cache=True, shard_teacher_cache=True)`` on the GPU: the sharded gather kernel against the
torch reference gather over the assembled cache (shards as separate allocations of one process), the sharded build and
gather through ``replay()`` against the replicated cache, bit for bit, and two processes on one GPU that build their
shards, map each other's through CUDA IPC and gather rows that sit mostly in the other's shard.  On >= 2 GPUs,
``tools/multirank_check.py --teacher-cache-sharded`` runs one process per GPU."""
import copy
import os
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mafed_b200 import teacher_cache as TC

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bitwise(a, b):
    bits = {4: torch.int32, 2: torch.int16}[a.element_size()]
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(bits), b.view(bits))


def _shards(cache, N, seed, misalign=0):
    """The full ``[M, T_c, D]`` cache split over N separate allocations, samples in a random order of owners and slots,
    at the layout of ``shard_layout`` (each shard's base moved by ``misalign`` bytes)."""
    M, T_c, D = cache[0].shape
    g = torch.Generator().manual_seed(seed)
    owner = torch.randint(0, N, (M,), generator=g).tolist()
    slot, count = [0] * M, [0] * N
    for i in torch.randperm(M, generator=g).tolist():
        slot[i], count[owner[i]] = count[owner[i]], count[owner[i]] + 1
    capacity = max(count)
    sizes = [c.element_size() for c in cache]
    offsets, nbytes = TC.shard_layout(capacity, T_c, D, sizes)
    bufs = [torch.zeros(nbytes + 256, dtype=torch.uint8, device="cuda") for _ in range(N)]
    for r, buf in enumerate(bufs):
        rows = [i for i in range(M) if owner[i] == r]
        for c, o, e in zip(cache, offsets, sizes):
            view = buf[misalign + o: misalign + o + capacity * T_c * D * e].view(c.dtype).view(capacity, T_c, D)
            if rows:
                view[torch.tensor([slot[i] for i in rows], device="cuda")] = c[torch.tensor(rows, device="cuda")]
    return bufs, [b.data_ptr() + misalign for b in bufs], offsets, owner, slot, capacity


def _gather(bases, offsets, owner, slot, capacity, cache, idx, T, n_vis, src=None):
    M, T_c, D = cache[0].shape
    out = [torch.full((len(idx), T, D), 7, dtype=c.dtype, device="cuda") for c in cache]
    ranks = src if src is not None else [owner[i] for i in idx]
    slots = [slot[i] if 0 <= i < M else i for i in idx] if src is None else idx
    for dtype in dict.fromkeys(c.dtype for c in cache):
        pick = [k for k, c in enumerate(cache) if c.dtype == dtype]
        TC.gather_sharded_raw([out[k].data_ptr() for k in pick], bases, [offsets[k] for k in pick], ranks, slots,
                              len(idx), capacity, T, T_c, n_vis, D, TC._DTYPES[dtype],
                              torch.cuda.current_stream().cuda_stream)
    return out


def _cache(L, M, T_c, D, dtypes, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn((M, T_c, D), generator=g, device="cuda").to(dtypes[l % len(dtypes)]) for l in range(L)]


@pytest.mark.parametrize("N", [2, 3, 8])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("L,M,T_c,D,short,n_vis", [(3, 11, 21, 64, 5, 8), (1, 9, 300, 2048, 0, 8),
                                                    (2, 13, 14, 24, 3, 0)])
def test_sharded_gather_matches_reference(N, dtype, L, M, T_c, D, short, n_vis):
    cache = _cache(L, M, T_c, D, [dtype], seed=N)
    bufs, bases, offsets, owner, slot, capacity = _shards(cache, N, seed=N + L)
    idx = [(5 * b + 3) % M for b in range(2 * M)]
    got = _gather(bases, offsets, owner, slot, capacity, cache, idx, T_c - short, n_vis)
    want = TC.reference_gather(cache, idx, T_c - short, n_vis)
    torch.cuda.synchronize()
    assert all(_bitwise(g, w) for g, w in zip(got, want))


@pytest.mark.parametrize("D,misalign", [(9, 2), (6, 4), (12, 8), (8, 16)])
def test_sharded_gather_unaligned_views(D, misalign):
    """Row sizes and shard bases that allow only 2 / 4 / 8 (or 16) byte copy units."""
    cache = _cache(3, 10, 12, D, [torch.bfloat16])
    bufs, bases, offsets, owner, slot, capacity = _shards(cache, 3, seed=D, misalign=misalign)
    idx = list(range(10))[::-1] * 2
    for n_vis, T in ((0, 6), (4, 12), (4, 4)):
        got = _gather(bases, offsets, owner, slot, capacity, cache, idx, T, n_vis)
        assert all(_bitwise(g, w) for g, w in zip(got, TC.reference_gather(cache, idx, T, n_vis)))


def test_sharded_gather_many_samples_many_layers_mixed_dtypes():
    """More than 2048 samples and 64 layers (several launches), bf16 layers next to fp32 ones (a launch per dtype)."""
    cache = _cache(140, 40, 6, 8, [torch.bfloat16, torch.float32])
    bufs, bases, offsets, owner, slot, capacity = _shards(cache, 8, seed=5)
    idx = [(7 * b) % 40 for b in range(2100)]
    for n_vis, T in ((0, 5), (2, 6)):
        got = _gather(bases, offsets, owner, slot, capacity, cache, idx, T, n_vis)
        assert all(_bitwise(g, w) for g, w in zip(got, TC.reference_gather(cache, idx, T, n_vis)))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_sharded_gather_out_of_range_writes_nan_rows(dtype):
    cache = _cache(2, 12, 20, 64, [dtype])
    bufs, bases, offsets, owner, slot, capacity = _shards(cache, 3, seed=9)
    good = [i for i in range(12) if owner[i] == 1][:1] + [i for i in range(12) if owner[i] == 2][:1]
    src = [1, 3, 2, -1, 0, 0]                                    # rank 3 and rank -1 do not exist
    slots = [slot[good[0]], 0, slot[good[1]], 0, capacity, -1]   # slot `capacity` and -1 are outside the shards
    got = _gather(bases, offsets, owner, slot, capacity, cache, slots, 16, 8, src=src)
    want = TC.reference_gather(cache, good, 16, 8)
    torch.cuda.synchronize()
    for g, w in zip(got, want):
        assert g[1:2].isnan().all() and g[3:].isnan().all()
        assert _bitwise(g[[0, 2]], w)


# ---------------------------------------------------------------- the build and the replay step
class Opts:
    tasks = ["a", "b", "c"]; batch_size = 4; seed = 1; pin_mem = False; accumulate_grad_batches = 2


def _strategy(shard, **kw):
    from mafed_b200.methods import CLMethod
    from vl_memory import collate
    fd = CLMethod["featdistill"](memory_size=16, opts=Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy="balanced",
                                 distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                 gamma=0.5, num_hidden_layers=4, distillation_coeff=2.0, teacher_cache=True,
                                 shard_teacher_cache=shard, **kw)
    fd.num_vision_tokens = 8
    fd.num_workers = 0
    fd.data_hooks = (collate, lambda loader: [{k: v.cuda() if torch.is_tensor(v) else v for k, v in b.items()}
                                              for b in loader])
    return fd


def _models():
    from tiny_vl import TinyVL
    torch.manual_seed(0)
    teacher = TinyVL().cuda()
    student = copy.deepcopy(teacher)
    with torch.no_grad():
        for p in student.parameters():
            p.add_(0.02 * torch.randn_like(p))
    return student, teacher


def _step(fd, student, batch):
    model = copy.deepcopy(student)
    fd.mem_dataloader = [batch]
    loss, _ = fd.replay(model)
    (loss / Opts.accumulate_grad_batches).backward()
    torch.cuda.synchronize()
    return loss.detach(), {n: p.grad for n, p in model.named_parameters()}, batch


def test_one_process_sharded_build_and_replay_equal_the_replicated_cache(tmp_path):
    """One rank of a gloo group: the option builds the replicated cache; ``build_sharded`` over that group (the whole
    sharded path: allocation, IPC handle, gather, release) holds the same rows, and a replay step fed from it is
    bit-identical to the ``teacher_cache=True`` step: loss, every gradient, the batch masks."""
    from vl_memory import VLSamples
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/rdv", rank=0, world_size=1)
    try:
        student, teacher = _models()
        plain, shard = _strategy(False), _strategy(True)
        for fd in (plain, shard):
            fd.update(dataset=VLSamples(40, seed=1, max_txt=9), model=teacher, dataloader=None)
        assert type(shard._teacher_cache) is TC.TeacherCache          # one rank: nothing to shard
        shard.past_model = plain.past_model
        shard._teacher_cache = TC.build_sharded(shard)
        assert isinstance(shard._teacher_cache, TC.ShardedTeacherCache)
        for a, b in zip(shard._teacher_cache.local_states, plain._teacher_cache.states):
            assert _bitwise(a, b)
        for drawn in plain.mem_dataloader:
            la, ga, ba = _step(shard, student, dict(drawn))
            lb, gb, bb = _step(plain, student, dict(drawn))
            assert torch.equal(la, lb)
            assert all((ga[n] is None) == (g is None) and (g is None or torch.equal(ga[n], g)) for n, g in gb.items())
            assert all(torch.equal(ba[k], bb[k]) for k in ("lang_masks", "image_masks"))
        shard._teacher_cache.release()
    finally:
        dist.destroy_process_group()


def _ipc_worker(rank, world, rdv, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"file://{rdv}", rank=rank, world_size=world)
    from vl_memory import VLSamples
    out = {}
    try:
        _, teacher = _models()
        fd = _strategy(True)
        prev = None
        for task, seed in enumerate((1, 2)):                    # the second update releases and rebuilds the shards
            fd.update(dataset=VLSamples(40, seed=seed, max_txt=9), model=teacher, dataloader=None)
            cache = fd._teacher_cache
            released = prev is None or (prev._handle is None and prev.local_states == [])
            prev = cache
            full = TC.build(fd)                                  # the replicated cache, same GPU, same batches
            mine = [i for i in range(cache.M) if cache.owner[i] == rank]
            local = all(_bitwise(a, b[mine]) for a, b in zip(cache.local_states, full.states))
            # mostly the other rank's rows, in a mixed order
            idx = [i for i in range(cache.M) if cache.owner[i] != rank][::-1] + mine[:1]
            T = cache.T_c - 2
            got = cache.gather(idx, T, fd.loss_weights.get_distillation_layers())
            want = TC.reference_gather(full.states, idx, T, cache.n_vis)
            torch.cuda.synchronize()
            out[task] = dict(kind=type(cache).__name__, local=local, equal=all(_bitwise(g, w) for g, w in zip(got, want)),
                             remote=sum(cache.owner[i] != rank for i in idx), n=len(idx), count=cache.count,
                             released=released)
            del full, got, want
        fd._teacher_cache.release()
    except Exception as exc:          # reported to the test, which fails with it
        out["error"] = repr(exc)
    ret[rank] = out
    dist.destroy_process_group()


def test_two_processes_on_one_gpu_map_each_others_shards(tmp_path):
    """The real IPC path on one GPU: each process builds its shard over a gloo group, maps the other's, and gathers a
    batch whose rows sit mostly in the other's shard; bit for bit the replicated build's rows.  Only the cache runs
    here: no distillation step, whose in-kernel exchange would make two ranks on one GPU wait on each other."""
    ret = mp.Manager().dict()
    mp.spawn(_ipc_worker, args=(2, str(tmp_path / "rdv"), ret), nprocs=2, join=True)
    for rank in (0, 1):
        res = ret[rank]
        assert "error" not in res, res
        for task in (0, 1):
            r = res[task]
            assert r["kind"] == "ShardedTeacherCache" and r["local"] and r["equal"] and r["released"], r
            assert r["remote"] == r["n"] - 1 and sum(r["count"]) in (8, 16) and r["count"][rank] > 0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_cache_across_gpus():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tools", "multirank_check.py"),
           "--teacher-cache-sharded"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
