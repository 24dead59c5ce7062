#!/usr/bin/env python
"""The teacher cache replicated on every rank (``teacher_cache=True``) against the cache sharded across the ranks
(``shard_teacher_cache=True``), one process per GPU of one box, on the VLPythia-1B stand-in of
``tools/teacher_cache_bench.py`` at the C4 shard (B = 64 per rank, 256 visual + 32 text tokens, a 500-sample memory,
``discounted`` over 15 states):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29541 \\
        tools/sharded_teacher_cache_bench.py [--steps 5] [--warmup 2] [--rounds 3] [--memory 500] \\
        [--parent-lib LIB] [--out FILE]

Per rank: the cache's bytes and build seconds (host clock around a synchronised build), the gather of the rank's batch
from the replicated and from the sharded cache (CUDA events around ``--gathers`` back-to-back calls, alternating, median),
and the
whole batch-sharded replay step (``replay()`` + ``backward()``, CUDA events) for three arms alternating in each round:
uncached (teacher forward), replicated cache, sharded cache.  The sharded gather is compared with the replicated one bit
for bit, and the first step's loss and gradients with the replicated arm's (next to the replicated arm against itself).
``--parent-lib`` names a build of ``libmafed_teacher_gather.so`` at ABI 1 (the one-rank gather before the sharded
kernel): its ``mafed_teacher_gather`` and this build's, called with the same arguments, are timed alternating.  At the end each rank measures the device memory
that releasing its shard returns.  Rank 0 prints one JSON object (card name and power limit read in the same run).
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from replay_step_bench import FULL, build, card  # noqa: E402
from teacher_cache_bench import FreshBatches, Memory, make_strategy  # noqa: E402


def timed(fn, reps):
    """ms per call of ``fn()`` over ``reps`` calls issued back to back between two CUDA events (the queue stays full, so
    host time between launches is hidden as it is in a step)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--gathers", type=int, default=20)
    ap.add_argument("--memory", type=int, default=500)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    from mafed_b200 import teacher_cache as TC
    from mafed_b200.teacher_cache import IndexedCollate
    from teacher_cache_bench import collate

    student, teacher, _ = build(FULL, "cuda")
    memory = Memory(args.memory, FULL)
    picked = torch.randperm(args.memory, generator=torch.Generator().manual_seed(7 + rank))[: FULL["bsz"]].tolist()
    host = IndexedCollate(collate)([(i, memory[i]) for i in picked])
    batch_on = {k: v.cuda() if torch.is_tensor(v) else v for k, v in host.items()}
    batch_off = {k: v for k, v in batch_on.items() if k != "memory_index"}

    arms = {"uncached": make_strategy("discounted15", False, False, teacher, memory),
            "replicated": make_strategy("discounted15", False, True, teacher, memory),
            "sharded": make_strategy("discounted15", False, True, teacher, memory)}
    arms["sharded"].shard_teacher_cache = True
    arms["uncached"].mem_dataloader = FreshBatches(batch_off)
    res = {"rank": rank}
    for name in ("replicated", "sharded"):
        fd = arms[name]
        fd.mem_dataloader = FreshBatches(batch_on)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fd._build_teacher_cache()
        torch.cuda.synchronize()
        res[f"{name}_build_s"] = round(time.perf_counter() - t0, 3)
        res[f"{name}_cache_bytes"] = fd._teacher_cache.nbytes
    rep, shd = arms["replicated"]._teacher_cache, arms["sharded"]._teacher_cache
    res["samples_held"] = shd.count[rank] if isinstance(shd, TC.ShardedTeacherCache) else shd.states[0].shape[0]
    layers = arms["replicated"].loss_weights.get_distillation_layers()
    T = FULL["n_vis"] + FULL["txt"]
    res["gather_bit_identical"] = all(torch.equal(a, b) for a, b in zip(rep.gather(picked, T, layers),
                                                                         shd.gather(picked, T, layers)))
    res["gather_rows_from_peers"] = sum(shd.owner[i] != rank for i in picked) if world > 1 else 0
    res["gather_bytes"] = sum(s.element_size() * s.shape[-1] for s in rep.states) * T * len(picked)
    g_rep, g_shd = [], []
    for _ in range(3):
        g_rep.append(timed(lambda: rep.gather(picked, T, layers), args.gathers))
        g_shd.append(timed(lambda: shd.gather(picked, T, layers), args.gathers))
    res["gather_ms"] = {"replicated": round(statistics.median(g_rep), 3), "sharded": round(statistics.median(g_shd), 3)}
    if args.parent_lib:
        lib = ctypes.CDLL(args.parent_lib)
        assert lib.mafed_teacher_gather_abi_version() == 1
        lib.mafed_teacher_gather.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                             ctypes.POINTER(ctypes.c_int64)] + [ctypes.c_int] * 2 + [ctypes.c_int64] + \
                                            [ctypes.c_int] * 5 + [ctypes.c_void_p]
        M, T_c, D = rep.states[0].shape
        out = [torch.empty((len(picked), T, D), dtype=s.dtype, device="cuda") for s in rep.states]
        vp = ctypes.c_void_p * len(out)
        outs, caches, ix = vp(*[o.data_ptr() for o in out]), vp(*[s.data_ptr() for s in rep.states]), \
            (ctypes.c_int64 * len(picked))(*picked)
        code = TC._DTYPES[rep.states[0].dtype]
        stream = torch.cuda.current_stream().cuda_stream

        def call(lib):
            assert lib.mafed_teacher_gather(outs, caches, ix, len(out), len(picked), M, T, T_c, FULL["n_vis"], D, code,
                                            stream) == 0

        this = TC.load()
        call(lib)
        same = all(torch.equal(a, b) for a, b in zip(out, rep.gather(picked, T, layers)))
        p_ms, n_ms = [], []
        for _ in range(7):
            p_ms.append(timed(lambda: call(lib), args.gathers))
            n_ms.append(timed(lambda: call(this), args.gathers))
        res["one_rank_gather_ms"] = {"what": "mafed_teacher_gather of the replicated cache, same prebuilt arguments",
                                     "parent_build": [round(x, 4) for x in p_ms], "this_build": [round(x, 4) for x in n_ms],
                                     "parent_median": round(statistics.median(p_ms), 4),
                                     "this_median": round(statistics.median(n_ms), 4), "outputs_equal": same}

    def step(fd, grads=False):
        student.zero_grad(set_to_none=True)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        loss, _ = fd.replay(student)
        loss.backward()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), loss.detach(), [p.grad.clone() if grads and p.grad is not None else None
                                                  for p in student.parameters()] if grads else None

    def diff(x, y):
        return {"loss_equal": bool(torch.equal(x[0], y[0])),
                "max_abs_grad_diff": max(float((a - b).abs().max()) for a, b in zip(x[1], y[1]) if a is not None)}

    first = {k: step(fd, grads=True)[1:] for k, fd in arms.items()}
    again = step(arms["replicated"], grads=True)[1:]
    # the stand-in's attention backward is not bit-reproducible run to run, so the replicated arm against itself is the
    # yardstick of the sharded arm's gradient difference (the tests check bit-identity with the math backend)
    res["first_step"] = {"sharded_vs_replicated": diff(first["sharded"], first["replicated"]),
                         "replicated_vs_itself": diff(again, first["replicated"])}
    del first, again
    rows = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fd in arms.items():
            for _ in range(args.warmup):
                step(fd)
            rows[k].append(statistics.median(step(fd)[0] for _ in range(args.steps)))
    res["replay_step_ms"] = {k: round(statistics.median(v), 3) for k, v in rows.items()}
    res["replay_step_ms_rounds"] = {k: [round(x, 3) for x in v] for k, v in rows.items()}
    ms = res["replay_step_ms"]
    saved_rep, saved_shd = ms["uncached"] - ms["replicated"], ms["uncached"] - ms["sharded"]
    res["saved_ms"] = {"replicated": round(saved_rep, 3), "sharded": round(saved_shd, 3),
                       "sharded_over_replicated": round(saved_shd / saved_rep, 4) if saved_rep > 0 else None}
    if isinstance(shd, TC.ShardedTeacherCache):
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        shd.release()
        res["release_returned_bytes"] = torch.cuda.mem_get_info()[0] - free0
    every = [None] * world
    dist.all_gather_object(every, res)
    if rank == 0:
        name, power = card()
        result = {"tool": "sharded_teacher_cache_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
                  "gpus": world, "torch": torch.__version__, "shape": FULL, "memory_samples": args.memory,
                  "case": "discounted15", "weights": "fp32, bf16 autocast (replay)", "steps": args.steps,
                  "warmup": args.warmup, "rounds": args.rounds, "gathers": args.gathers, "ranks": every}
        print(json.dumps(result))
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(json.dumps(result, indent=1) + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
