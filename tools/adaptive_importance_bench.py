#!/usr/bin/env python
"""Wall time of one ``compute_adaptive_weights`` pass on a VLPythia-1B stand-in at the C4 shard, with the importances
kept per rank (``process_group=False``, the default) and computed over every rank's shard (``process_group=None``, what
``FeatureDistillation(global_importances=True)`` passes), one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 \
        tools/adaptive_importance_bench.py [--batches 2] [--rounds 5] [--out FILE]

Model and batch: ``tools/replay_step_bench.py``'s stand-in (L = 16, D = 2048, vocab 50304, fp32 weights under the pass's
bf16 autocast), B = 64 and 32 text tokens (T = 288) per batch, importances over 15 hidden states (``discounted``).
Each rank's loader holds ``--batches`` such batches.  After one untimed pass of each, every round times one pass with
the option off and one with it on (host clock around the pass, a device synchronise and a barrier on each side); the
median over ``--rounds`` rounds is reported, with rank 0's card name and power limit read in the same run.  On one rank
there is nothing to exchange and only the option-off time is measured.  Prints one JSON object.
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from replay_step_bench import FULL, VLStandIn, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29531")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    from mafed_b200.methods import DistillationWeights

    torch.manual_seed(0)
    with torch.device("cuda"):
        model = VLStandIn(**FULL)
    g = torch.Generator().manual_seed(1 + rank)
    batches = []
    for _ in range(args.batches):
        ids = torch.randint(0, FULL["vocab"], (FULL["bsz"], FULL["txt"]), generator=g)
        b = {"input_ids": ids, "pixel_values": torch.randn(FULL["bsz"], FULL["n_vis"], FULL["patch"], generator=g),
             "attention_mask": torch.ones_like(ids), "labels": ids.clone()}
        batches.append({k: v.cuda() for k, v in b.items()})
    dw = DistillationWeights("adaptive", "discounted", num_hidden_layers=15, distillation_layer=None,
                             num_vision_tokens=FULL["n_vis"])
    modes = {"off": False} if world == 1 else {"off": False, "on": None}

    def one_pass(group):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        imp = dw.compute_adaptive_weights(model, [dict(b) for b in batches], process_group=group)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        dist.barrier()
        return ms, imp

    first = {m: one_pass(group)[1] for m, group in modes.items()}
    times = {m: [] for m in modes}
    for _ in range(args.rounds):
        for m, group in modes.items():
            times[m].append(one_pass(group)[0])
    name, power = card()
    result = {"tool": "adaptive_importance_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
              "torch": torch.__version__, "ranks": world, "shape": FULL, "batches_per_rank": args.batches,
              "hidden_states": 15, "weights": "fp32, bf16 autocast", "rounds": args.rounds, "rank": rank}
    for m in modes:
        result[m] = {"pass_ms": round(statistics.median(times[m]), 3), "pass_ms_rounds": [round(x, 3) for x in times[m]]}
    if world == 1:
        result["on"] = "not measured (one rank: nothing to exchange)"
    else:
        result["on_minus_off_ms"] = round(result["on"]["pass_ms"] - result["off"]["pass_ms"], 3)
        every = [None] * world
        dist.all_gather_object(every, first["on"].cpu().tolist())
        result["on_lang_coeff_same_on_all_ranks"] = all(e == every[0] for e in every)
    dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(result))
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
