#!/usr/bin/env python
"""The distillation step of a cached replay batch, three ways, at the C4 shard (B = 64, 256 visual + 32 text tokens,
D = 2048, 15 hidden states, every row live) with a teacher cache of M = 500 memory samples (T_c = T = 288):

* ``gather``: ``teacher_cache.gather`` (``mafed_teacher_gather``) into fresh [B, T, D] tensors, then ``distill_loss``
  on them -- what a cached replay step ran before the step could read the cache;
* ``fused``: ``cached_distill_loss`` -- the one-pass step reading the teacher rows straight from the cache;
* ``pregathered``: ``distill_loss`` on tensors gathered once, outside the timed region (the floor of the two above).

Each step includes its backward (``torch.autograd.grad`` at the assumed upstream gradient: the gate / fix-up that
finds nothing to fix).  States in bf16 and in fp32, mse and cosine.  Each round runs every arm (``--warmup`` untimed
steps, then ``--steps`` steps between two CUDA events) in turn; the median over ``--rounds`` rounds is reported, with
the algorithmic bytes of each arm (student + teacher read and gradient written: 3 L B T D e; the gather adds a read
and a write of the teacher rows, 2 L B T D e) and the peak memory a step allocates above what is resident
(``max_memory_allocated``, peak reset before one step).  The losses and gradients of the three arms are compared
bitwise.  Prints one JSON object (card name, power limit and max SM clock read in the same run).

    python tools/cached_step_bench.py [--steps 20] [--warmup 3] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from replay_step_bench import card  # noqa: E402

SHAPE = dict(L=15, B=64, n_vis=256, txt=32, D=2048, M=500)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    from mafed_b200 import cabi
    from mafed_b200 import teacher_cache as TC
    from mafed_b200.distill_op import DistillPlan, cached_distill_loss, distill_loss

    s = SHAPE
    L, B, n_vis, D, M = s["L"], s["B"], s["n_vis"], s["D"], s["M"]
    T = T_c = n_vis + s["txt"]
    name, limits = card()
    result = dict(bench="cached_step", gpu=name, power_limit_and_max_sm_clock=limits, shape=dict(s, T=T, T_c=T_c),
                  steps=args.steps, warmup=args.warmup, rounds=args.rounds, cases={})
    idx = torch.randperm(M, generator=torch.Generator().manual_seed(7))[:B].tolist()
    mask = torch.ones((B, T - n_vis), dtype=torch.int64, device="cuda")
    for dtype in (torch.bfloat16, torch.float32):
        e = torch.empty((), dtype=dtype).element_size()
        g = torch.Generator(device="cuda").manual_seed(1)
        cache = [torch.randn((M, T_c, D), generator=g, device="cuda").to(dtype) for _ in range(L)]
        students = [torch.randn((B, T, D), generator=g, device="cuda").to(dtype).requires_grad_(True) for _ in range(L)]
        pre = TC.gather(cache, idx, T, n_vis)
        for loss in ("mse", "cosine"):
            plan = DistillPlan(layers=list(range(L)), layer_coeffs=[1.0 / (l + 1) for l in range(L)], distill_coeff=1.0,
                               modality_kind=cabi.MODW_TABLE, lang_weights=[0.5] * L, n_vis=n_vis,
                               loss_kind=cabi.LOSS_COSINE if loss == "cosine" else cabi.LOSS_MSE)

            def gather_step():
                total, _ = distill_loss(students, TC.gather(cache, idx, T, n_vis), mask, plan)
                return total, torch.autograd.grad(total, students)

            def fused_step():
                total, _ = cached_distill_loss(students, cache, idx, T_c, mask, plan)
                return total, torch.autograd.grad(total, students)

            def pregathered_step():
                total, _ = distill_loss(students, pre, mask, plan)
                return total, torch.autograd.grad(total, students)

            arms = {"gather": gather_step, "fused": fused_step, "pregathered": pregathered_step}
            outs = {k: fn() for k, fn in arms.items()}
            torch.cuda.synchronize()
            bitwise = all(torch.equal(outs[k][0], outs["gather"][0]) and
                          all(torch.equal(a, b) for a, b in zip(outs[k][1], outs["gather"][1])) for k in arms)
            del outs
            peak = {}
            for k, fn in arms.items():
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                fn()
                torch.cuda.synchronize()
                peak[k] = torch.cuda.max_memory_allocated() - base
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, fn in arms.items():
                    for _ in range(args.warmup):
                        fn()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(args.steps):
                        fn()
                    b.record()
                    b.synchronize()
                    times[k].append(a.elapsed_time(b) / args.steps)
            ms = {k: statistics.median(v) for k, v in times.items()}
            step_bytes = 3 * L * B * T * D * e
            gather_bytes = 2 * L * B * T * D * e
            case = dict(ms_per_step=ms, ms_per_step_rounds=times,
                        algorithmic_bytes=dict(gather=step_bytes + gather_bytes, fused=step_bytes, pregathered=step_bytes),
                        gathered_bytes=L * B * T * D * e, peak_allocated_bytes=peak, bitwise_equal=bitwise,
                        fused_over_pregathered=ms["fused"] / ms["pregathered"],
                        gather_time_saved=(ms["gather"] - ms["fused"]) / max(ms["gather"] - ms["pregathered"], 1e-9),
                        peak_saved_bytes=peak["gather"] - peak["fused"])
            result["cases"][f"{str(dtype).split('.')[-1]}_{loss}"] = case
            print(f"{dtype} {loss}: " + ", ".join(f"{k} {v:.3f} ms" for k, v in ms.items()) +
                  f"; peak saved {case['peak_saved_bytes'] / 1e9:.2f} GB; bitwise {bitwise}", file=sys.stderr)
        del cache, students, pre
        torch.cuda.empty_cache()
    text = json.dumps(result)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
