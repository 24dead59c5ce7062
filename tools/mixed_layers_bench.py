#!/usr/bin/env python
"""A step over layers of two dtypes at the C4 shard (VLPythia-1B held in bf16: B=64, T=256+32, D=2048, every row
live; 15 bf16 hidden states and the fp32 output of the final layer norm, 16 distilled layers), timed through
``FeatureDistillation.distill`` + ``backward``:

  grouped    -- the states as they are: one launch per dtype group, bf16 (6 * D bytes per token*layer: read student 2,
                teacher 2, write gradient 2) and fp32 (12 * D)
  upcast     -- every state cast with ``.float()`` by the caller first, the path such a step took before it was split:
                per bf16 layer 30 * D (casts of student and teacher 12, the fp32 step 12, autograd's cast of the gradient
                back to bf16 6), the fp32 layer 12 * D
  bf16_alone, fp32_alone -- each group's launch alone through ``distill_loss`` with the sub-plan the grouped step uses
                (the first one also writes the modality masks, as in the grouped step); ``groups_alone_sum`` adds them.
                ``grouped_distill_loss`` is the grouped step through the same call, for the comparison without the
                strategy's host bookkeeping.

Timed region as in bench.py: warm-up steps, one untimed step, then CUDA events around ``--steps`` steps.  The arms
alternate within each of ``--rounds`` rounds; the median round is reported.  GB/s is the byte basis above over the
measured time.  Peak memory: ``max_memory_allocated`` during one step above what was allocated before it.  Prints one
JSON object (card name, power limit and max SM clock read in the same run).

    python tools/mixed_layers_bench.py [--steps 20] [--warmup 5] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

N_BF16, B, TXT, N_VIS, D = 15, 64, 32, 256, 2048
N_SEL = N_BF16 + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    from gpu_util import Out, make_method
    from mafed_b200.distill_op import distill_loss
    from mixed_teacher_bench import card

    g = torch.Generator(device="cuda").manual_seed(0)
    T = N_VIS + TXT
    dtypes = [torch.bfloat16] * N_BF16 + [torch.float32]
    s32 = [torch.randn(B, T, D, device="cuda", generator=g) for _ in range(N_SEL)]
    students = [s.to(d) for s, d in zip(s32, dtypes)]
    teachers = [(s + 0.1 * torch.randn(B, T, D, device="cuda", generator=g)).to(d) for s, d in zip(s32, dtypes)]
    del s32
    mask = torch.ones(B, TXT, dtype=torch.int64, device="cuda")
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=N_SEL,
                layer=None, n_vis=N_VIS, coeff=1.0, cls=False, lang_coeff=None)
    fd = make_method(meta)
    layers = list(fd.loss_weights.get_distillation_layers())
    assert layers == list(range(N_SEL))
    leaves = [s.requires_grad_(True) for s in students]

    def clear():
        for l in leaves:
            l.grad = None

    def api_step(arm):
        clear()
        if arm == "upcast":
            fd.past_model = lambda **kw: Out(tuple(t.float() for t in teachers))
            out = Out(tuple(l.float() for l in leaves))
        else:
            fd.past_model = lambda **kw: Out(tuple(teachers))
            out = Out(tuple(leaves))
        loss = fd.distill(out, {"attention_mask": mask})
        loss.backward()
        return loss

    # the grouped step's sub-plans, as distill_loss builds them
    api_step("grouped")
    plan = fd._step_plan(layers)
    (idx_a, plan_a), (idx_b, plan_b) = plan.split(tuple((s.dtype, t.dtype) for s, t in zip(students, teachers)))[0]
    assert idx_a == list(range(N_BF16)) and idx_b == [N_BF16]
    masks = torch.empty(2, B, T, dtype=torch.int64, device="cuda")

    def call_step(arm):
        clear()
        if arm == "grouped_distill_loss":
            total, _ = distill_loss(leaves, teachers, mask, plan, group=False, teachers_detached=True, mask_out=masks)
        else:
            idx, sub = (idx_a, plan_a) if arm == "bf16_alone" else (idx_b, plan_b)
            total, _ = distill_loss([leaves[i] for i in idx], [teachers[i] for i in idx], mask, sub, group=False,
                                    teachers_detached=True, mask_out=masks if arm == "bf16_alone" else None)
        total.backward()
        return total

    arms = {"grouped": api_step, "upcast": api_step, "grouped_distill_loss": call_step, "bf16_alone": call_step,
            "fp32_alone": call_step}

    def timed(arm):
        step = arms[arm]
        for _ in range(args.warmup):
            step(arm)
        torch.cuda.synchronize()
        step(arm)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(arm)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    def peak(arm):
        clear()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        arms[arm](arm)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    # results before times: the grouped step and the up-cast step give the same gradients (mse), bit for bit
    loss_g = float(api_step("grouped").detach())
    grads_g = [l.grad.clone() for l in leaves]
    loss_u = float(api_step("upcast").detach())
    same_grads = all(torch.equal(a, l.grad) for a, l in zip(grads_g, leaves))
    del grads_g
    peaks = {arm: peak(arm) for arm in arms}

    name, power = card()
    rows = {arm: [] for arm in arms}
    for _ in range(args.rounds):
        for arm in arms:
            rows[arm].append(timed(arm))
    rows_elems = B * T * D
    basis = {"grouped": 6 * N_BF16 + 12, "upcast": 30 * N_BF16 + 12, "grouped_distill_loss": 6 * N_BF16 + 12,
             "bf16_alone": 6 * N_BF16, "fp32_alone": 12}
    result = {"tool": "mixed_layers_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
              "shape": {"B": B, "T": T, "D": D, "distilled_layers": N_SEL, "bf16_layers": N_BF16, "fp32_layers": 1,
                        "loss": "mse", "rows_live": "all"},
              "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
              "loss": {"grouped": loss_g, "upcast": loss_u, "rel_diff": abs(loss_g - loss_u) / abs(loss_u)},
              "grouped_vs_upcast_gradients_bit_identical": same_grads, "arms": {}}
    for arm in arms:
        ms = statistics.median(rows[arm])
        gb = basis[arm] * rows_elems / 1e9
        result["arms"][arm] = {"bytes_per_token_basis": f"{basis[arm]} * D", "gb_per_step": round(gb, 3),
                               "ms_per_step": round(ms, 4), "gbs": round(gb / (ms * 1e-3), 1),
                               "peak_allocated_gb": round(peaks[arm] / 1e9, 3),
                               "ms_rounds": [round(x, 4) for x in rows[arm]]}
    alone = [a + b for a, b in zip(rows["bf16_alone"], rows["fp32_alone"])]
    result["groups_alone_sum_ms"] = round(statistics.median(alone), 4)
    result["grouped_distill_loss_over_groups_alone_sum"] = round(
        result["arms"]["grouped_distill_loss"]["ms_per_step"] / result["groups_alone_sum_ms"], 4)
    result["grouped_over_groups_alone_sum"] = round(result["arms"]["grouped"]["ms_per_step"] /
                                                    result["groups_alone_sum_ms"], 4)
    result["upcast_over_grouped"] = round(result["arms"]["upcast"]["ms_per_step"] /
                                          result["arms"]["grouped"]["ms_per_step"], 3)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
