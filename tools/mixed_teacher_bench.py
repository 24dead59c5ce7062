#!/usr/bin/env python
"""fp32 student hidden states at the C4 shard (VLPythia-1B: 17 hidden states, 15 distilled, B=64, T=256+32, D=2048,
every row live) against three teachers, timed through ``FeatureDistillation.distill`` + ``backward`` (API) and through
the one-pass step's ctypes calls (kernel level):

  fp32      -- an fp32 teacher: 12 * D bytes per token*layer (read student 4, teacher 4, write gradient 4)
  bf16      -- a bf16 teacher read as it is by the kernels: 10 * D bytes (4 + 2 + 4)
  bf16_cast -- the same bf16 teacher cast with ``.float()`` before the step: 18 * D bytes (the cast reads 2 and writes
               4 per element, then the 12-byte step), plus a transient fp32 copy of every teacher layer

Timed region as in bench.py: warm-up steps, one untimed step, then CUDA events around ``--steps`` steps.  The
variants alternate within each of ``--rounds`` rounds; the median round is reported.  GB/s is the byte basis above
over the measured time.  Prints one JSON object (card name and power limit read in the same run).

    python tools/mixed_teacher_bench.py [--steps 20] [--warmup 5] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_TUPLE, N_SEL, B, TXT, N_VIS, D = 17, 15, 64, 32, 256, 2048
VARIANTS = {"fp32": 12, "bf16": 10, "bf16_cast": 18}   # bytes per element of one token*layer row


def card():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}",
                              "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


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
    from mafed_b200.distill_op import distill_backward, distill_fused

    g = torch.Generator(device="cuda").manual_seed(0)
    T = N_VIS + TXT
    students = [torch.randn(B, T, D, device="cuda", generator=g) for _ in range(N_TUPLE)]
    t32 = [s + 0.1 * torch.randn(B, T, D, device="cuda", generator=g) for s in students]
    t16 = [t.bfloat16() for t in t32]
    mask = torch.ones(B, TXT, dtype=torch.int64, device="cuda")
    meta = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=N_SEL,
                layer=None, n_vis=N_VIS, coeff=1.0, cls=False, lang_coeff=None)
    fd = make_method(meta)
    layers = list(fd.loss_weights.get_distillation_layers())
    assert len(layers) == N_SEL
    leaves = [s.requires_grad_(i in layers) for i, s in enumerate(students)]
    st_sel = [students[l].detach() for l in layers]

    def teacher_tuple(v):
        if v == "fp32":
            return tuple(t32)
        if v == "bf16":
            return tuple(t16)
        return tuple(t16[i].float() if i in layers else t16[i] for i in range(N_TUPLE))

    def api_step(v):
        for l in layers:
            leaves[l].grad = None
        fd.past_model = lambda **kw: Out(teacher_tuple(v))
        loss = fd.distill(Out(tuple(leaves)), {"attention_mask": mask})
        loss.backward()
        return loss

    plan = fd._step_plan(layers)             # the tables distill() uses
    grads = [torch.empty_like(s) for s in st_sel]
    gout = torch.ones((), device="cuda")

    def kernel_step(v):
        if v == "bf16_cast":
            te = [t16[l].float() for l in layers]
        else:
            te = [(t32 if v == "fp32" else t16)[l] for l in layers]
        out, scale, ln = distill_fused(st_sel, te, grads, mask, plan, group=False)
        distill_backward(ln, grads, scale, gout, skip_if_equals=plan.assumed_grad_out * plan.grad_multiplier,
                         grad_out_scale=plan.grad_multiplier)
        return out[0]

    def timed(step, v):
        for _ in range(args.warmup):
            step(v)
        torch.cuda.synchronize()
        step(v)                                   # the region opens behind one untimed step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(v)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    # results before times: the bf16 teacher read as it is and the same teacher cast to fp32 give the same step
    losses = {v: float(api_step(v).detach()) for v in VARIANTS}
    api_step("bf16")
    grads_b = [leaves[l].grad.clone() for l in layers]
    api_step("bf16_cast")
    same_grads = all(torch.equal(a, leaves[l].grad) for a, l in zip(grads_b, layers))
    k_loss = {v: float(kernel_step(v)) for v in VARIANTS}

    name, power = card()
    rows = {v: {"api_ms": [], "kernel_ms": []} for v in VARIANTS}
    for _ in range(args.rounds):
        for v in VARIANTS:
            rows[v]["api_ms"].append(timed(api_step, v))
        for v in VARIANTS:
            rows[v]["kernel_ms"].append(timed(kernel_step, v))
    elems = B * T * D * N_SEL
    result = {"tool": "mixed_teacher_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
              "shape": {"B": B, "T": T, "D": D, "distilled_layers": N_SEL, "student": "fp32", "rows_live": "all"},
              "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "elements_per_step": elems,
              "loss_api": losses, "loss_kernel": k_loss,
              "bf16_vs_bf16_cast_gradients_bit_identical": same_grads, "variants": {}}
    for v, basis in VARIANTS.items():
        api, kern = statistics.median(rows[v]["api_ms"]), statistics.median(rows[v]["kernel_ms"])
        gb = basis * elems / 1e9
        result["variants"][v] = {"bytes_per_element_basis": basis, "gb_per_step": round(gb, 3),
                                 "api_ms_per_step": round(api, 4), "kernel_ms_per_step": round(kern, 4),
                                 "api_gbs": round(gb / (api * 1e-3), 1), "kernel_gbs": round(gb / (kern * 1e-3), 1),
                                 "api_ms_rounds": [round(x, 4) for x in rows[v]["api_ms"]],
                                 "kernel_ms_rounds": [round(x, 4) for x in rows[v]["kernel_ms"]]}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
