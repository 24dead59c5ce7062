#!/usr/bin/env python
"""``FeatureDistillation.distill`` + ``backward`` four ways, at the C4 shard (VLPythia-1B shape: 17 hidden states, the
16 the `discounted` recipe distils, bf16, B=64, T=256+32, D=2048) and at the smallest C5 point (8 samples per GPU, same shape otherwise):

  eager            -- the compiled autograd node (what bench.py times)
  compile          -- ``torch.compile(distill)`` (default mode): the ``mafed::`` ops inside an Inductor graph
  reduce_overhead  -- ``torch.compile(distill, mode="reduce-overhead")``: the same graph replayed as a CUDA graph
  capture          -- ``fd.capture()`` (``GraphedDistillStep``): the path alone captured over static buffers

The compiled variants call ``fd.record_step()`` after each step, the bookkeeping eager ``distill`` does itself.

Per step: ``host_us``, the host time to enqueue ``--steps`` steps (perf_counter from the first call to the last
return, no synchronisation in between) over the steps; ``device_ms``, CUDA events around the same steps over the
steps (the wall per step as the device sees it; a host-bound loop shows its host time here).  The hidden states are
the same static tensors every step (student and teacher states and the mask are marked static for reduce-overhead,
so the CUDA graph reads them in place instead of copying them into its own buffers).  The
variants alternate within each of ``--rounds`` rounds; the median round is reported.  Prints one JSON object with
the card's name and power limit read in the same run.

``--profile FILE`` also writes, per point and variant, torch.profiler's host-side table of ten steps (run after the
timed rounds, so the tracing does not touch the timings): where the host time of a step goes.

    python tools/compiled_step_bench.py [--steps 50] [--warmup 10] [--rounds 5] [--out FILE] [--profile FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_TUPLE, TXT, N_VIS, D = 17, 32, 256, 2048
POINTS = {"C4_shard_B64": 64, "C5_smallest_B8": 8}
VARIANTS = ("eager", "compile", "reduce_overhead", "capture")
META = dict(modality="balanced", layer_strategy="discounted", loss="mse", gamma=0.5, num_hidden_layers=N_TUPLE - 1,
            layer=None, n_vis=N_VIS)


def card():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}",
                              "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def make_runners(B):
    from gpu_util import Out, make_method
    g = torch.Generator(device="cuda").manual_seed(B)
    T = N_VIS + TXT
    students = [torch.randn(B, T, D, device="cuda", generator=g, dtype=torch.bfloat16) for _ in range(N_TUPLE)]
    teachers = [s + 0.1 * torch.randn(B, T, D, device="cuda", generator=g, dtype=torch.bfloat16) for s in students]
    am = torch.ones(B, TXT, dtype=torch.int64, device="cuda")
    for b in range(B):
        am[b, : b % TXT] = 0
    runners = {}
    for v in VARIANTS:
        fd = make_method(META)
        fd.populate_batch_masks = False
        fd.past_model = lambda **kw: Out(tuple(teachers))
        layers = fd.loss_weights.get_distillation_layers()
        leaves = [s.detach().requires_grad_(i in layers) for i, s in enumerate(students)]
        batch = {"attention_mask": am}
        if v == "capture":
            step = fd.capture(students, teachers, am)
            runners[v] = step.replay
            continue
        fd.distill(Out(tuple(leaves)), batch)     # host tables of the plan, built eagerly once
        if v == "reduce_overhead":
            for t in leaves + teachers + [am]:
                torch._dynamo.mark_static_address(t)
        fn = lambda fd=fd, leaves=leaves: fd.distill(Out(tuple(leaves)), batch)
        if v != "eager":
            fn = torch.compile(fn, fullgraph=True, mode="reduce-overhead" if v == "reduce_overhead" else None)

        def run(fn=fn, fd=fd, leaves=leaves, layers=layers, compiled=v != "eager"):
            for l in layers:
                leaves[l].grad = None
            fn().backward()
            if compiled:
                fd.record_step()      # the host bookkeeping eager distill() does itself
        runners[v] = run
    return runners


def time_one(run, steps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    host = time.perf_counter() - t0
    end.record()
    torch.cuda.synchronize()
    return host / steps * 1e6, start.elapsed_time(end) / steps


def profile_tables(point, runners, steps=10):
    from torch.profiler import ProfilerActivity, profile
    out = []
    for v, run in runners.items():
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU]) as prof:
            for _ in range(steps):
                run()
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="self_cpu_time_total", row_limit=25, max_name_column_width=70)
        out.append(f"==== {point} / {v}: {steps} steps\n{table}")
    return "\n".join(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    name, power = card()
    result = {"gpu": name, "power_limit,max_sm_clock": power, "torch": torch.__version__, "steps": args.steps,
              "rounds": args.rounds, "points": {}}
    tables = []
    for point, B in POINTS.items():
        runners = make_runners(B)
        for run in runners.values():
            for _ in range(args.warmup):
                run()
        torch.cuda.synchronize()
        rounds = {v: [] for v in VARIANTS}
        for _ in range(args.rounds):
            for v in VARIANTS:
                rounds[v].append(time_one(runners[v], args.steps))
        if args.profile:
            tables.append(profile_tables(point, runners))
        res = {}
        for v in VARIANTS:
            host = statistics.median(r[0] for r in rounds[v])
            dev = statistics.median(r[1] for r in rounds[v])
            res[v] = {"host_us": round(host, 2), "device_ms": round(dev, 4)}
        from gpu_util import make_method
        n_layers = len(make_method(META).loss_weights.get_distillation_layers())
        result["points"][point] = {"B": B, "T": N_VIS + TXT, "D": D, "layers": n_layers, "dtype": "bf16",
                                   "variants": res}
        del runners
        torch._dynamo.reset()
        torch.cuda.empty_cache()
    if args.profile:
        with open(args.profile, "w") as f:
            f.write(f"{name}, power limit / max SM clock {power}, torch {torch.__version__}\n\n" + "\n".join(tables))
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
