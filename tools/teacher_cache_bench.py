#!/usr/bin/env python
"""A whole replay step -- student forward, teacher states, distillation, backward -- with
``FeatureDistillation(teacher_cache=False)`` and ``teacher_cache=True``, on the VLPythia-1B stand-in of
``tools/replay_step_bench.py`` at the C4 shard (B = 64, 256 visual + 32 text tokens, every row live).

The episodic memory is 500 seeded samples (32 text tokens each, so T_c = T = 288); the step's batch is 64 of them,
drawn once.  With the option off the step runs the teacher forward (``_past_states``); with it on, ``_past_states``
gathers the batch's rows from the cache (one kernel launch per dtype of the cached layers).  Cases: ``discounted`` over
15 hidden states and ``single`` at layer 8, each with and without ``early_exit``.

Per step: CUDA events around ``_past_states`` (teacher forward, or gather) and around ``replay()`` + ``backward()``, and
``torch.cuda.max_memory_allocated`` (peak reset before each step).  Every case's cache stays allocated through the run,
so the reported peak takes them all out and adds back the case's own cache when the option is on: model, step and,
with the option on, its cache.  Each round
runs every case off and then on (``--warmup`` untimed steps, then ``--steps`` timed ones, each ending in a
synchronise); the median over ``--rounds`` rounds is reported.  The cache build (one teacher pass over the memory, as
``update()`` runs it once per task) is timed with a host clock around a synchronised build, ``--builds`` times per case.
The first step's loss of each case is compared off against on.  Prints one JSON object (card name and power limit read
in the same run).

    python tools/teacher_cache_bench.py [--steps 5] [--warmup 2] [--rounds 3] [--builds 2] [--memory 500] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from replay_step_bench import FULL, build, card  # noqa: E402

CASES = {
    "discounted15": dict(distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                         num_hidden_layers=15),
    "single8": dict(distillation_layer_weighing_strategy="single", distillation_layer=8, num_hidden_layers=15),
}


class Opts:
    tasks = ["a", "b"]; batch_size = 64; seed = 1; pin_mem = False; accumulate_grad_batches = 1


class Memory(torch.utils.data.Dataset):
    """Seeded memory samples at the C4 shard's text length."""

    def __init__(self, n, shape):
        self.n, self.shape = n, shape

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(10_000 + int(i))
        s = self.shape
        ids = torch.randint(0, s["vocab"], (s["txt"],), generator=g)
        return {"input_ids": ids, "pixel_values": torch.randn(s["n_vis"], s["patch"], generator=g),
                "attention_mask": torch.ones_like(ids), "labels": ids.clone()}


def collate(items):
    return {k: torch.stack([it[k] for it in items]) for k in items[0]}


class FreshBatches:
    """A memory loader that yields a new dict per step (replay pops keys and adds the masks to the one it gets)."""

    def __init__(self, batch):
        self.batch = batch

    def __iter__(self):
        yield dict(self.batch)


def make_strategy(case, early_exit, cache, teacher, memory):
    from mafed_b200.methods import CLMethod
    fd = CLMethod["featdistill"](memory_size=len(memory), opts=Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy="balanced", gamma=0.5,
                                 early_exit=early_exit, teacher_cache=cache, **CASES[case])
    fd.num_vision_tokens = FULL["n_vis"]
    fd.task_id = 1
    fd.num_workers = 0
    fd.past_model = teacher                 # shared: _update_model would deep-copy 4 GB per strategy
    fd.datasets = [memory]
    fd.data_hooks = (collate, lambda loader: loader)
    return fd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--builds", type=int, default=2)
    ap.add_argument("--memory", type=int, default=500)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    from mafed_b200.teacher_cache import IndexedCollate
    student, teacher, _ = build(FULL, "cuda")
    memory = Memory(args.memory, FULL)
    picked = torch.randperm(args.memory, generator=torch.Generator().manual_seed(7))[: FULL["bsz"]].tolist()
    host = IndexedCollate(collate)([(i, memory[i]) for i in picked])
    batch_on = {k: v.cuda() if torch.is_tensor(v) else v for k, v in host.items()}
    batch_off = {k: v for k, v in batch_on.items() if k != "memory_index"}

    fds, build_s, cache_bytes = {}, {}, {}
    for c in CASES:
        builder = make_strategy(c, False, True, teacher, memory)
        times = []
        for _ in range(args.builds):
            builder._teacher_cache = None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            builder._build_teacher_cache()
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        build_s[c] = times
        cache_bytes[c] = builder._teacher_cache.nbytes
        for e in (False, True):
            off = make_strategy(c, e, False, teacher, memory)
            off.mem_dataloader = FreshBatches(batch_off)
            on = make_strategy(c, e, True, teacher, memory)
            on._teacher_cache = builder._teacher_cache
            on.mem_dataloader = FreshBatches(batch_on)
            fds[(c, e, False)], fds[(c, e, True)] = off, on
        del builder

    all_caches = sum(cache_bytes.values())

    def step(fd):
        """One replay step: (_past_states ms, step ms, peak GB with the step's own cache only, loss)."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        inner = type(fd)._past_states

        def timed(*a, **kw):
            ev[1].record()
            out = inner(fd, *a, **kw)
            ev[2].record()
            return out

        fd._past_states = timed
        student.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        ev[0].record()
        loss, _ = fd.replay(student)
        loss.backward()
        ev[3].record()
        torch.cuda.synchronize()
        del fd._past_states
        own = fd._teacher_cache.nbytes if fd.teacher_cache else 0
        return (ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[3]),
                (torch.cuda.max_memory_allocated() - all_caches + own) / 1e9, float(loss.detach()))

    first_loss = {k: step(fd)[3] for k, fd in fds.items()}
    name, power = card()
    rows = {k: {"teacher_ms": [], "step_ms": [], "peak_gb": []} for k in fds}
    for _ in range(args.rounds):
        for k, fd in fds.items():            # per case: off, then on
            for _ in range(args.warmup):
                step(fd)
            t, s, m = [], [], []
            for _ in range(args.steps):
                tt, ss, mm, _ = step(fd)
                t.append(tt); s.append(ss); m.append(mm)
            rows[k]["teacher_ms"].append(statistics.median(t))
            rows[k]["step_ms"].append(statistics.median(s))
            rows[k]["peak_gb"].append(max(m))
    result = {"tool": "teacher_cache_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
              "torch": torch.__version__, "shape": FULL, "memory_samples": args.memory,
              "weights": "fp32, bf16 autocast (replay)", "steps": args.steps, "warmup": args.warmup,
              "rounds": args.rounds, "cases": {}}
    for c in CASES:
        for e in (False, True):
            off_loss, on_loss = first_loss[(c, e, False)], first_loss[(c, e, True)]
            entry = {"layers": fds[(c, e, False)].loss_weights.get_distillation_layers(),
                     "cache_bytes": cache_bytes[c], "cache_build_s": [round(x, 3) for x in build_s[c]],
                     "first_loss_off": off_loss, "first_loss_on": on_loss,
                     "first_loss_rel_diff": abs(on_loss - off_loss) / abs(off_loss)}
            for cached in (False, True):
                r = rows[(c, e, cached)]
                entry["on" if cached else "off"] = {
                    ("gather_ms" if cached else "teacher_forward_ms"): round(statistics.median(r["teacher_ms"]), 3),
                    "replay_step_ms": round(statistics.median(r["step_ms"]), 3),
                    "peak_allocated_gb": round(max(r["peak_gb"]), 3),
                    "teacher_states_ms_rounds": [round(x, 3) for x in r["teacher_ms"]],
                    "replay_step_ms_rounds": [round(x, 3) for x in r["step_ms"]]}
            off, on = entry["off"], entry["on"]
            entry["saved"] = {"teacher_states_ms": round(off["teacher_forward_ms"] - on["gather_ms"], 3),
                              "replay_step_ms": round(off["replay_step_ms"] - on["replay_step_ms"], 3),
                              "replay_step_fraction": round(1 - on["replay_step_ms"] / off["replay_step_ms"], 4),
                              "peak_allocated_gb": round(off["peak_allocated_gb"] - on["peak_allocated_gb"], 3)}
            result["cases"][f"{c}{'_early_exit' if e else ''}"] = entry
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
