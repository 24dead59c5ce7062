#!/usr/bin/env python
"""A whole replay step -- student forward, teacher forward, distillation, backward -- with
``FeatureDistillation(early_exit=False)`` and ``early_exit=True``, on a VLPythia-1B stand-in at the C4 shard.

Model: HF ``GPTNeoXModel`` with VLPythia-1B's decoder shape (L = 16, D = 2048, 8 heads, FFN 8192, vocab 50304) and
seeded random weights, a linear connector for 256 visual tokens and an LM head, with the keyword interface of
``tests/tiny_vl.py`` (no download).  fp32 weights under ``replay()``'s bf16 autocast; B = 64, 32 text tokens
(T = 288, every row live).  The teacher is the same weights plus noise, shared by every strategy.

Cases: ``discounted`` over 15 hidden states (0..14: the last distilled entry is the input of layer 14, so layers 14
and 15, the final norm and the LM head are what early exit saves), ``single`` at layer 8, and ``discounted`` with
``replay_coeff=0`` (no replay loss: the student forward stops too).

Per step: CUDA events around the teacher forward (``_past_states``, inside ``distill``) and around ``replay()`` +
``backward()``, and ``torch.cuda.max_memory_allocated`` (peak reset before each step).  Each round runs every case with
the option off and then on (``--warmup`` untimed steps, then ``--steps`` timed ones, each ending in a synchronise);
the median over ``--rounds`` rounds is reported.  The first step's loss of each case is compared off against on.
Prints one JSON object (card name and power limit read in the same run).

    python tools/replay_step_bench.py [--steps 5] [--warmup 2] [--rounds 3] [--out FILE]
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from tiny_vl import TinyVL  # noqa: E402

FULL = dict(dim=2048, layers=16, heads=8, ffn=8192, vocab=50304, n_vis=256, patch=1024, bsz=64, txt=32)
CASES = {
    "discounted15": dict(distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                         num_hidden_layers=15),
    "single8": dict(distillation_layer_weighing_strategy="single", distillation_layer=8, num_hidden_layers=15),
    "discounted15_no_replay_loss": dict(distillation_layer_weighing_strategy="discounted", distillation_layer=None,
                                        num_hidden_layers=15, replay_coeff=0.0),
}


class VLStandIn(TinyVL):
    """TinyVL's forward (connector tokens, then text, through an HF GPTNeoXModel, then the LM head) at a given shape."""

    def __init__(self, dim, layers, heads, ffn, vocab, n_vis, patch, **_):
        nn.Module.__init__(self)
        from transformers import GPTNeoXConfig, GPTNeoXModel
        cfg = GPTNeoXConfig(hidden_size=dim, num_hidden_layers=layers, num_attention_heads=heads,
                            intermediate_size=ffn, vocab_size=vocab, max_position_embeddings=2048,
                            hidden_dropout=0.0, attention_dropout=0.0)
        self.fp32_island = False
        self.gpt_neox = GPTNeoXModel(cfg)
        self.connector = nn.Linear(patch, dim)
        self.embed_out = nn.Linear(dim, vocab, bias=False)
        self.n_vis = n_vis


class Opts:
    tasks = ["a", "b"]; batch_size = 64; seed = 1; pin_mem = False; accumulate_grad_batches = 1


class FreshBatches:
    """A memory loader that yields a new dict per step (replay pops `labels` and adds the masks to the one it gets)."""

    def __init__(self, batch):
        self.batch = batch

    def __iter__(self):
        yield dict(self.batch)


def build(shape, device, seed=0):
    """Student, teacher (student + noise, frozen) and one memory batch at ``shape``."""
    torch.manual_seed(seed)
    with torch.device(device):
        student = VLStandIn(**shape)
    teacher = copy.deepcopy(student).eval()
    with torch.no_grad():
        for p in teacher.parameters():
            p.add_(0.01 * torch.randn_like(p))
    teacher.requires_grad_(False)
    g = torch.Generator().manual_seed(seed + 1)
    ids = torch.randint(0, shape["vocab"], (shape["bsz"], shape["txt"]), generator=g)
    batch = {"input_ids": ids, "pixel_values": torch.randn(shape["bsz"], shape["n_vis"], shape["patch"], generator=g),
             "attention_mask": torch.ones_like(ids), "labels": ids.clone()}
    return student, teacher, {k: v.to(device) for k, v in batch.items()}


def make_strategy(case, early_exit, teacher, batch, n_vis):
    from mafed_b200.methods import CLMethod
    kw = dict(CASES[case])
    fd = CLMethod["featdistill"](memory_size=64, opts=Opts(), model_type="vlpythia",
                                 distillation_modality_weighing_strategy="balanced", gamma=0.5,
                                 early_exit=early_exit, **kw)
    fd.num_vision_tokens = n_vis
    fd.task_id = 1
    fd.past_model = teacher                 # shared: _update_model would deep-copy 4 GB per strategy
    fd.mem_dataloader = FreshBatches(batch)
    return fd


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
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    student, teacher, batch = build(FULL, "cuda")
    fds = {(c, e): make_strategy(c, e, teacher, batch, FULL["n_vis"]) for c in CASES for e in (False, True)}

    def step(fd):
        """One replay step: (teacher-forward ms, step ms, peak GB, loss)."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        inner = type(fd)._past_states

        def timed_teacher(*a, **kw):
            ev[1].record()
            out = inner(fd, *a, **kw)
            ev[2].record()
            return out

        fd._past_states = timed_teacher
        student.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        ev[0].record()
        loss, _ = fd.replay(student)
        loss.backward()
        ev[3].record()
        torch.cuda.synchronize()
        del fd._past_states
        return (ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[3]), torch.cuda.max_memory_allocated() / 1e9,
                float(loss.detach()))

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
    result = {"tool": "replay_step_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
              "torch": torch.__version__, "shape": FULL, "weights": "fp32, bf16 autocast (replay)",
              "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "cases": {}}
    for c in CASES:
        entry = {"loss_off_equals_on": first_loss[(c, False)] == first_loss[(c, True)],
                 "layers": fds[(c, False)].loss_weights.get_distillation_layers()}
        for e in (False, True):
            r = rows[(c, e)]
            entry["on" if e else "off"] = {
                "teacher_forward_ms": round(statistics.median(r["teacher_ms"]), 3),
                "replay_step_ms": round(statistics.median(r["step_ms"]), 3),
                "peak_allocated_gb": round(max(r["peak_gb"]), 3),
                "teacher_forward_ms_rounds": [round(x, 3) for x in r["teacher_ms"]],
                "replay_step_ms_rounds": [round(x, 3) for x in r["step_ms"]]}
        off, on = entry["off"], entry["on"]
        entry["saved"] = {"teacher_forward_ms": round(off["teacher_forward_ms"] - on["teacher_forward_ms"], 3),
                          "replay_step_ms": round(off["replay_step_ms"] - on["replay_step_ms"], 3),
                          "replay_step_fraction": round(1 - on["replay_step_ms"] / off["replay_step_ms"], 4),
                          "peak_allocated_gb": round(off["peak_allocated_gb"] - on["peak_allocated_gb"], 3)}
        result["cases"][c] = entry
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
