#!/usr/bin/env python
"""Kernel-level step time for the non-headline variants: cosine loss, fp32 / fp16 hidden states, 'equal'
weights, at the 1B and base shapes (one-pass and two-pass), both kernel families.

    python tools/variants_bench.py [--only cosine_base] [--out FILE]

``--only cosine_base`` runs just the cosine one-pass step at the base shape (the case to profile under ncu).
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mafed_b200 import cabi  # noqa: E402
from mafed_b200.distill_op import DistillPlan, distill_backward, distill_forward, distill_fused  # noqa: E402

dev = torch.device("cuda", 0)


def time_ms(fn, iters=50, warm=8):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "variants_bench.json"))
    args = ap.parse_args()
    cabi.load()
    shapes = [("1B bf16", 15, 64, 2048, torch.bfloat16), ("1B fp32", 15, 32, 2048, torch.float32),
              ("1B fp16", 15, 64, 2048, torch.float16), ("base bf16", 11, 128, 768, torch.bfloat16),
              ("base fp32", 11, 64, 768, torch.float32), ("410M bf16", 23, 128, 1024, torch.bfloat16),
              ("410M fp32", 23, 64, 1024, torch.float32)]
    losses, variants, iters = (cabi.LOSS_MSE, cabi.LOSS_COSINE), (2, 1), 50
    if args.only == "cosine_base":
        shapes, losses, variants, iters = [shapes[3]], (cabi.LOSS_COSINE,), (2,), 6
    out = []
    for name, L, B, D, dtype in shapes:
        T = 288
        g = torch.Generator(device=dev).manual_seed(1)
        st = [torch.randn(B, T, D, generator=g, device=dev).to(dtype) for _ in range(L)]
        te = [(s.float() + 0.1 * torch.randn(B, T, D, generator=g, device=dev)).to(dtype) for s in st]
        grads = [torch.empty_like(s) for s in st]
        am = torch.ones(B, 32, dtype=torch.int64, device=dev)
        gout = torch.ones((), device=dev)
        esize = st[0].element_size()
        units = B * T * L
        for loss in losses:
            plan = DistillPlan(layers=list(range(L)), layer_coeffs=[1.0 / L] * L, modality_kind=cabi.MODW_EQUAL,
                               loss_kind=loss)
            for variant in variants:
                with cabi.tuning(variant=variant):
                    def one():
                        o, s, l = distill_fused(st, te, grads, am, plan, group=False)
                        distill_backward(l, grads, s, gout, skip_if_equals=1.0)

                    def two():
                        o, s, l = distill_forward(st, te, am, plan, group=False)
                        distill_backward(l, grads, s, gout)

                    m1 = time_ms(one, iters=iters, warm=3 if args.only else 8)
                    m2 = time_ms(two, iters=iters) if not args.only else None
                rec = dict(shape=name, loss="mse" if loss == 0 else "cosine", variant="tma" if variant == 2 else "ldg",
                           one_ms=m1, one_gbs=3 * D * esize * units / m1 / 1e6)
                if m2 is not None:
                    rec.update(two_ms=m2, two_gbs=5 * D * esize * units / m2 / 1e6)
                out.append(rec)
                print(json.dumps(rec), flush=True)
        del st, te, grads
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
