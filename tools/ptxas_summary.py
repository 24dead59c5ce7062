#!/usr/bin/env python
"""Registers, stack and spill bytes of every kernel of the main translation unit, as ptxas reports them
(`nvcc -Xptxas=-v`, sm_100a; no GPU needed): one line per kernel family, every TMA-ring kernel, every spilling
kernel.  Usage: python tools/ptxas_summary.py > profiles/<round>_ptxas_summary.txt  (compiles for ~2 minutes)."""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from mafed_b200 import build as b
    src = os.path.join(ROOT, "mafed_b200", "csrc", "distill_abi.cu")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [b._nvcc(), *b.NVCC_FLAGS, "-Xptxas=-v", "-I" + os.path.join(ROOT, "include"),
               "-I" + os.path.join(ROOT, "mafed_b200", "csrc"), "-c", src, "-o", os.path.join(tmp, "abi.o")]
        log = subprocess.run(cmd, capture_output=True, text=True, check=True).stderr.splitlines()
    rows, cur = [], None
    for ln in log:
        m = re.search(r"Compiling entry function '(\S+)' for 'sm_100a'", ln)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", ln)
        if m and cur:
            rows.append({"sym": cur, "stack": int(m.group(1)), "st": int(m.group(2)), "ld": int(m.group(3)), "regs": None})
            continue
        m = re.search(r"Used (\d+) registers", ln)
        if m and cur and rows and rows[-1]["sym"] == cur:
            rows[-1]["regs"] = int(m.group(1))
    names = subprocess.run(["c++filt"] + [r["sym"] for r in rows], capture_output=True, text=True).stdout.splitlines()
    for r, n in zip(rows, names):
        r["name"] = re.sub(r"\(.*$", "", n).replace("void ", "").replace("mafed::", "")
    print(" ".join(cmd[:1] + ["..."] + [c for c in cmd if c.startswith("-") and not c.startswith("-I")]))
    print(f"{len(rows)} kernels in distill_abi.cu; {sum(1 for r in rows if r['st'] or r['ld'])} with spill traffic\n")
    fam = collections.defaultdict(list)
    for r in rows:
        fam[r["name"].split("<")[0]].append(r)
    print("family: instantiations, registers min-max, spilling instantiations")
    for k, v in fam.items():
        regs = [r["regs"] for r in v]
        print(f"  {k}: {len(v)}, {min(regs)}-{max(regs)}, {sum(1 for r in v if r['st'] or r['ld'])}")
    print("\nTMA-ring kernels <dtype, loss (0 mse, 1 cosine, 2 L2 norm)[, pass (1 backward, 2 one-pass step)]>:")
    for r in rows:
        if "_tma" in r["name"]:
            print(f"  {r['name']}: {r['regs']} registers, stack {r['stack']} B, spill stores / loads {r['st']} / {r['ld']} B")
    print("\nother kernels with spill traffic:")
    for r in rows:
        if "_tma" not in r["name"] and (r["st"] or r["ld"]):
            print(f"  {r['name']}: {r['regs']} registers, stack {r['stack']} B, spill stores / loads {r['st']} / {r['ld']} B")


if __name__ == "__main__":
    main()
