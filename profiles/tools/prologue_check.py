#!/usr/bin/env python
"""Static check of a step kernel's prologue in the built object (no GPU needed): every global load of the prologue must be ISSUED
before the first instruction that consumes an in-flight load.  A consumer in between makes the warp wait out one HBM round trip and
only then issue the remaining loads -- two serialised round trips at the top of every warp, which is how 3-5 % were lost twice in
round 1 (a load predicate on `tick`; a per-env scalar spilled right after its load; profiles/README.md v11/v12).

usage: prologue_check.py [build/obj]      prints one line per kernel; exit code 1 if a kernel violates the rule."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
# (object, substring of the mangled name): the hot variants that ship
KERNELS = [("kernels_kg8.o", "step_kernelILi8ELi0E"), ("kernels_kg8.o", "step_kernelILi8ELi1E"),
           ("kernels_kg8.o", "step_kernelILi8ELi2E"), ("kernels_kg8.o", "step_kernelILi8ELi3E"),
           ("kernels_kg8.o", "step_kernelILi8ELi4E"), ("kernels_kg8.o", "step_kernelILi8ELi6E"),
           ("kernels_kg32.o", "step_kernelILi32ELi0E"), ("kernels_kg4.o", "fork_step_kernelILi4E")]
WINDOW = 200          # instructions from the first state load that count as prologue


def analyse(obj, sub):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    for block in re.split(r"\n\s*Function : ", out):
        name = block.split("\n", 1)[0]
        if sub not in name:
            continue
        ins = [re.sub(r"/\*[0-9a-f]+\*/", "", l).strip().split(";")[0].strip() for l in block.splitlines()
               if re.match(r"\s+/\*[0-9a-f]{4}\*/", l)]
        pending, first_use, loads = {}, None, []
        # the prologue = everything up to WINDOW instructions past the first 16-byte state load (round 2: the generator loop of the
        # step's regular draws runs BEFORE the loads, behind L2 prefetches of the same rows, so the loads no longer sit at the entry)
        first_ld = next((k for k, i in enumerate(ins) if "LDG.E" in i and ".128" in i), 0)
        for k, i in enumerate(ins[:first_ld + WINDOW]):
            body = re.sub(r"^@!?U?P\d+\s+", "", i)
            toks = body.split(None, 1)
            if len(toks) < 2:
                continue
            op, args = toks
            parts = [a.strip() for a in args.split(",")]
            dst, srcs = parts[0], ",".join(parts[1:])
            used = [r for r in pending if re.search(r"\b" + r + r"\b(?!\d)", srcs) or (op.startswith("ST") and re.search(r"\b" + r + r"\b", args))]
            if used and first_use is None:
                first_use = (k, i)
            # LDG.CONSTANT: table loads of the libm slow paths; LDG.STRONG: the hot blocks' own look-up of their tile (reset-first
            # scheduling, executed by the first few blocks of the grid only) -- neither is prologue traffic of the state
            if "LDG" in op and "CONSTANT" not in op and "STRONG" not in op:
                loads.append(k)
                m = re.match(r"R(\d+)", dst)
                if m:
                    for j in range(4 if ".128" in op else (2 if ".64" in op else 1)):
                        pending[f"R{int(m.group(1)) + j}"] = k
        late = [k for k in loads if first_use and k > first_use[0]]
        return dict(kernel=sub, loads=len(loads), first_use=first_use, late_loads=late)
    return None


def main():
    objdir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "build", "obj")
    bad = 0
    for obj, sub in KERNELS:
        r = analyse(os.path.join(objdir, obj), sub)
        if r is None:
            print(f"{sub}: not found in {obj}")
            continue
        print(f"{sub}: {r['loads']} prologue loads, first consumer at #{r['first_use'][0] if r['first_use'] else '-'}, "
              f"loads issued after it: {r['late_loads']}")
        bad += bool(r["late_loads"])
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
