#!/usr/bin/env python
"""Tuning aid: rebuild ONLY one lane-group translation unit (KG=8, or QS_VARIANT_KG) with extra -D defines and link it with the other objects of the
last full build -> build/variants/<name>.so (load it with QS_LIB_PATH).  usage: build_variant.py <name> [DEFINE ...]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from quad_swarm_rl_stable_baselines3_b200 import _capi  # noqa: E402

name, defines = sys.argv[1], sys.argv[2:]
KG = int(os.environ.get("QS_VARIANT_KG", "8"))          # which lane-group translation unit to rebuild
vdir = os.path.join(ROOT, "build", "variants")
os.makedirs(vdir, exist_ok=True)
obj = os.path.join(vdir, f"{name}_kg{KG}.o")
flags = [f for f in _capi.NVCC_FLAGS if f != "-shared"] + [f"-D{d}" for d in defines] + ["-Xptxas", "-v"]
r = subprocess.run(["nvcc"] + flags + [f"-DQS_KG={KG}", "-c", os.path.join(_capi.CSRC, "kernels_kg.cu"), "-o", obj], capture_output=True, text=True)
lines = r.stderr.split("\n")
for i, l in enumerate(lines):
    if "Function properties" in l and f"11step_kernelILi{KG}E" in l:
        print(l.split(f"11step_kernelILi{KG}E")[1][:6], lines[i + 1].strip(), "|", lines[i + 2].strip().replace("ptxas info    : ", ""))
if r.returncode:
    sys.stderr.write(r.stderr)
    sys.exit(1)
objdir = os.path.join(ROOT, "build", "obj")
objs = [os.path.join(objdir, "quadsim.o"), os.path.join(objdir, "policy.o")] + [os.path.join(objdir, f"kernels_kg{k}.o") for k in (1, 2, 4, 8, 16, 32) if k != KG] + [obj]
outdir = os.path.join(ROOT, "variants")      # travels to the GPU box (build/ is gpurun-ignored); *.so is git-ignored
os.makedirs(outdir, exist_ok=True)
subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", os.path.join(outdir, f"{name}.so")] + objs)
print("->", os.path.join(outdir, f"{name}.so"))
