#!/usr/bin/env python
"""Fused tcgen05 policy forward vs the torch module it replaces, one JSON line per case:
  * cfg2: the rollout batch of BASELINE configs[4] (65536 envs x 8 quads = 524288 observation rows, obs 54: S 18, W 6, V 6);
  * cfg3_obstacles: the same number of rows of the obstacle scenario's observation (BASELINE configs[2]: obs 40 = S 19, W 6, V 2, O 9);
  * cfg2_mlp: cfg2's rows with the MLP neighbour encoder (neighbor_encoder="mlp": the 36 neighbour columns as one vector -> 256 -> 256 -> 256).
Device time per forward (CUDA events on the launching stream, median of `reps` after warm-up), achieved dense TFLOP/s (and, when
MEASURED_PEAKS.json is present, the fraction of its sustained bf16 peak); the card's name and power limit go into every line.
python policy_bench.py [rows] [reps] [case ...]"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic  # noqa: E402

rows = int(sys.argv[1]) if len(sys.argv) > 1 else 524288
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
CASES = {   # name: (config, neighbour encoder)
    "cfg2": (lambda: QuadSimConfig(num_envs=8, num_agents=8), "mean_embed"),
    "cfg3_obstacles": (lambda: QuadSimConfig(num_envs=8, num_agents=8, quads_mode="mix", use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor",
                                             neighbor_visible_num=2), "mean_embed"),
    "cfg2_mlp": (lambda: QuadSimConfig(num_envs=8, num_agents=8), "mlp"),
}
cases = sys.argv[3:] or list(CASES)
dev = torch.device("cuda:0")
peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else None
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()


def timed(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


for case in cases:
    make, encoder = CASES[case]
    cfg = make()
    torch.manual_seed(0)
    pol = QuadActorCritic(cfg, neighbor_encoder=encoder).to(dev)
    fp = FusedPolicy(pol, dev)
    obs = torch.randn(rows, cfg.obs_dim, device=dev)
    S, W, V, O, A = fp.S, fp.W, fp.V, fp.O, fp.A
    ff_in = 256 * (1 + (V > 0) + (O > 0))
    # multiply-adds per row and tower: self encoder, V neighbour passes (MLP: one W V -> 256 -> 256 -> 256 pass), obstacle encoder, feed-forward;
    # heads A (actor) and 1 (critic)
    nbr = W * V * 256 + 2 * 256 * 256 if encoder == "mlp" else V * (W * 256 + 256 * 256)
    flop_row = 2 * 2 * (S * 256 + 256 * 256 + nbr + (O * 256 + 256 * 256 if O else 0) + ff_in * 512 + 512 * (A + 1) / 2)

    def eager_fp32():
        with torch.no_grad():
            return pol.action_net(pol.actor(obs)), pol.value(obs)

    def eager_bf16():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return pol.action_net(pol.actor(obs)), pol.value(obs)

    nbr_desc = (f", MLP neighbours {W * V}-256-256-256" if encoder == "mlp" else f", deep-sets {W}-256-256 x {V}") if V else ""
    policy = f"2 towers x (self {S}-256-256" + nbr_desc + (f", obstacles {O}-256-256" if O else "") + \
        f", ff {ff_in}-512, heads {A}/1)"
    out = {"case": case, "rows": rows, "obs_dim": cfg.obs_dim, "flop_per_row": flop_row, "policy": policy, "card": card}
    for name, fn in (("fused_tcgen05", lambda: fp.forward(obs)), ("torch_bf16_autocast", eager_bf16), ("torch_fp32", eager_fp32)):
        med, best = timed(fn)
        out[name] = {"ms_median": med, "ms_min": best, "rows_per_s": rows / med * 1e3, "tflops": flop_row * rows / med * 1e-9}
        if peaks:
            out[name]["frac_of_sustained_bf16_peak"] = flop_row * rows / med * 1e-9 / peaks["bf16_tflops_sustained"]
    m, v = fp.forward(obs)
    rm, rv = eager_fp32()
    out["max_abs_diff_vs_fp32"] = float(torch.maximum((m - rm).abs().max(), (v - rv).abs().max()))
    fp.close()
    print(json.dumps(out), flush=True)
