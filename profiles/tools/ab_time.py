#!/usr/bin/env python
"""A/B timing of library variants on ONE box: ab_time.py <case> <lib.so[:ENV=VAL...]> [<lib.so> ...]
Each variant runs in its own process (QS_LIB_PATH), `rounds` times in alternation; prints min / median ms per step.
case: cfg2 | cfg3 | cfg4 | fork | mix  (65536 envs; cfg4: 16384).  AB_STEADY=0 skips the steady-state pre-roll (round-1 behaviour)."""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CHILD = r'''
import sys, torch
sys.path.insert(0, %r)
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig
from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
case = sys.argv[1]
import os
n = int(os.environ.get("AB_ENVS", "16384" if case == "cfg4" else "65536"))
cfg = {"cfg2": lambda: QuadSimConfig(num_envs=n, num_agents=8),
       "mix": lambda: QuadSimConfig(num_envs=n, num_agents=8, quads_mode="mix"),
       "cfg3": lambda: QuadSimConfig(num_envs=n, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                                     obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2),
       "cfg4": lambda: QuadSimConfig(num_envs=n, num_agents=32),
       "fork": lambda: QuadSimConfig.fork_default(num_envs=n)}[case]()
sim = QuadSwarmSim(cfg, device="cuda:0")
sim.want_terminal_obs = False
g = torch.Generator(device="cuda").manual_seed(1)
pool = torch.rand((8, cfg.num_envs * cfg.num_agents, cfg.act_dim), device="cuda", generator=g) * 2 - 1
sim.reset()
if os.environ.get("AB_STEADY", "1") == "1":      # the bench's steady state: staggered episode clocks + more than one episode of pre-roll
    sim.set_state(tick=torch.randint(0, cfg.ep_len, (cfg.num_envs,), generator=g, device="cuda", dtype=torch.int32))
    pre = cfg.ep_len // (cfg.fork.substeps if cfg.env_mode == "fork" else 1) + 64
    for i in range(pre):
        sim.step(pool[i %% 8])
for i in range(50):
    sim.step(pool[i %% 8])
out = []
for rep in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(300):
        sim.step(pool[i %% 8])
    e1.record()
    torch.cuda.synchronize()
    out.append(e0.elapsed_time(e1) / 300)
print("RESULT", min(out))
''' % ROOT

case, libs = sys.argv[1], sys.argv[2:]
rounds = int(os.environ.get("AB_ROUNDS", "3"))
res = {l: [] for l in libs}
for r in range(rounds):
    for l in libs:
        path, *extra = l.split(":")            # "lib.so:QS_HOT=0:QS_BLOCK=64" sets environment knobs for that variant
        env = dict(os.environ, QS_LIB_PATH=os.path.abspath(path), **dict(kv.split("=", 1) for kv in extra))
        p = subprocess.run([sys.executable, "-c", CHILD, case], env=env, capture_output=True, text=True)
        line = [x for x in p.stdout.splitlines() if x.startswith("RESULT")]
        if not line:
            sys.stderr.write(p.stderr[-2000:])
            continue
        res[l].append(float(line[0].split()[1]))
for l in libs:
    v = res[l]
    print(f"{case:5s} {os.path.basename(l):28s} min {min(v) * 1e3:8.2f} us  median {statistics.median(v) * 1e3:8.2f} us  n={len(v)}")
print(json.dumps({os.path.basename(l): res[l] for l in libs}))
