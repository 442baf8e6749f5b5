#!/usr/bin/env python
"""BASELINE.json configs[4] "with PPO update": rollout (policy inference + simulator) and update throughput of the device
PPO loop.  Single GPU: python ppo_throughput.py [envs] [n_steps] [config] [rollout]; N GPUs: torchrun --nproc-per-node N ppo_throughput.py ...
config: "cfg2" (default: 8 quads, deep-sets neighbours) or "cfg3" (the obstacle scenario of configs[2]: mix, obstacles, S 19, V 2);
rollout: "fused" (default: the tcgen05 forward where the architecture is covered) or "torch" (PPOConfig.fused_rollout = False)."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim  # noqa: E402

envs = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
n_steps = int(sys.argv[2]) if len(sys.argv) > 2 else 32
config = sys.argv[3] if len(sys.argv) > 3 else "cfg2"
rollout = sys.argv[4] if len(sys.argv) > 4 else "fused"
if config not in ("cfg2", "cfg3") or rollout not in ("fused", "torch"):
    raise SystemExit("config must be cfg2 or cfg3, rollout fused or torch")
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
extra = dict(quads_mode="mix", use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2) if config == "cfg3" else {}
cfg = QuadSimConfig(num_envs=envs, num_agents=8, seed=0, env_id_offset=rank * envs, **extra)
sim = QuadSwarmSim(cfg, device=dev)
sim.want_terminal_obs = False
ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=n_steps, batch_size=65536, n_epochs=1, autocast_bf16=True, fused_rollout=rollout == "fused"))
ppo.learn(1)                                                    # warm-up (cuBLAS heuristics, allocator)
hist = ppo.learn(2)
n = envs * 8
roll = sum(r["rollout_s"] for r in hist) / len(hist)
upd = sum(r["update_s"] for r in hist) / len(hist)
t = torch.tensor([roll, upd], device=dev, dtype=torch.float64)
if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
if rank == 0:
    roll, upd = float(t[0]), float(t[1])
    enc = ppo.policy.actor
    arch = f"self {enc.S}-256-256" + (f", deep-sets neighbours {enc.W}x{enc.V}-256-256" if enc.V else "") + (f", obstacles {enc.O}-256-256" if enc.O else "")
    print(json.dumps({"config": config, "rollout_forward": "tcgen05 kernel" if ppo.fused is not None else "torch bf16 autocast",
                      "n_gpus": world, "envs_per_gpu": envs, "agents": 8, "n_steps": n_steps,
                      "rollout_drone_steps_per_s": world * n * n_steps / roll, "update_samples_per_s": world * n * n_steps / upd,
                      "train_drone_steps_per_s": world * n * n_steps / (roll + upd), "rollout_s": roll, "update_s": upd,
                      "policy": f"2 towers x ({arch}, ff {enc.feed_forward[0].in_features}-512), bf16 autocast"}))
if world > 1:
    dist.destroy_process_group()
