#!/usr/bin/env python
"""Size and wall time of an exact save / resume at training scale: qs_snapshot / qs_restore (pinned and pageable host buffers) and
DevicePPO.save / load (checkpoint file written under --out).  Configurations: cfg2 and cfg3 at 65536 envs x 8 drones, the fork env at
65536 x 4.  Every time is a host clock around a call that returns after its stream has drained; median of --reps calls.  Each restore
is followed by a snapshot compared byte for byte with the restored blob.  Last, a resharded resume: qs_restore_shards of two cfg2
snapshots of --envs / 2 envs each into one handle of --envs (pinned).  The card's name and power limit go into every line.

    python profiles/tools/snapshot_time.py --out DIR [--envs 65536] [--reps 5] [--only-merge]
"""
import argparse
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from quad_swarm_rl_stable_baselines3_b200.config import QsConfigC, QuadSimConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", required=True, help="directory for the checkpoint files and snapshot_time.json")
ap.add_argument("--envs", type=int, default=65536)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--only-merge", action="store_true", help="time the resharded resume only")
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("snapshot_time.py measures on a CUDA device; none is visible")
os.makedirs(args.out, exist_ok=True)
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip()
CONFIGS = {
    "cfg2": lambda n: QuadSimConfig(num_envs=n, num_agents=8, seed=0),
    "cfg3": lambda n: QuadSimConfig(num_envs=n, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                                    obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, seed=0),
    "fork": lambda n: QuadSimConfig.fork_default(num_envs=n, seed=0),
}


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def steady_sim(cfg):
    """A handle in steady state: staggered clocks as bench.py sets them, a few steps, so that records and counters are filled."""
    sim = QuadSwarmSim(cfg, device=dev)
    sim.reset()
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    sim.set_state(tick=torch.randint(0, cfg.to_c().ep_len, (cfg.num_envs,), generator=g, device=dev, dtype=torch.int32))
    a = torch.zeros((sim.N * sim.K, sim.A), device=dev)
    for _ in range(8):
        sim.step(a)
    torch.cuda.synchronize(dev)
    return sim


rows = []
for name, make in ({} if args.only_merge else CONFIGS).items():
    cfg = make(args.envs)
    sim = steady_sim(cfg)
    lib, h, st = sim._lib, sim._h, sim._stream()
    n = int(lib.qs_snapshot_size(h))
    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pageable = np.empty(n, dtype=np.uint8)
    row = {"config": name, "envs": cfg.num_envs, "agents": cfg.num_agents, "card": card, "blob_bytes": n}
    for kind, ptr in (("pinned", C.c_void_p(pinned.data_ptr())), ("pageable", C.c_void_p(pageable.ctypes.data))):
        t, _ = timed(lambda: lib.qs_snapshot(h, ptr, n, st), args.reps)
        row[f"qs_snapshot_{kind}_s"] = t
        t, _ = timed(lambda: lib.qs_restore(h, ptr, n, st), args.reps)
        row[f"qs_restore_{kind}_s"] = t
    assert lib.qs_snapshot(h, C.c_void_p(pinned.data_ptr()), n, st) == 0
    again = torch.empty_like(pinned)
    assert lib.qs_restore(h, C.c_void_p(pinned.data_ptr()), n, st) == 0
    assert lib.qs_snapshot(h, C.c_void_p(again.data_ptr()), n, st) == 0
    assert torch.equal(again, pinned), "snapshot after restore differs from the restored blob"
    assert np.array_equal(pageable, pinned.numpy()), "pageable and pinned snapshots differ"
    row["gb_per_s_snapshot_pinned"] = n / row["qs_snapshot_pinned_s"] / 1e9
    row["gb_per_s_restore_pinned"] = n / row["qs_restore_pinned_s"] / 1e9
    del pinned, pageable, again
    sim.close()

    # DevicePPO checkpoint: hidden 256 policy, default optimiser, 8-step rollouts (the rollout buffers are not in the file)
    sim = QuadSwarmSim(cfg, device=dev)
    sim.want_terminal_obs = False
    ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=8, batch_size=65536, n_epochs=1, autocast_bf16=True))
    ppo.learn(1)
    path = os.path.join(args.out, f"ckpt_{name}.pt")
    row["ppo_save_s"], _ = timed(lambda: ppo.save(path), args.reps)
    row["ppo_file_bytes"] = os.path.getsize(path)
    ref = ppo.sim.snapshot()["blob"]
    del ppo
    sim.close()
    sim2 = QuadSwarmSim(cfg, device=dev)
    sim2.want_terminal_obs = False
    ppo2 = DevicePPO(sim2, cfg, PPOConfig(n_steps=8, batch_size=65536, n_epochs=1, autocast_bf16=True))
    row["ppo_load_s"], _ = timed(lambda: ppo2.load(path), args.reps)
    assert torch.equal(ppo2.sim.snapshot()["blob"], ref), "DevicePPO.load did not restore the saved simulator state"
    row["rollout_forward"] = "tcgen05 kernel" if ppo2.fused is not None else "torch"
    del ppo2
    sim2.close()
    torch.cuda.empty_cache()
    print(json.dumps(row), flush=True)
    rows.append(row)


# Resharded resume: the snapshots of two cfg2 shards of --envs / 2 envs merged into one handle of --envs (qs_restore_shards), pinned.
# Checked afterwards: every env-major section of the merged handle's snapshot is the two shards' sections back to back.
def sections(raw):
    """(offset, bytes) of every section of a blob, from its header's table (include/quadsim.h)."""
    base = 16 + C.sizeof(QsConfigC)
    count = int(np.frombuffer(raw[base + 4:base + 8].tobytes(), np.uint32)[0])
    sizes = np.frombuffer(raw[base + 8:base + 8 + 8 * count].tobytes(), np.uint64).astype(np.int64)
    offs = base + 8 + 8 * count + np.concatenate([[0], np.cumsum(sizes)[:-1]])
    return list(zip(offs.tolist(), sizes.tolist()))


cfg = CONFIGS["cfg2"](args.envs)
half = args.envs // 2
parts = [steady_sim(dataclasses.replace(cfg, num_envs=half, env_id_offset=r * half)) for r in range(2)]
blobs = []
for p in parts:
    n = int(p._lib.qs_snapshot_size(p._h))
    blobs.append(torch.empty(n, dtype=torch.uint8, pin_memory=True))
    assert p._lib.qs_snapshot(p._h, C.c_void_p(blobs[-1].data_ptr()), n, p._stream()) == 0
    p.close()
merged = QuadSwarmSim(cfg, device=dev)
lib, h, st = merged._lib, merged._h, merged._stream()
ptrs = (C.c_void_p * 2)(*[b.data_ptr() for b in blobs])
sizes = (C.c_size_t * 2)(*[b.numel() for b in blobs])
row = {"config": "cfg2_merge", "envs": cfg.num_envs, "agents": cfg.num_agents, "card": card,
       "source_blobs": [b.numel() for b in blobs]}
row["qs_restore_shards_2_to_1_pinned_s"], _ = timed(lambda: lib.qs_restore_shards(h, ptrs, sizes, 2, st), args.reps)
row["gb_per_s_restore_shards_pinned"] = sum(b.numel() for b in blobs) / row["qs_restore_shards_2_to_1_pinned_s"] / 1e9
n = int(lib.qs_snapshot_size(h))
out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
assert lib.qs_snapshot(h, C.c_void_p(out.data_ptr()), n, st) == 0
m, b0, b1 = out.numpy(), blobs[0].numpy(), blobs[1].numpy()
for (om, nm), (o0, n0), (o1, n1) in zip(sections(m), sections(b0), sections(b1)):
    if nm == 2 * n0 and n0 == n1 and nm > 0:                                   # env-major (the stats section is not)
        assert np.array_equal(m[om:om + n0], b0[o0:o0 + n0]) and np.array_equal(m[om + n0:om + nm], b1[o1:o1 + n1]), "merge differs"
merged.close()
print(json.dumps(row), flush=True)
rows.append(row)

with open(os.path.join(args.out, "snapshot_time.json"), "w") as f:
    json.dump(rows, f, indent=1)
