#!/usr/bin/env python
"""bench.py -- drone-steps/sec of the batched quadrotor-swarm step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --steps K --dump-outputs DIR                   # + what the last timed step returned, as DIR/*.npy
    python bench.py --impl reference [--gpus N] ...                 # CPU arm: the oracle port on all host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU, weak scaling

Headline workload = the simulator leg of BASELINE.json configs[4] ("synthetic random-action throughput sweep: 65536 envs
x 8 quads"), with the environment of configs[1]: 8-quad swarm, static_same_goal, pos_vel observations of the 6 nearest
neighbours (obs 54), sensor + thrust noise on, episodes of 1500 control steps, synthetic i.i.d. U(-1,1) actions resident in
HBM, 65536 envs PER GPU (weak scaling: env shards are independent, no collective in the step).  A "step" is one control
step of every env = one launch of the fused step kernel.

Every workload is measured IN STEADY STATE: the episode clocks are staggered uniformly over [0, ep_len) and the batch is
pre-rolled for more than one episode before anything is timed, so every timed step contains ~N/ep_len auto-resets (with
scenario resampling) and the real mix of floor contact / collisions of a random-action rollout; the number of episodes that
ended inside the timed window is reported (`resets_in_window`).  The timed region is exactly K = --steps steps after W =
--warmup untimed ones, split into up to 10 blocks of back-to-back steps, each bracketed by its own CUDA-event pair on the
launching stream; the reported time per step is that of the MEDIAN block (max over ranks).  The number of steps a workload
runs is fixed by the arguments, not by the clock, so with the same arguments every run computes the same outputs
(--dump-outputs).  NCCL is initialised and warmed up before the warm-up steps.

Per-step working set at 65536 envs (260 MB) exceeds the 126 MB L2 -> back-to-back steps, no flush.  The small BASELINE
points (configs[1] 4096x8, configs[2] 4096x8 obstacles, configs[3] 1024x32) are measured with per-step events and an L2
flush between steps.  Further keys: cfg3_obstacles / cfg4_k32 / mix / fork at the large batch, `cfg5_strong` (65536 envs
TOTAL split over the ranks) and `cfg5_ppo` (the same with policy inference + PPO update in the loop).
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 65536
ENVS_CFG2 = 4096
ENVS_CFG4 = 1024
AGENTS = 8
TIMED_BLOCKS = 10           # the --steps timed steps are split into this many event-bracketed blocks (median reported)
DUMP_ROWS = 131072          # --dump-outputs: at most this many drones (seeded sample), 29 MB at obs 54
# Algorithmic HBM bytes per drone-step (SURVEY.md 8d, restated in DESIGN.md "Roofline"):
# state 120 B read + 120 B written, goal 12 R, tick/flags 4 R+W, action 16 R, obs 4*D W, reward 4 + done 1 W
ALGO_BYTES = {"cfg2": 497.0, "cfg3": 453.0, "cfg4": 501.0, "mix": 497.0 + 16.0 + 12.0}
WORKLOAD = ("cfg5 simulator leg: 65536 envs x 8 quads per GPU, env = cfg2 (static_same_goal, pos_vel x6 neighbours, "
            "obs 54, noise on, ep 1500 steps), steady state (staggered episode clocks, auto-resets inside the window)")


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic_per_launch():
    """dram bytes per launch of the step kernel from the committed `ncu --set full` capture, if any."""
    p = os.path.join(ROOT, "profiles", "step_kernel_cfg2_traffic.json")
    try:
        with open(p) as f:
            return float(json.load(f)["dram_bytes_per_launch"])
    except Exception:
        return None


def dump_outputs(out_dir, tensors):
    """(obs, rew, done) of one step -> out_dir/{obs,rew,done}.npy, float32.  With more than DUMP_ROWS drones all three keep the
    same rows, drawn once from a fixed seed, so two builds run with the same arguments can be compared array for array."""
    import numpy as np
    obs, rew, done = (t.float().cpu().numpy() for t in tensors)
    if obs.shape[0] > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(obs.shape[0], DUMP_ROWS, replace=False))
        obs, rew, done = obs[rows], rew[rows], done[rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("obs", obs), ("rew", rew), ("done", done)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_port_throughput(envs, agents, budget_s, threads):
    """The CPU oracle (float64 C port of the reference's step, oracle/quadsim_oracle.c) on `threads` OpenMP threads inside one
    native call (static env slices, one barrier per step), same workload config, same steady state (staggered episode clocks,
    drones pre-rolled until the random-action rollout has reached its floor-contact mix).
    Returns (drone-steps/s, description)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import OracleBatch
    from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig
    cfg = QuadSimConfig(num_envs=envs, num_agents=agents, seed=0)
    b = OracleBatch(cfg, threads=threads)
    b.reset()
    rs = np.random.RandomState(0)
    b.set_ticks(rs.randint(0, cfg.ep_len, envs))
    acts = rs.uniform(-1, 1, (8, envs * agents, 4))
    t0 = time.perf_counter()
    b.run(acts, 10)
    per = (time.perf_counter() - t0) / 10
    pre = int(max(10, min(200, 0.25 * budget_s / max(per, 1e-6))))        # pre-roll: drones land within ~100 steps
    b.run(acts, pre)
    n = int(max(5, min(20000, budget_s / max(per, 1e-6))))
    t0 = time.perf_counter()
    resets = b.run(acts, n)
    dt = time.perf_counter() - t0
    return envs * agents * n / dt, (f"{envs} envs x {agents} drones x {n} control steps after {pre + 10} pre-roll steps, staggered episode "
                                    f"clocks ({resets} resets in the sample), {b.threads} OpenMP threads, {dt:.1f} s")


def run_reference(args, rank, world):
    """--impl reference: the reference's algorithm on the host cores (the reference is pure Python and cannot
    travel to the GPU box, so this is its C port, the oracle).  Rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    envs = ENVS_CFG2
    budget = min(20.0, max(4.0, 0.02 * (args.steps + args.warmup)))
    v, sample = cpu_port_throughput(envs, AGENTS, budget, threads)
    line = {
        "impl": "reference", "metric": "drone-steps/sec", "value": v, "unit": "drone-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * ENVS_PER_GPU * AGENTS / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": ENVS_PER_GPU, "agents": AGENTS, "obs_dim": 54,
                   "note": "CPU arm: C port of the reference step (oracle), all host threads (OpenMP), bounded sample of 4096 envs; "
                           "ms_per_step is the time this arm would need for one 65536-env step. The reference's own numba path is "
                           "~100x slower per core than this port (BASELINE.md, measured in the build container)"},
        "cpu_baseline": {"value": v, "unit": "drone-steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "drone-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps of every workload")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write obs / rew / done of the last timed step of the headline workload (rank 0) as DIR/<name>.npy, float32; "
                         f"more than {DUMP_ROWS} drones -> the same seeded sample of rows in all three")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU, help="override for size sweeps (not the bench line)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-small", action="store_true", help="headline + e2e only (skip the secondary workloads)")
    ap.add_argument("--skip-ppo", action="store_true")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "mix"],
                    help="another workload as the timed one (profiling aid; the bench line is cfg2)")
    ap.add_argument("--no-steady", action="store_true", help="profiling aid: skip the staggering + pre-roll (round-1 behaviour)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        w = torch.ones(1, device=dev)
        for _ in range(3):                      # communicator set-up happens here, not between the warm-up and the timed window
            dist.all_reduce(w)
            dist.barrier()
    stream = torch.cuda.current_stream(dev)
    POOL = 8

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def config(workload, n_envs, offset):
        if workload == "cfg3":
            # BASELINE.json configs[2]: 8x8 m obstacle area, density 0.2 -> 12 obstacles of 0.6 m, SDF obs, downwash, 2 neighbours, obs 40
            return QuadSimConfig(num_envs=n_envs, num_agents=AGENTS, quads_mode="mix", use_obstacles=True, use_downwash=True,
                                 obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, seed=0, env_id_offset=offset)
        if workload == "mix":        # the upstream training recipe --quads_mode=mix (swarm_rl/runs/quad_multi_mix_baseline.py:13-16)
            return QuadSimConfig(num_envs=n_envs, num_agents=AGENTS, quads_mode="mix", seed=0, env_id_offset=offset)
        if workload == "cfg4":       # BASELINE.json configs[3]: 32-quad scale scenario
            return QuadSimConfig(num_envs=n_envs, num_agents=32, seed=0, env_id_offset=offset)
        if workload == "fork":       # configs[0] family: the fork env sb_train.py trains on
            return QuadSimConfig.fork_default(num_envs=n_envs, seed=0, env_id_offset=offset)
        return QuadSimConfig(num_envs=n_envs, num_agents=AGENTS, seed=0, env_id_offset=offset)

    def make(workload, n_envs):
        """Simulator + action pool, brought to steady state: staggered episode clocks, then a pre-roll of more than one episode."""
        cfg = config(workload, n_envs, rank * n_envs)
        sim = QuadSwarmSim(cfg, device=dev)
        sim.want_terminal_obs = False
        gen = torch.Generator(device=dev)
        gen.manual_seed(1234 + rank)
        pool = (torch.rand((POOL, n_envs * cfg.num_agents, cfg.act_dim), device=dev, generator=gen) * 2.0 - 1.0).contiguous()
        sim.reset()
        pre = 0
        if not args.no_steady:
            calls_per_episode = cfg.ep_len // (cfg.fork.substeps if cfg.env_mode == "fork" else 1)
            ticks = torch.randint(0, cfg.ep_len, (n_envs,), generator=gen, device=dev, dtype=torch.int32)
            sim.set_state(tick=ticks)
            pre = calls_per_episode + 64
            for i in range(pre):
                sim.step(pool[i % POOL])
            torch.cuda.synchronize(dev)
            sim.episode_stats(reset=True)
        return sim, pool, cfg, pre

    def timed_steps(sim, pool, flush=None):
        """--warmup untimed steps, then exactly --steps timed ones in up to TIMED_BLOCKS blocks of back-to-back steps, one
        CUDA-event pair per block on the launching stream (an event between every two steps would cost ~2 us each).
        flush: a buffer larger than L2 rewritten before every step (then one step per block, the flush outside the events).
        ms_per_step is the median over blocks of block time / steps.  Returns a dict of timings and the (obs, rew, done)
        tensors of the last timed step (they alias the simulator's buffers)."""
        for i in range(args.warmup):
            sim.step(pool[i % POOL])
        nblk = args.steps if flush is not None else min(args.steps, TIMED_BLOCKS)
        bounds = [args.steps * b // nblk for b in range(nblk + 1)]
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nblk)]
        ep0 = sim.episode_stats()["episodes"]
        l0 = sim.launch_count
        barrier()
        for i in range(3):                        # the barrier idles the GPU: a few untimed steps before the first event
            sim.step(pool[i % POOL])
        t_wall = time.perf_counter()
        for b in range(nblk):
            if flush is not None:
                flush.fill_(float(b))
            ev[b][0].record(stream)
            for j in range(bounds[b], bounds[b + 1]):
                last = sim.step(pool[j % POOL])
            ev[b][1].record(stream)
        barrier()
        wall = time.perf_counter() - t_wall
        blk_ms = [a.elapsed_time(e) for a, e in ev]
        per = sorted(t / (bounds[b + 1] - bounds[b]) for b, t in enumerate(blk_ms))
        return {"ms_per_step": per[len(per) // 2], "step_ms_min": per[0], "step_ms_max": per[-1], "steps": args.steps,
                "blocks": nblk, "timed_s": sum(blk_ms) * 1e-3, "wall_s": wall,
                "resets_in_window": int(sim.episode_stats()["episodes"] - ep0), "launches": int(sim.launch_count - l0 - 3)}, last

    def reduce_max(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def reduce_sum(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t)

    peak, peak_src = measured_hbm_peak()

    def point(workload, n_envs, flush=None, algo=None, label=None):
        """One secondary workload -> its JSON sub-object (max over ranks)."""
        sim, pool, cfg, pre = make(workload, n_envs)
        r, _ = timed_steps(sim, pool, flush=flush)
        ms = reduce_max(r["ms_per_step"])
        resets = reduce_sum(r["resets_in_window"])
        nd_ = n_envs * cfg.num_agents
        sub = cfg.fork.substeps if cfg.env_mode == "fork" else 1
        out = {"workload": label, "envs_per_gpu": n_envs, "agents": cfg.num_agents, "obs_dim": sim.D, "ms_per_step": ms,
               "value": world * nd_ * sub / (ms * 1e-3), "unit": "drone-steps/s", "steps": r["steps"], "blocks": r["blocks"],
               "timed_s": r["timed_s"], "pre_roll_steps": pre, "resets_in_window": int(resets),
               "l2": "flushed before every timed step (256 MiB write), per-step CUDA events" if flush is not None else "working set > L2, back-to-back steps"}
        if algo is not None:
            out["algorithmic_bytes_per_drone_step"] = algo
            out["roofline_frac"] = algo * nd_ / (ms * 1e-3) / 1e9 / peak
        sim.close()
        del sim, pool
        return out

    # ---- headline: device-resident path -> value ---------------------------------------------------------------------
    n_envs = args.envs_per_gpu
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()            # nvidia-smi takes ~1 s to deliver its first sample: start it before the pre-roll
    sim, act_pool, cfg, pre_roll = make(args.workload, n_envs)
    nd = n_envs * cfg.num_agents
    head, last = timed_steps(sim, act_pool)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)     # before anything else steps this simulator
    del last
    clocks = None
    if rank == 0:
        if head["wall_s"] < 3.0:      # keep the GPU under the same load a little longer so that nvidia-smi samples it
            t_end = time.perf_counter() + 3.0 - head["wall_s"]
            j = 0
            while time.perf_counter() < t_end:
                sim.step(act_pool[j % POOL]); j += 1
            torch.cuda.synchronize(dev)
        clocks = sampler.stop()

    # ---- host-buffer path through the public API: e2e (pinned numpy in, pinned numpy out, every step) ------------
    host_acts = []
    for i in range(POOL):
        t = torch.empty((nd, cfg.act_dim), dtype=torch.float32, pin_memory=True)
        t.copy_(act_pool[i])
        host_acts.append(t.numpy())
    out_t = (torch.empty((nd, sim.D), dtype=torch.float32, pin_memory=True),
             torch.empty((nd,), dtype=torch.float32, pin_memory=True), torch.empty((nd,), dtype=torch.uint8, pin_memory=True))
    out = tuple(t.numpy() for t in out_t)
    e2e_steps = args.steps
    for i in range(3):
        sim.step_host(host_acts[i % POOL], out)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    for i in range(e2e_steps):
        sim.step_host(host_acts[i % POOL], out)
    e1.record(stream)
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))     # the call is synchronous: host clock == device clock
    e2e_ms = reduce_max(e2e_ms)
    d_head = sim.D
    sim.close()
    del sim, act_pool, out_t, out, host_acts

    ms_per_step = reduce_max(head["ms_per_step"])
    head_resets = reduce_sum(head["resets_in_window"])

    extra = {}
    if not args.skip_small:
        flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
        extra["cfg2_4096"] = point("cfg2", ENVS_CFG2, flush=flush_buf, algo=ALGO_BYTES["cfg2"],
                                   label="configs[1]: 4096 envs x 8 quads per GPU, static_same_goal, obs 54")
        extra["cfg3_4096"] = point("cfg3", ENVS_CFG2, flush=flush_buf, algo=ALGO_BYTES["cfg3"],
                                   label="configs[2]: 4096 envs x 8 quads per GPU, 12 obstacles, SDF obs, downwash, obs 40")
        extra["cfg4_k32_1024"] = point("cfg4", ENVS_CFG4, flush=flush_buf, algo=ALGO_BYTES["cfg4"],
                                       label="configs[3]: 1024 envs x 32 quads per GPU, obs 54")
        del flush_buf
        extra["cfg3_obstacles"] = point("cfg3", n_envs, algo=ALGO_BYTES["cfg3"],
                                        label="configs[2] at the sweep size: 65536 envs x 8 quads per GPU, 12 obstacles, SDF obs, downwash, obs 40")
        extra["cfg4_k32_16384"] = point("cfg4", n_envs // 4, algo=ALGO_BYTES["cfg4"],
                                        label="configs[3] at the sweep size: 16384 envs x 32 quads per GPU (the same 524288 drones), obs 54")
        extra["mix_scenarios"] = point("mix", n_envs, algo=ALGO_BYTES["mix"],
                                       label="upstream training recipe quads_mode=mix: 65536 envs x 8 quads per GPU, one of 9 formation scenarios per "
                                             "episode (goals moving every step in 3 of them), obs 54; +16 B goal written, +12 B scenario row read per drone-step")
        extra["fork_k4"] = point("fork", n_envs,
                                 label="fork env of sb_train.py: 65536 envs x 4 chasers per GPU, dynamic_repulsive, one call = 8 control steps "
                                       "(value counts control steps; ms_per_step is per call)")
        # configs[4] as written: 65536 envs TOTAL, sharded over the ranks (strong scaling)
        if world > 1:
            s = point("cfg2", ENVS_PER_GPU // world, algo=ALGO_BYTES["cfg2"],
                      label=f"configs[4] strong scaling: 65536 envs x 8 quads in total = {ENVS_PER_GPU // world} envs per GPU")
        else:
            s = {"workload": "configs[4] strong scaling: 65536 envs x 8 quads in total (1 GPU: the headline run)", "envs_per_gpu": n_envs,
                 "ms_per_step": ms_per_step, "value": nd / (ms_per_step * 1e-3), "unit": "drone-steps/s",
                 "roofline_frac": ALGO_BYTES["cfg2"] * nd / (ms_per_step * 1e-3) / 1e9 / peak}
        s["scaling"] = "strong"
        extra["cfg5_strong"] = s

    ppo_line = None
    if not args.skip_ppo and not args.skip_small:
        try:
            from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
            n_ppo = ENVS_PER_GPU // world
            pcfg = config("cfg2", n_ppo, rank * n_ppo)
            psim = QuadSwarmSim(pcfg, device=dev)
            psim.want_terminal_obs = False
            algo = DevicePPO(psim, pcfg, PPOConfig(n_steps=8, batch_size=65536, n_epochs=1, autocast_bf16=True), seed=0)
            algo.collect(); algo.update()                          # warm-up iteration (allocator, cuBLAS heuristics, NCCL buckets)
            barrier()
            t0 = time.perf_counter()
            r = algo.collect()
            barrier()
            t1 = time.perf_counter()
            u = algo.update()
            barrier()
            t2 = time.perf_counter()
            roll_s, upd_s = reduce_max(t1 - t0), reduce_max(t2 - t1)
            samples = world * n_ppo * AGENTS * algo.p.n_steps
            ppo_line = {"workload": "configs[4] with PPO update: 65536 envs x 8 quads in total, two-tower policy (self 18-256-256, deep-sets neighbours, "
                                    "512-512), rollout of 8 steps + 1 epoch of 65536-row minibatches",
                        "rollout_value": samples / roll_s, "loop_value": samples / (roll_s + upd_s), "unit": "drone-steps/s",
                        "rollout_s": roll_s, "update_s": upd_s,
                        "policy_path": ("rollout forward + GAE: hand-written sm_100a kernels (qp::policy_forward_kernel, tcgen05 / TMEM; qp::gae_kernel); "
                                        "update: torch autograd + cuBLAS under bf16 autocast with the elementwise work on qp::bias_tanh* kernels") if algo.fused is not None
                                       else "torch (bf16 autocast)",
                        "simulator_launches_per_env_step": 1}
            if algo.fused is not None:
                # the rollout's dense forward alone, device-timed: fused tcgen05 kernel vs the torch module it replaces (same weights, same rows)
                def ev_ms(fn, reps):
                    for _ in range(2):
                        fn()
                    torch.cuda.synchronize()
                    ts = []
                    for _ in range(reps):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                        ts.append(e0.elapsed_time(e1))
                    return sorted(ts)[len(ts) // 2]

                def eager():
                    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                        return algo.policy.action_net(algo.policy.actor(algo.obs)), algo.policy.value(algo.obs)

                fp = algo.fused
                rows = algo.obs.shape[0]
                flop_row = 4.0 * (fp.S * 256 + 65536 + fp.V * (fp.W * 256 + 65536) + 262144 + 256 * (fp.A + 1))
                ms_f, ms_t = ev_ms(lambda: fp.forward(algo.obs), 10), ev_ms(eager, 3)
                try:
                    tf_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"]
                except Exception:
                    tf_peak = None
                ppo_line["policy_forward"] = {
                    "kernel": "qp::policy_forward_kernel", "rows": rows, "flop_per_row": flop_row, "ms_fused": ms_f, "ms_torch_bf16_autocast": ms_t,
                    "tflops": flop_row * rows / ms_f * 1e-9, "bound": "tensor", "peak_tflops": tf_peak,
                    "frac": (flop_row * rows / ms_f * 1e-9 / tf_peak) if tf_peak else None,
                    "peak_source": "measured (MEASURED_PEAKS.json, sustained cuBLAS bf16)", "speedup_vs_torch": ms_t / ms_f}
            psim.close()
            del algo, psim
        except Exception as ex:      # the PPO loop is a secondary key: never lose the bench line over it
            ppo_line = {"error": repr(ex)}

    if rank == 0:
        value = world * nd / (ms_per_step * 1e-3)
        e2e_value = world * nd / (e2e_ms / e2e_steps * 1e-3)
        algo_b = ALGO_BYTES.get(args.workload, 497.0)
        bytes_per_launch = algo_b * nd
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        cpu = None
        if not args.skip_cpu:
            threads = os.cpu_count() or 1
            v, sample = cpu_port_throughput(ENVS_CFG2, AGENTS, 12.0, threads)
            cpu = {"value": v, "unit": "drone-steps/s", "cores": threads, "kind": "port", "sample": sample}
            try:      # the Python reference cannot travel to this box: its per-core rate relative to the port was measured where it exists
                rv = json.load(open(os.path.join(ROOT, "profiles", "r2_reference_vs_port.json")))
                k = next(k for k in rv if k.startswith("cfg2"))
                cpu["python_reference"] = {"port_over_reference_per_core": rv[k]["port_over_reference"],
                                           "reference_drone_steps_per_s_per_core": rv[k]["reference_drone_steps_per_s_per_core"],
                                           "source": "profiles/r2_reference_vs_port.json (build container, numba JIT on, 1 core; profiles/tools/ref_vs_port.py)"}
            except Exception:
                pass
        line = {
            "metric": "drone-steps/sec", "value": value, "unit": "drone-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": n_envs, "agents": cfg.num_agents, "obs_dim": d_head,
                       "act_dim": 4, "l2": "inputs larger than L2 (260 MB touched per step vs 126 MB L2), no flush",
                       "timing": f"{args.steps} back-to-back steps in {head['blocks']} blocks, one CUDA-event pair per block on the "
                                 f"launching stream ({head['timed_s']:.2f} s of device time), median block, max over ranks; "
                                 f"barrier + synchronize on both sides",
                       "steady_state": f"episode clocks staggered uniformly, {pre_roll} pre-roll steps (> 1 episode) before the warm-up",
                       "parallelism": f"env-sharded x{world}, no collective in the step"},
            "timed_window": {"steps": head["steps"], "blocks": head["blocks"], "step_ms_median": head["ms_per_step"],
                             "step_ms_min": head["step_ms_min"], "step_ms_max": head["step_ms_max"], "timed_s": head["timed_s"],
                             "resets_in_window": int(head_resets), "pre_roll_steps": pre_roll},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "drone-steps/s", "h2d_bytes_per_step": nd * 4 * 4,
                    "d2h_bytes_per_step": nd * (d_head * 4 + 4 + 1), "steps": e2e_steps,
                    "api": "QuadSwarmSim.step_host -> qs_step_host: pinned numpy actions H2D, step kernel, "
                           "obs/rew/done D2H into pinned numpy, stream sync, every step"},
            "gpu_launches": int(head["launches"]),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": committed_traffic_per_launch(), "algorithmic_bytes_per_launch": bytes_per_launch,
                         "kernel": "qs::step_kernel<8>", "peak_source": peak_src},
            "cpu_baseline": cpu,
        }
        line.update(extra)
        if ppo_line is not None:
            line["cfg5_ppo"] = ppo_line
        if args.workload != "cfg2":
            line["config"]["workload"] = "PROFILING AID, not the bench line: " + args.workload
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
