"""Resharded resume: the envs of N old shards restored into M new handles (qs_restore_shards, include/quadsim.h;
QuadSwarmSim.restore_shards; DevicePPO.load_shards).  Shards are emulated on one device by handles with different env_id_offset.

  1. merge (37 + 91 -> 128), split (128 -> 50 + 78) and uneven (3 x 40 -> 64 + 56) reshards of the cfg2, cfg3, formation-mix, fork and
     K = 6 families continue bitwise: obs, reward, done, terminal observation, reset_success, every get_state field and the episode
     records of the new handles concatenate to the old handles', stepped with the same seeded actions, and the episode-stat totals
     over the new handles equal those over the old ones (integers exact, double sums to 1e-12).  Clocks are staggered and episodes
     short, so episodes end before the snapshot and at least twice per env after it;
  2. restore_shards of one blob into a handle of the blob's own range is qs_restore, byte for byte;
  3. a gap, an overlap, shards of different steps, another seed or ep_len, qs_set_param values that differ between the sources, a fork
     blob into an upstream handle, a truncated or damaged blob, count = 0 and NULL arrays are rejected with the reason named, and a
     snapshot whose observation does not fit its blob is refused by the torch layer, the handle untouched in every case;
  4. DevicePPO: a world-1 run resumed as two shards, and two shards resumed as one run, continue the simulator bitwise with the saved
     policy and Adam state; rank files whose policies differ are refused.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from quad_swarm_rl_stable_baselines3_b200.config import QsConfigC, QsStatsC, QuadSimConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim  # noqa: E402

QS_ERR_BAD_CONFIG, QS_ERR_SHAPE, QS_ERR_NULL = -1, -3, -4
OBST = dict(use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor")

# name: (config of the whole run, changed parameter).  0.4 s upstream episodes are 40 control steps; 1 s fork episodes 100 control
# steps, 13 calls of 8.
FAMILIES = {
    "cfg2_k8": (lambda: QuadSimConfig(num_agents=8, ep_time=0.4, seed=21), ("rew", dict(pos=1.7, quadcol_bin=3.0))),
    "cfg3_obst_downwash": (lambda: QuadSimConfig(num_agents=8, quads_mode="mix", use_downwash=True, neighbor_visible_num=2, ep_time=0.4,
                                                 seed=22, **OBST), ("rew", dict(quadcol_bin_obst=2.5))),
    "formation_mix_k8": (lambda: QuadSimConfig(num_agents=8, quads_mode="mix", ep_time=0.4, seed=23), ("rew", dict(crash=0.5))),
    "fork_k4": (lambda: QuadSimConfig.fork_default(ep_time=1.0, capture_radius=2.4, seed=24), ("capture", 1.9)),
    "k6": (lambda: QuadSimConfig(num_agents=6, neighbor_visible_num=5, ep_time=0.4, seed=25), ("rew", dict(effort=0.2))),
}
# name: (old shard sizes, new shard sizes), both from global env 0
SHAPES = {"merge_37_91_to_128": ((37, 91), (128,)), "split_128_to_50_78": ((128,), (50, 78)), "uneven_3x40_to_64_56": ((40, 40, 40), (64, 56))}
PRE = 20


def bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def assert_bitwise(a, b, what):
    assert a.shape == b.shape and torch.equal(bits(a), bits(b)), what


def shard(cfg, n, off):
    return dataclasses.replace(cfg, num_envs=n, env_id_offset=off)


def make_shards(cfg, sizes):
    offs = np.concatenate([[0], np.cumsum(sizes)[:-1]]).tolist()
    return [QuadSwarmSim(shard(cfg, n, o), device="cuda:0") for n, o in zip(sizes, offs)]


def window(cfg):
    """Steps after the snapshot in which every env ends at least two episodes."""
    c = cfg.to_c()
    per_call = c.fork.substeps if cfg.env_mode == "fork" else 1
    return 2 * -(-c.ep_len // per_call) + 4


def extent(sims):
    """Global envs [0, extent) cover every handle of `sims`."""
    return max(s.cfg.env_id_offset + s.N for s in sims)


def global_actions(sims, n, seed):
    """Per step one action row per drone of global envs [0, extent): a handle takes the rows of its env range."""
    s = sims[0]
    total = extent(sims)
    g = torch.Generator(device=s.device)
    g.manual_seed(seed)
    return [torch.rand((total * s.K, s.A), device=s.device, generator=g) * 2.0 - 1.0 for _ in range(n)]


def rows(sim, a):
    return a[sim.cfg.env_id_offset * sim.K:(sim.cfg.env_id_offset + sim.N) * sim.K].contiguous()


def prepare(sims, change):
    """reset, staggered clocks, a changed reward coefficient / capture radius, PRE steps: the state of a run when it is saved."""
    L = sims[0].cfg.to_c().ep_len
    ticks = np.random.RandomState(sims[0].cfg.seed).randint(0, L, extent(sims)).astype(np.int32)
    for s in sims:
        s.reset()
        s.set_state(tick=ticks[s.cfg.env_id_offset:s.cfg.env_id_offset + s.N])
        kind, val = change
        if kind == "rew":
            s.set_rew_coeff(**val)
        else:
            s.set_capture_radius(val)
    for a in global_actions(sims, PRE, 100):
        for s in sims:
            s.step(rows(s, a))


def run(sims, n):
    """n steps with seeded actions over the whole env range; per step the concatenated (obs, rew, done, terminal_obs, reset_success).
    The outputs that only finished envs write are filled with a canary first, so that the whole buffer compares."""
    out = []
    for a in global_actions(sims, n, 200):
        step = []
        for s in sims:
            s.terminal_obs.fill_(float("nan"))
            s.reset_success.fill_(0x5A)
            o, r, d = s.step(rows(s, a))
            step.append((o.clone(), r.clone(), d.clone(), s.terminal_obs.clone(), s.reset_success.clone()))
        out.append(tuple(torch.cat(parts) for parts in zip(*step)))
    return out


def assert_runs_equal(ref, got, what):
    for t, (x, y) in enumerate(zip(ref, got)):
        for name, a, b in zip(("obs", "rew", "done", "terminal_obs", "reset_success"), x, y):
            assert_bitwise(a, b, f"{what}: {name} of step {t}")


def concat_state(sims):
    parts = [s.get_state() for s in sims]
    return {k: torch.cat([p[k] for p in parts]) for k in parts[0]}


def concat_records(sims):
    recs = [s.episode_records() for s in sims]
    return torch.cat([r["env"] for r in recs]), torch.cat([r["agent"] for r in recs])


def total_stats(sims):
    tot = None
    for s in sims:
        st = s.episode_stats()
        tot = st if tot is None else {k: tot[k] + st[k] for k in tot}
    return tot


def assert_stats_equal(x, y, what):
    for k in x:
        if isinstance(x[k], float):
            assert abs(x[k] - y[k]) <= 1e-12 * max(1.0, abs(x[k])), (what, k, x[k], y[k])
        else:
            assert x[k] == y[k], (what, k, x[k], y[k])


def assert_same_sims(old, new, what):
    so, sn = concat_state(old), concat_state(new)
    assert set(so) == set(sn)
    for k in so:
        assert_bitwise(so[k], sn[k], f"{what}: get_state {k}")
    for name, a, b in zip(("env records", "agent records"), concat_records(old), concat_records(new)):
        assert_bitwise(a, b, f"{what}: {name}")
    assert_stats_equal(total_stats(old), total_stats(new), f"{what}: episode_stats totals")


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("family", list(FAMILIES))
def test_reshard_continues_bitwise(family, shape):
    make, change = FAMILIES[family]
    cfg = make()
    old_sizes, new_sizes = SHAPES[shape]
    old = make_shards(cfg, old_sizes)
    prepare(old, change)
    assert sum(int((s.episode_records()["env"][:, 0] > 0).sum()) for s in old) > 0, "no episode ended before the snapshot"
    snaps = [s.snapshot() for s in old]

    new = make_shards(cfg, new_sizes)
    for s in new:
        s.restore_shards(snaps)                                # every new shard gets the full list of old ones
        assert s.rew_coeff_overrides == old[0].rew_coeff_overrides
    assert_bitwise(torch.cat([s.obs for s in new]), torch.cat([s.obs for s in old]), "restored obs")
    assert_same_sims(old, new, "right after the restore")

    n = window(cfg)
    ref = run(old, n)
    ends = torch.stack([x[2] for x in ref]).view(n, -1, cfg.num_agents)[:, :, 0].sum(0)
    assert int(ends.min()) >= 2, f"an env ended {int(ends.min())} episodes in the window"
    assert_runs_equal(ref, run(new, n), f"{family} {shape}")
    assert_same_sims(old, new, "after the window")
    print(f"[{family} {shape}] {n} steps, episode ends per env {int(ends.min())}..{int(ends.max())}")


@pytest.mark.parametrize("family", ["cfg2_k8", "formation_mix_k8", "fork_k4"])
def test_one_blob_into_its_own_range_is_restore(family):
    make, change = FAMILIES[family]
    cfg = make()
    src = make_shards(cfg, (91, 37))[1]                        # envs [91, 128)
    prepare([src], change)
    snap = src.snapshot()
    a, b = (QuadSwarmSim(shard(cfg, 37, 91), device="cuda:0") for _ in range(2))
    a.restore(snap)
    b.restore_shards([snap])
    assert_bitwise(b.obs, a.obs, "restored obs")
    assert a.rew_coeff_overrides == b.rew_coeff_overrides
    assert torch.equal(a.snapshot()["blob"], b.snapshot()["blob"]), "restore_shards([blob]) differs from restore(blob)"
    assert torch.equal(b.snapshot()["blob"], snap["blob"])
    assert_runs_equal(run([a], 12), run([b], 12), "after restore vs restore_shards")


# ---------------------------------------------------------------------------------------------------------------------------------
# rejections
# ---------------------------------------------------------------------------------------------------------------------------------
BASE = QuadSimConfig(num_agents=8, ep_time=0.4, seed=21)
FORK = QuadSimConfig.fork_default(num_agents=8, ep_time=1.0, capture_radius=2.4, seed=24)
STATS_SECTION = 11 + 7      # blob order (include/quadsim.h): 11 state planes, tick, svd, counters, obstacles, scenario, 2 records, stats


def section_spans(b):
    raw = b.numpy()
    base = 16 + C.sizeof(QsConfigC)
    count = int(np.frombuffer(raw[base + 4:base + 8].tobytes(), np.uint32)[0])
    sizes = np.frombuffer(raw[base + 8:base + 8 + 8 * count].tobytes(), np.uint64).astype(np.int64)
    offs = base + 8 + 8 * count + np.concatenate([[0], np.cumsum(sizes)[:-1]])
    return list(zip(offs.tolist(), sizes.tolist()))


def assert_same_state(x, y, what):
    """Byte-identical blobs, except the double sums of qs_stats, whose atomic adds run in an order that varies between launches."""
    assert x.numel() == y.numel(), what
    off, n = section_spans(x)[STATS_SECTION]
    assert n == C.sizeof(QsStatsC)
    assert torch.equal(x[:off], y[:off]) and torch.equal(x[off + n:], y[off + n:]), f"{what}: state differs"
    sx, sy = (QsStatsC.from_buffer_copy(t[off:off + n].numpy().tobytes()).as_dict() for t in (x, y))
    assert_stats_equal(sx, sy, what)


def sources(case):
    """The snapshots a rejection case passes, and the configuration of the target (128 envs from global env 0)."""
    cfg, change = BASE, ("rew", dict(pos=1.7))
    if case in ("capture_radius", "fork_into_upstream"):
        cfg, change = FORK, ("capture", 1.9)
    if case == "seed":
        cfg = dataclasses.replace(BASE, seed=99)
    if case == "ep_len":
        cfg = dataclasses.replace(BASE, ep_time=0.5)
    old = make_shards(cfg, (37, 91))
    prepare(old, change)
    if case == "rng_step":
        old[1].step(rows(old[1], global_actions(old, 1, 7)[0]))     # one shard a step ahead
    if case == "capture_radius":
        old[1].set_capture_radius(2.0)
    snaps = [s.snapshot() for s in old]
    target = FORK if case == "capture_radius" else BASE
    if case == "gap":
        snaps = snaps[:1]
    elif case == "overlap":
        snaps = [snaps[0], snaps[0], snaps[1]]
    elif case == "truncated":
        snaps[1] = dict(snaps[1], blob=snaps[1]["blob"][:-100].clone())
    elif case == "magic":
        damaged = snaps[1]["blob"].clone()
        damaged[0] ^= 0xFF
        snaps[1] = dict(snaps[1], blob=damaged)
    elif case == "obs_rows":                         # a snapshot dict whose observation is not its blob's: the blobs are fine
        snaps[1] = dict(snaps[1], obs=snaps[1]["obs"][:-8].clone())
    return snaps, dataclasses.replace(target, num_envs=128, env_id_offset=0)


REJECT = {
    # name: (code, words of the message)
    "gap": (QS_ERR_SHAPE, ("gap", "env 37")),
    "overlap": (QS_ERR_SHAPE, ("blob 1", "overlaps blob 0")),
    "rng_step": (QS_ERR_BAD_CONFIG, ("blob 1", "rng_step")),
    "seed": (QS_ERR_BAD_CONFIG, ("blob 0", "seed")),
    "ep_len": (QS_ERR_BAD_CONFIG, ("blob 0", "ep_len")),
    "capture_radius": (QS_ERR_BAD_CONFIG, ("blob 1", "fork.capture_radius", "blob 0's")),
    "fork_into_upstream": (QS_ERR_BAD_CONFIG, ("blob 0", "scenario")),     # the first qs_config field in which they differ
    "truncated": (QS_ERR_SHAPE, ("blob 1", "bytes")),
    "magic": (QS_ERR_SHAPE, ("blob 1", "magic")),
    "obs_rows": (0, ()),                             # the C call accepts these blobs; QuadSwarmSim.restore_shards refuses the obs
    "count_0": (QS_ERR_SHAPE, ("count",)),
    "null_arrays": (QS_ERR_NULL, ("null",)),
}


def _restore_shards_rc(sim, blobs, count=None, null=False):
    datas = [(C.c_uint8 * b.numel()).from_buffer_copy(b.numpy().tobytes()) for b in blobs]
    ptrs = (C.c_void_p * max(len(datas), 1))(*[C.cast(d, C.c_void_p).value for d in datas])
    sizes = (C.c_size_t * max(len(datas), 1))(*[b.numel() for b in blobs])
    n = len(blobs) if count is None else count
    rc = sim._lib.qs_restore_shards(sim._h, None if null else ptrs, None if null else sizes, n, sim._stream())
    return rc, sim._lib.qs_last_error(sim._h).decode()


@pytest.mark.parametrize("case", list(REJECT))
def test_restore_shards_rejects_and_leaves_the_handle_untouched(case):
    snaps, tcfg = sources(case)
    blobs = [s["blob"] for s in snaps]
    target, twin = QuadSwarmSim(tcfg, device="cuda:0"), QuadSwarmSim(tcfg, device="cuda:0")
    for s in (target, twin):
        s.reset()
        s.step(global_actions([s], 1, 5)[0])
    before = target.snapshot()["blob"].clone()
    code, words = REJECT[case]
    if case == "obs_rows":
        with pytest.raises(ValueError, match=rf"snapshot 1 has {(91 * 8 - 8) * 54} observation values"):   # 91 envs x 8, one env short
            target.restore_shards(snaps)
    else:
        if case == "count_0":
            rc, msg = _restore_shards_rc(target, blobs, count=0)
        elif case == "null_arrays":
            rc, msg = _restore_shards_rc(target, blobs, null=True)
        else:
            rc, msg = _restore_shards_rc(target, blobs)
        assert rc == code and all(w in msg for w in words), (rc, msg)
        if case not in ("count_0", "null_arrays"):   # the torch layer reports the same reason
            with pytest.raises(RuntimeError, match=words[-1]):
                target.restore_shards(snaps)
    assert target.rew_coeff_overrides == {}
    assert torch.equal(target.snapshot()["blob"], before), "a rejected call changed the handle"
    assert_runs_equal(run([twin], 2), run([target], 2), "step after a rejected restore_shards")
    assert_same_state(target.snapshot()["blob"], twin.snapshot()["blob"], "after a rejected restore_shards")


# ---------------------------------------------------------------------------------------------------------------------------------
# DevicePPO.load_shards
# ---------------------------------------------------------------------------------------------------------------------------------
def ppo_parts():
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    cfg = QuadSimConfig(num_envs=256, num_agents=8, ep_time=0.3, seed=1)
    return DevicePPO, cfg, PPOConfig(n_steps=16, batch_size=4096, n_epochs=2)


def on_cpu(x):
    if isinstance(x, dict):
        return {k: on_cpu(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return type(x)(on_cpu(v) for v in x)
    return x.detach().cpu() if torch.is_tensor(x) else x


def assert_saved_policy(ppo, ck, what):
    from quad_swarm_rl_stable_baselines3_b200.ppo import _first_difference
    assert _first_difference(on_cpu(ck["policy"]), on_cpu(ppo.policy.state_dict()), "policy") is None, what
    assert _first_difference(on_cpu(ck["optimizer"]), on_cpu(ppo.opt.state_dict()), "optimizer") is None, what
    assert ppo.total_agent_steps == ck["total_agent_steps"], what


def assert_continues(old, new, what, n=40):
    """The simulators of `old` and `new` (lists of DevicePPO covering the same env range) hold the same state and observation and
    continue bitwise under the same actions."""
    assert_bitwise(torch.cat([p.obs for p in new]), torch.cat([p.obs for p in old]), f"{what}: DevicePPO.obs")
    os_, ns = [p.sim for p in old], [p.sim for p in new]
    assert_bitwise(torch.cat([s.obs for s in ns]), torch.cat([s.obs for s in os_]), f"{what}: simulator obs")
    assert_same_sims(os_, ns, what)
    ref = run(os_, n)
    assert bool(torch.stack([x[2] for x in ref]).any()), "no episode ended in the compared steps"
    assert_runs_equal(ref, run(ns, n), what)
    assert_same_sims(os_, ns, f"{what}, after {n} steps")


def test_device_ppo_world_1_resumes_as_2_shards(tmp_path):
    from quad_swarm_rl_stable_baselines3_b200.sharding import shard_config
    DevicePPO, cfg, pc = ppo_parts()
    a = DevicePPO(QuadSwarmSim(cfg, device="cuda:0"), cfg, pc)
    a.learn(2)
    path = tmp_path / "rank0.pt"
    a.save(path)
    ck = torch.load(path, weights_only=True)
    shards = []
    for r in range(2):
        c = shard_config(cfg, r, 2)
        p = DevicePPO(QuadSwarmSim(c, device="cuda:0"), c, pc)
        p.load_shards([path])
        assert all(g["lr"] == pc.learning_rate for g in p.opt.param_groups)
        assert_saved_policy(p, ck, f"shard {r}")
        shards.append(p)
    other = dataclasses.replace(shard_config(cfg, 0, 2), ep_time=0.4)     # another simulator configuration is refused
    with pytest.raises(ValueError, match="sim_config.ep_time"):
        DevicePPO(QuadSwarmSim(other, device="cuda:0"), other, pc).load_shards([path])
    assert_continues([a], shards, "1 -> 2")
    for p in shards:                                                        # and the resumed shards train
        row = p.learn(1)[0]
        assert np.isfinite(row["pg"]) and np.isfinite(row["vf"]), row


def test_device_ppo_2_shards_resume_as_world_1(tmp_path):
    from quad_swarm_rl_stable_baselines3_b200.sharding import shard_config
    DevicePPO, cfg, pc = ppo_parts()
    cs = [shard_config(cfg, r, 2) for r in range(2)]
    s = [DevicePPO(QuadSwarmSim(c, device="cuda:0"), c, pc) for c in cs]
    for p in s:
        p.learn(2)
    paths = [tmp_path / f"rank{r}.pt" for r in range(2)]
    for p, path in zip(s, paths):
        p.save(path)
    probe = DevicePPO(QuadSwarmSim(cfg, device="cuda:0"), cfg, pc)
    with pytest.raises(ValueError, match=r"policy\.\S+ differs"):         # each shard trained on its own: the files disagree
        probe.load_shards(paths)
    # the gradient all-reduce keeps the ranks' policy and Adam state identical: copying rank 0's stands in for it
    s[1].policy.load_state_dict(s[0].policy.state_dict())
    s[1].opt.load_state_dict(s[0].opt.state_dict())
    for p, path in zip(s, paths):
        p.save(path)
    ck = torch.load(paths[0], weights_only=True)
    t = DevicePPO(QuadSwarmSim(cfg, device="cuda:0"), cfg, pc)
    t.load_shards(paths)
    assert_saved_policy(t, ck, "merged")
    assert_continues(s, [t], "2 -> 1")
    row = t.learn(1)[0]
    assert np.isfinite(row["pg"]) and np.isfinite(row["vf"]), row
