"""Exact save / resume: simulator snapshots (qs_snapshot / qs_restore, include/quadsim.h) and DevicePPO checkpoints.

The RNG is counter-based (global env id, launch counter), so a restored handle must continue BITWISE where the snapshotted one stood:
  1. every step-kernel family continues bitwise after a restore, into a fresh handle and into the rewound original, and the state
     at the end of both runs is byte-identical (counters, records, RNG launch counter), the double sums of qs_stats aside;
  2. the blob does not depend on the launch shape: a handle with another block size and reset-first scheduling off continues the same;
  3. taking a snapshot changes nothing;
  4. a snapshot of another configuration, or a damaged blob, is rejected with the field named and the target left untouched;
  5. DevicePPO.save / load: the rollout after a resume is bitwise the one the saved run collects.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from quad_swarm_rl_stable_baselines3_b200.config import QsConfigC, QsStatsC, QuadSimConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim  # noqa: E402

QS_ERR_BAD_CONFIG, QS_ERR_SHAPE = -1, -3
OBST = dict(use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor")
CAM = dict(neighbor_obs_type="ndist_nsangle", obs_repr="cdist_cdistdot_ndist_distdot_nsangle_angledot", camera=dict(cam_pixel_noise=0.7))

# name: (config factory, changed parameter).  Env counts leave the last warp-tile partial; 0.4 s upstream episodes (40 control steps)
# and 1 s fork episodes (12.5 calls of 8 control steps) end several times inside the 60 compared steps.
CASES = {
    "cfg2_k8": (lambda: QuadSimConfig(num_envs=37, num_agents=8, ep_time=0.4, seed=11), ("rew", dict(pos=1.7, quadcol_bin=3.0))),
    "cfg3_obst_mix": (lambda: QuadSimConfig(num_envs=37, num_agents=8, quads_mode="mix", use_downwash=True, neighbor_visible_num=2,
                                            ep_time=0.4, seed=12, **OBST), ("rew", dict(quadcol_bin_obst=2.5))),
    "formation_mix_k8": (lambda: QuadSimConfig(num_envs=37, num_agents=8, quads_mode="mix", ep_time=0.4, seed=13), ("rew", dict(crash=0.5))),
    "k32": (lambda: QuadSimConfig(num_envs=9, num_agents=32, ep_time=0.4, seed=14), ("rew", dict(quadcol_bin_smooth_max=4.0))),
    "k3_partial_lane_group": (lambda: QuadSimConfig(num_envs=53, num_agents=3, neighbor_visible_num=1, ep_time=0.4, seed=15),
                              ("rew", dict(effort=0.2))),
    "k1": (lambda: QuadSimConfig(num_envs=101, num_agents=1, neighbor_obs_type="none", neighbor_visible_num=0, ep_time=0.4, seed=16),
           ("rew", dict(spin=0.3))),
    "fork_default": (lambda: QuadSimConfig.fork_default(num_envs=45, ep_time=1.0, capture_radius=2.4, seed=17), ("capture", 1.9)),
    "fork_camera": (lambda: QuadSimConfig.fork_default(num_envs=45, ep_time=1.0, capture_radius=2.3, seed=18, **CAM), ("capture", 2.0)),
}
PRE, WINDOW = 20, 60


def bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def assert_bitwise(a, b, what):
    assert a.shape == b.shape and torch.equal(bits(a), bits(b)), what


def make_sim(cfg, monkeypatch=None, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    try:
        return QuadSwarmSim(cfg, device="cuda:0")
    finally:
        for k in env:
            monkeypatch.delenv(k)


def actions(sim, n, seed):
    g = torch.Generator(device=sim.device)
    g.manual_seed(seed)
    return [torch.rand((sim.N * sim.K, sim.A), device=sim.device, generator=g) * 2.0 - 1.0 for _ in range(n)]


def prepare(sim, change):
    """reset, staggered clocks, a changed reward coefficient / capture radius, PRE steps: the state a snapshot is taken of."""
    sim.reset()
    L = sim.cfg.to_c().ep_len
    sim.set_state(tick=np.random.RandomState(sim.cfg.seed).randint(0, L, sim.N).astype(np.int32))
    kind, val = change
    if kind == "rew":
        sim.set_rew_coeff(**val)
    else:
        sim.set_capture_radius(val)
    for a in actions(sim, PRE, 100):
        sim.step(a)


def run(sim, n=WINDOW):
    """n steps with seeded actions; per step (obs, rew, done, terminal_obs, reset_success).  The outputs that only finished envs
    write are filled with a canary first, so that the whole buffer compares."""
    out = []
    for a in actions(sim, n, 200):
        sim.terminal_obs.fill_(float("nan"))
        sim.reset_success.fill_(0x5A)
        o, r, d = sim.step(a)
        out.append((o.clone(), r.clone(), d.clone(), sim.terminal_obs.clone(), sim.reset_success.clone()))
    return out


def assert_runs_equal(ref, got, what):
    for t, (x, y) in enumerate(zip(ref, got)):
        for name, a, b in zip(("obs", "rew", "done", "terminal_obs", "reset_success"), x, y):
            assert_bitwise(a, b, f"{what}: {name} of step {t}")


def blob(sim):
    return sim.snapshot()["blob"].clone()


STATS_SECTION = 11 + 7      # blob order (include/quadsim.h): 11 state planes, tick, svd, counters, obstacles, scenario, 2 records, stats


def section_spans(b):
    """(offset, bytes) of every section, from the header's table."""
    raw = b.numpy()
    base = 16 + C.sizeof(QsConfigC)
    count = int(np.frombuffer(raw[base + 4:base + 8].tobytes(), np.uint32)[0])
    sizes = np.frombuffer(raw[base + 8:base + 8 + 8 * count].tobytes(), np.uint64).astype(np.int64)
    offs = base + 8 + 8 * count + np.concatenate([[0], np.cumsum(sizes)[:-1]])
    return list(zip(offs.tolist(), sizes.tolist()))


def assert_same_state(x, y, what):
    """Byte-identical blobs, except the floating-point sums of qs_stats: the episodes of one step add their terms with double
    atomicAdd, in an order that varies between launches, which moves the last bits (the terms themselves are the per-drone records,
    compared bytewise)."""
    assert x.numel() == y.numel(), what
    off, n = section_spans(x)[STATS_SECTION]
    assert n == C.sizeof(QsStatsC)
    assert torch.equal(x[:off], y[:off]) and torch.equal(x[off + n:], y[off + n:]), f"{what}: state differs"
    sx, sy = (QsStatsC.from_buffer_copy(t[off:off + n].numpy().tobytes()).as_dict() for t in (x, y))
    for k in sx:
        if isinstance(sx[k], float):
            assert abs(sx[k] - sy[k]) <= 1e-12 * max(1.0, abs(sx[k])), (what, k, sx[k], sy[k])
        else:
            assert sx[k] == sy[k], (what, k, sx[k], sy[k])


@pytest.mark.parametrize("name", list(CASES))
def test_restore_continues_bitwise(name):
    make, change = CASES[name]
    cfg = make()
    a = make_sim(cfg)
    prepare(a, change)
    snap = a.snapshot()
    assert_bitwise(snap["obs"].cuda(), a.obs, "snapshot obs")
    ref = run(a)
    end = blob(a)
    dones = sum(int(x[2].sum()) for x in ref) // cfg.num_agents
    assert dones >= 1, "no episode ended in the compared window"
    if name == "cfg2_k8":                                       # 192 bytes per drone, 128 per env, behind the header
        header = 16 + C.sizeof(QsConfigC) + 8 + 8 * len(section_spans(snap["blob"]))
        assert snap["blob"].numel() == header + 192 * cfg.num_envs * cfg.num_agents + 128 * cfg.num_envs + C.sizeof(QsStatsC)

    b = make_sim(cfg)                                           # (a) a fresh handle, never reset or stepped
    assert_bitwise(b.restore(snap), snap["obs"].cuda(), "restored obs")
    assert b.rew_coeff_overrides == a.rew_coeff_overrides
    assert_runs_equal(ref, run(b), "fresh handle")
    assert_same_state(blob(b), end, "after the window (fresh handle)")

    a.restore(snap)                                             # (b) the original, rewound
    assert_runs_equal(ref, run(a), "rewound handle")
    assert_same_state(blob(a), end, "after the window (rewound handle)")
    print(f"[{name}] blob {snap['blob'].numel()} bytes, env episodes ended in the window {dones}")


@pytest.mark.parametrize("name", list(CASES))
def test_restore_is_independent_of_launch_shape(name, monkeypatch):
    """Snapshot of a 128-thread-block handle with reset-first scheduling (where the mode has it), restored into a 64-thread-block
    handle with the scheduling off."""
    make, change = CASES[name]
    cfg = make()
    a = make_sim(cfg, monkeypatch, QS_BLOCK="128")
    prepare(a, change)
    snap = a.snapshot()
    ref = run(a)
    b = make_sim(cfg, monkeypatch, QS_BLOCK="64", QS_HOT="0")
    b.restore(snap)
    assert_runs_equal(ref, run(b), "other launch shape")
    assert_same_state(blob(b), blob(a), "after the window")


@pytest.mark.parametrize("name", ["cfg2_k8", "cfg3_obst_mix", "fork_default"])
def test_snapshot_changes_nothing(name):
    make, change = CASES[name]
    cfg = make()
    a, b = make_sim(cfg), make_sim(cfg)
    prepare(a, change)
    prepare(b, change)
    n0 = a.launch_count
    for _ in range(3):
        a.snapshot()
    assert a.launch_count == n0, "qs_snapshot launched a kernel"
    assert_runs_equal(run(b), run(a), "stepping after snapshots")
    assert_same_state(blob(a), blob(b), "after the window")


def _restore_rc(sim, data: bytes):
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    rc = sim._lib.qs_restore(sim._h, C.cast(buf, C.c_void_p), len(data), sim._stream())
    return rc, sim._lib.qs_last_error(sim._h).decode()


BASE = dict(num_envs=37, num_agents=8, ep_time=0.4, seed=11)
REJECT = {
    # name: (target config kwargs, expected code, field named in the message)
    "num_envs": (dict(BASE, num_envs=38), QS_ERR_BAD_CONFIG, "num_envs"),
    "num_agents": (dict(BASE, num_agents=6, neighbor_visible_num=5), QS_ERR_BAD_CONFIG, "num_agents"),
    "scenario": (dict(BASE, quads_mode="mix"), QS_ERR_BAD_CONFIG, "scenario"),
    "obs_repr": (dict(BASE, obs_repr="xyz_vxyz_R_omega_floor"), QS_ERR_BAD_CONFIG, "obs_repr"),
    "seed": (dict(BASE, seed=12), QS_ERR_BAD_CONFIG, "seed"),
    "env_id_offset": (dict(BASE, env_id_offset=37), QS_ERR_BAD_CONFIG, "env_id_offset"),
    "truncated": (BASE, QS_ERR_SHAPE, "bytes"),
    "magic": (BASE, QS_ERR_SHAPE, "magic"),
    "version": (BASE, QS_ERR_SHAPE, "version"),
}


@pytest.mark.parametrize("name", list(REJECT))
def test_restore_rejects_and_leaves_the_handle_untouched(name):
    src = make_sim(QuadSimConfig(**BASE))
    prepare(src, ("rew", dict(pos=1.7)))
    data = bytearray(src.snapshot()["blob"].numpy().tobytes())
    kw, code, field = REJECT[name]
    if name == "truncated":
        data = data[:-100]
    elif name == "magic":
        data[0] ^= 0xFF
    elif name == "version":
        data[4:8] = (2).to_bytes(4, "little")
    cfg = QuadSimConfig(**kw)
    target, twin = make_sim(cfg), make_sim(cfg)
    for s in (target, twin):
        s.reset()
        s.step(actions(s, 1, 5)[0])
    rc, msg = _restore_rc(target, bytes(data))
    assert rc == code and field in msg, (rc, msg)
    with pytest.raises(RuntimeError, match=field):
        target.restore({"blob": torch.frombuffer(bytearray(data), dtype=torch.uint8), "obs": target.obs.cpu()})
    assert target.rew_coeff_overrides == {}
    assert_runs_equal(run(twin, 2), run(target, 2), "step after a rejected restore")
    assert_same_state(blob(target), blob(twin), "after a rejected restore")


# ---------------------------------------------------------------------------------------------------------------------------------
# DevicePPO checkpoints
# ---------------------------------------------------------------------------------------------------------------------------------
PPO_CASES = {
    # name: (sim config factory, PPOConfig kwargs): hidden 256 runs the rollout forward on the fused kernel, hidden 64 on torch
    "cfg2_fused": (lambda: QuadSimConfig(num_envs=256, num_agents=8, ep_time=0.3, seed=1), dict(hidden=256, neighbor_hidden=256)),
    "cfg2_torch_h64": (lambda: QuadSimConfig(num_envs=256, num_agents=8, ep_time=0.3, seed=1), dict(hidden=64, neighbor_hidden=32)),
    "fork_fused": (lambda: QuadSimConfig.fork_default(num_envs=256, ep_time=1.0, seed=3), dict(hidden=256, neighbor_hidden=256)),
}
ROLLOUT = ("obs_buf", "act_buf", "logp_buf", "val_buf", "rew_buf", "done_buf", "adv", "ret")


@pytest.mark.parametrize("name", list(PPO_CASES))
def test_device_ppo_resume_is_bitwise(name, tmp_path):
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    make, kw = PPO_CASES[name]
    cfg = make()
    pc = PPOConfig(n_steps=16, batch_size=4096, n_epochs=2, **kw)
    a = DevicePPO(QuadSwarmSim(cfg, device="cuda:0"), cfg, pc)
    assert (a.fused is not None) == (kw["hidden"] == 256)
    a.learn(1)
    path = tmp_path / "a.pt"
    a.save(path)
    # the saved run goes on first: building another DevicePPO reseeds the global torch generators
    a.collect()
    ref = {k: getattr(a, k).clone() for k in ROLLOUT}
    rng_after = torch.cuda.get_rng_state()
    with pytest.raises(RuntimeError, match="update"):
        a.save(tmp_path / "refused.pt")

    ck = torch.load(path, weights_only=True)
    assert ck["version"] == DevicePPO.CHECKPOINT_VERSION and ck["ppo_config"]["hidden"] == kw["hidden"]
    assert ck["sim_config"]["num_envs"] == cfg.num_envs and ck["total_agent_steps"] == 16 * cfg.num_envs * cfg.num_agents

    b = DevicePPO(QuadSwarmSim(cfg, device="cuda:0"), cfg, pc)
    b.load(path)
    assert b.total_agent_steps == ck["total_agent_steps"]
    assert all(g["lr"] == pc.learning_rate for g in b.opt.param_groups)
    b.save(tmp_path / "b.pt")                                   # save -> load -> save: the same simulator state
    assert torch.equal(torch.load(tmp_path / "b.pt", weights_only=True)["sim"]["blob"], ck["sim"]["blob"])
    b.collect()
    for k in ROLLOUT:
        assert_bitwise(getattr(b, k), ref[k], f"{k} of the resumed rollout")
    assert bool(ref["done_buf"].any()), "no episode ended in the rollout"
    assert torch.equal(torch.cuda.get_rng_state(), rng_after), "the resumed rollout drew a different amount of exploration noise"

    # One update each.  Both runs share this process's CUDA generator, so each update starts from the generator state that follows
    # the rollout (the minibatch permutations), as two separate processes would.  Not bitwise: the bias-gradient kernels reduce
    # with atomics, so the summation order (and the last bits of every gradient) varies between runs.  Every parameter must agree to
    # a quarter of one Adam step (~learning_rate) and the two updates to 1e-2 of the update's own size; measured on a B200 over the 16
    # Adam steps: at most 3e-6 per parameter and 8e-4 of the update (cfg2_fused, the widest bias reductions), 1e-6 for the others.
    w0 = torch.cat([p.detach().reshape(-1) for p in a.policy.parameters()]).clone()
    torch.cuda.set_rng_state(rng_after)
    a.update()
    torch.cuda.set_rng_state(rng_after)
    b.update()
    wa = torch.cat([p.detach().reshape(-1) for p in a.policy.parameters()])
    wb = torch.cat([p.detach().reshape(-1) for p in b.policy.parameters()])
    step, diff = float((wa - w0).norm()), float((wa - wb).norm())
    print(f"[{name}] update norm {step:.3e}, |a - b| {diff:.3e}, max abs {float((wa - wb).abs().max()):.3e}")
    assert step > 0 and diff <= 1e-2 * step, (step, diff)
    assert float((wa - wb).abs().max()) <= 0.25 * pc.learning_rate
