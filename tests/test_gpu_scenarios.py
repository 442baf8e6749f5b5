"""GPU parity of the formation scenarios (SURVEY.md 8 f2: scenarios/*.py of the upstream env) against the CPU oracle, which is
pinned against taped runs of the reference (tests/test_oracle_golden.py, trace_scen_*).  Same protocol as
test_gpu_parity.py: the GPU state -- including each env's scenario row -- is copied into the oracle before every step, both
step with the same actions and Philox draws, and goals, scenario rows, observations, rewards and dones are compared."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import OracleEnv  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402
from test_gpu_parity import _sim, oracle_state, run_parity  # noqa: E402

SC_FORMATION, SC_SIZE, SC_HIGHEST, SC_LOWEST, SC_CTL, SC_INCREASE = 1, 2, 4, 5, 9, 10


def fast_timers(row):
    """control_step_for_sec is 400..599 control steps in the reference; shorten it to 5 + e % 7 so that the goal-changing branch
    runs many times inside a short test, every env with its own period.  Rewrites the [N, QS_SC_COUNT] rows in place and returns
    whether any changed (after a reset the row holds a fresh reference timer again)."""
    ctl = row[:, SC_CTL]
    slow = ctl > 50
    if slow.any():
        row[:, SC_CTL] = torch.where(slow, 5.0 + (torch.arange(row.shape[0], device=row.device) % 7).float(), ctl)
    return bool(slow.any())


def near_turning_points(row):
    """dynamic_formations: put the even envs just below / above the turning points of the breathing formation (in place)."""
    half = torch.arange(row.shape[0], device=row.device) % 2 == 0
    sign = torch.where(row[:, SC_INCREASE] > 0, 1.0, -1.0)
    row[:, SC_SIZE] = torch.where(half, sign * (row[:, SC_HIGHEST] - 0.004), row[:, SC_SIZE])

SCENARIO_CONFIGS = {
    # name: (config kwargs, steps, timer override: goals change every few steps instead of every 4-6 s)
    "static_diff_k8": (dict(num_envs=40, num_agents=8, quads_mode="static_diff_goal", ep_time=0.2), 50, False),
    "static_diff_k12": (dict(num_envs=24, num_agents=12, quads_mode="static_diff_goal", ep_time=0.15), 40, False),
    "static_diff_k27": (dict(num_envs=16, num_agents=27, quads_mode="static_diff_goal", ep_time=0.12), 30, False),
    "dyn_same_k3": (dict(num_envs=40, num_agents=3, quads_mode="dynamic_same_goal", neighbor_visible_num=2, ep_time=0.4), 90, True),
    "dyn_diff_k4": (dict(num_envs=40, num_agents=4, quads_mode="dynamic_diff_goal", neighbor_visible_num=3, ep_time=0.4), 90, True),
    "dyn_diff_k9": (dict(num_envs=24, num_agents=9, quads_mode="dynamic_diff_goal", ep_time=0.3), 70, True),
    "swap_k3": (dict(num_envs=40, num_agents=3, quads_mode="swap_goals", neighbor_visible_num=1, ep_time=0.4), 90, True),
    "swap_k8": (dict(num_envs=32, num_agents=8, quads_mode="swap_goals", ep_time=0.4), 90, True),
    "runaway_k5": (dict(num_envs=40, num_agents=5, quads_mode="run_away", neighbor_visible_num=2, ep_time=1.2), 140, False),
    "runaway_k2": (dict(num_envs=24, num_agents=2, quads_mode="run_away", neighbor_visible_num=1, ep_time=1.2), 130, False),
    "swarm_k6": (dict(num_envs=32, num_agents=6, quads_mode="swarm_vs_swarm", neighbor_visible_num=2, ep_time=0.4), 90, True),
    "swarm_k4": (dict(num_envs=32, num_agents=4, quads_mode="swarm_vs_swarm", neighbor_visible_num=2, ep_time=0.3), 70, True),
    "swarm_k7": (dict(num_envs=24, num_agents=7, quads_mode="swarm_vs_swarm", ep_time=0.3), 70, True),
    "dynform_k5": (dict(num_envs=40, num_agents=5, quads_mode="dynamic_formations", neighbor_visible_num=2, ep_time=0.5), 110, False),
    "lissajous_k3": (dict(num_envs=40, num_agents=3, quads_mode="ep_lissajous3D", neighbor_visible_num=2, ep_time=0.4), 90, False),
    "bezier_k3": (dict(num_envs=40, num_agents=3, quads_mode="ep_rand_bezier", neighbor_visible_num=2, ep_time=5.2), 70, False),
    "mix_k8": (dict(num_envs=64, num_agents=8, quads_mode="mix", ep_time=0.3, use_downwash=True), 100, True),
    "mix_k1": (dict(num_envs=70, num_agents=1, quads_mode="mix", neighbor_obs_type="none", neighbor_visible_num=0, ep_time=0.3), 70, True),
}


@pytest.mark.parametrize("name", list(SCENARIO_CONFIGS))
def test_scenario_parity(name):
    kw, steps, fast_timer = SCENARIO_CONFIGS[name]
    cfg = QuadSimConfig(seed=17, **kw)
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(cfg.num_envs)]
    N, K = cfg.num_envs, cfg.num_agents

    # reset parity: goals, spawn positions around them, scenario rows
    obs = sim.reset().cpu().numpy()
    ref = np.concatenate([o.reset() for o in oracles])
    st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
    os_ = oracle_state(oracles)
    rows = np.stack([o.get_scenario() for o in oracles])
    np.testing.assert_allclose(st["goal"], os_["goal"], atol=3e-6)
    np.testing.assert_allclose(st["scenario"], rows, atol=3e-6)
    yaw_ok = np.abs(st["rot"] - os_["rot"]).max(axis=1) < 1e-5          # spawn-yaw rejection ties aside
    assert yaw_ok.mean() > 0.98
    np.testing.assert_allclose(st["pos"][yaw_ok], os_["pos"][yaw_ok], atol=3e-6)
    ok_rows = np.repeat(yaw_ok.reshape(N, K).all(axis=1), K)
    np.testing.assert_allclose(obs[ok_rows], ref[ok_rows], atol=3e-5)

    def hook(s):
        row = sim.get_state(("scenario",))["scenario"]
        changed = fast_timer and fast_timers(row)
        if name.startswith("dynform") and s % 25 == 3:
            near_turning_points(row)
            changed = True
        if changed:
            sim.set_state(scenario=row)
        if name.startswith("bezier") and s == 4:
            # jump to just before the 5 s resampling of the Bezier arc (tick % 500 == 0)
            sim.set_state(tick=torch.full((N,), 496, dtype=torch.int32))

    # the Bezier test jumps the tick forward, which breaks the fixed-length-episode assumption of the distance windows
    worst, cnt = run_parity("scen_" + name, cfg, sim, oracles, "hover", steps, hook, check_records=not name.startswith("bezier"))
    assert worst["goal"] <= 3e-6
    if not name.startswith("static") and not name.startswith("bezier"):
        assert cnt["done"] >= N
    if not name.startswith("static"):
        assert cnt["goal_moves"] >= N, cnt          # the goal-changing branches did run
    if name.startswith("mix"):
        seen = set()
        for _ in range(3):
            seen |= set(int(v) for v in sim.get_state(("scenario",))["scenario"][:, 0].cpu().numpy())
        assert len(seen) >= (4 if K == 1 else 7), seen


def test_mix_long_run_statistics():
    """65536 drones of the upstream training recipe (quads_mode=mix) free-running for 700 steps: every scenario is drawn with
    probability 1/9, goals stay finite and inside a generous box, timers are in the reference's 400..599 range."""
    cfg = QuadSimConfig(seed=23, num_envs=8192, num_agents=8, quads_mode="mix", ep_time=3.0)
    sim = _sim(cfg)
    sim.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    counts = np.zeros(14)
    for s in range(700):
        a = torch.rand((cfg.num_envs * 8, 4), device="cuda", generator=g) * 0.3 - 0.1
        sim.step(a)
        if s % 100 == 50:
            st = sim.get_state(("scenario", "goal"))
            row, goal = st["scenario"].cpu().numpy(), st["goal"].cpu().numpy()
            counts += np.bincount(row[:, 0].astype(int), minlength=14)
            assert np.isfinite(goal).all() and np.abs(goal).max() < 12.0
            timed = np.isin(row[:, 0], (6, 7, 8, 13))
            assert ((row[timed, SC_CTL] >= 400) & (row[timed, SC_CTL] <= 599)).all()
            assert (row[~timed & (row[:, 0] != 9), SC_CTL] == 0).all()
    frac = counts / counts.sum()
    used = [0, 5, 6, 7, 8, 9, 11, 12, 13]
    assert np.abs(frac[used] - 1 / 9).max() < 0.02, frac
    assert frac[[1, 2, 3, 4, 10]].sum() == 0
    assert sim.episode_stats()["episodes"] >= 2 * cfg.num_envs


def test_mix_goal_invariants_full_size():
    """Size-independent properties at the BASELINE batch size (65536 envs x 8 quads, quads_mode=mix): scenarios with one common
    goal give every drone the same goal; circle / grid / cube formations are centred on formation_center by construction
    (scenarios/base.py:60-112), for swarm_vs_swarm each half on its own goal centre; a shuffle permutes rows, it never duplicates one."""
    cfg = QuadSimConfig(seed=31, num_envs=65536, num_agents=8, quads_mode="mix", ep_time=1.0)
    sim = _sim(cfg)
    sim.reset()
    g = torch.Generator(device="cuda").manual_seed(3)
    checked = dict(common=0, centred=0, swarm=0)
    for s in range(230):
        sim.step(torch.rand((cfg.num_envs * 8, 4), device="cuda", generator=g) * 0.3 - 0.1)
        if s % 45 != 44:
            continue
        st = sim.get_state(("scenario", "goal"))
        row, goal = st["scenario"].double(), st["goal"].double().reshape(cfg.num_envs, 8, 3)
        scen, form = row[:, 0].long(), row[:, 1].long()
        common = (scen == 0) | (scen == 6) | (scen == 11) | (scen == 12)
        spread = (goal - goal[:, :1]).abs().amax(dim=(1, 2))
        assert spread[common].max().item() == 0.0
        checked["common"] += int(common.sum())
        symmetric = (form != 3)                                         # every formation but the sphere is mean-centred / symmetric
        cen = ((scen == 5) | (scen == 7) | (scen == 8) | (scen == 9)) & symmetric
        err = (goal.mean(dim=1) - row[:, 6:9]).abs().amax(dim=1)
        assert err[cen].max().item() < 2e-6, err[cen].max().item()
        checked["centred"] += int(cen.sum())
        sw = (scen == 13) & symmetric
        e1 = (goal[:, :4].mean(dim=1) - row[:, 12:15]).abs().amax(dim=1)
        e2 = (goal[:, 4:].mean(dim=1) - row[:, 15:18]).abs().amax(dim=1)
        assert e1[sw].max().item() < 2e-6 and e2[sw].max().item() < 2e-6
        checked["swarm"] += int(sw.sum())
        # distinct rows: formations with a positive size never give two drones the same goal
        sized = ((scen == 5) | (scen == 7) | (scen == 8)) & (row[:, 2] > 0.2)
        d = (goal[:, :, None, :] - goal[:, None, :, :]).norm(dim=-1) + torch.eye(8, device=goal.device, dtype=goal.dtype) * 10
        assert d[sized].amin().item() > 0.05
    assert min(checked.values()) > 10000, checked


def test_mix_shards_reproduce_the_single_gpu_run():
    """Multi-GPU sharding of the formation scenarios: two handles owning envs [0, 32) and [32, 64) (env_id_offset) reproduce the
    64-env handle bit for bit -- scenario draws, goals, observations, episode records -- because every draw is keyed by the
    global env id."""
    kw = dict(num_agents=8, quads_mode="mix", ep_time=0.25, seed=77)
    whole = _sim(QuadSimConfig(num_envs=64, **kw))
    parts = [_sim(QuadSimConfig(num_envs=32, env_id_offset=o, **kw)) for o in (0, 32)]
    o_w = whole.reset().clone()
    o_p = torch.cat([p.reset() for p in parts])
    assert torch.equal(o_w, o_p)
    g = torch.Generator(device="cuda").manual_seed(5)
    for s in range(60):
        a = torch.rand((64 * 8, 4), device="cuda", generator=g) * 0.4 - 0.1
        ow, rw, dw = whole.step(a)
        outs = [p.step(a[i * 256:(i + 1) * 256].contiguous()) for i, p in enumerate(parts)]
        assert torch.equal(ow, torch.cat([o[0] for o in outs])) and torch.equal(rw, torch.cat([o[1] for o in outs]))
        assert torch.equal(dw, torch.cat([o[2] for o in outs]))
    sw = whole.get_state(("scenario", "goal"))
    sp = [p.get_state(("scenario", "goal")) for p in parts]
    assert torch.equal(sw["scenario"], torch.cat([x["scenario"] for x in sp])) and torch.equal(sw["goal"], torch.cat([x["goal"] for x in sp]))
    rw_ = whole.episode_records()
    rp = [p.episode_records() for p in parts]
    assert torch.equal(rw_["env"], torch.cat([x["env"] for x in rp])) and torch.equal(rw_["agent"], torch.cat([x["agent"] for x in rp]))
    assert int(rw_["env"][:, 0].min()) >= 2                       # every env finished at least two episodes
