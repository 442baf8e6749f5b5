"""Goal events of the formation scenarios against the oracle at every lane-group width, with event timing that differs between the
env groups of a warp.

scenario_event (scenario_kernels.cuh) runs on a step where an env's timer, its run_away second or its 5 s Bezier period comes
round; dynamic_formations and ep_lissajous3D move the goals on every step.  Its K-dependent paths -- circles stacked in layers of 8,
grid_dims of a prime K, the cube's floor dimension, swarm halves of different sizes, shuffles of more than 9 rows (more than two
Philox draws), padding lanes of a 32-lane group, the sphere's 3 rows for formations of fewer than 3 drones -- and, at 16 lanes, a
warp whose two envs do not fire on the same step (scenario_event syncs its group and uses the warp's exchange buffer while the other
group has no event) are what these cases reach.  Each case drives its events so that they fire early and often:
  timer     control_step_for_sec cut to 5 + e % 7 after every reset (test_gpu_scenarios.fast_timers);
  forced    the same, and every env that starts an episode evaluates formation e % 8 (the row is teacher-forced into the oracle, so
            parity holds for any row): all eight formations at every K of the table;
  dynform   formation e % 8 after every reset, and the even envs put next to a turning point every 25 steps;
  runaway   clocks moved to just before the 1 s events (95 + e % 4, then 195 + e % 4) and on to the episode's end;
  bezier    clocks moved to just before the 5 s resampling (496 + e % 3, then 996 + e % 3) and to the episode's end, which starts
            new episodes (tick 1 resamples too) at a step of each env's own;
  perstep   nothing to drive: the goal moves on every step.
The protocol is test_gpu_parity.run_parity's (goals and scenario rows compared every step, ids and timers exactly, the rest at
3e-6) over the whole batch through test_gpu_staggered.CheckedSim (done rule, terminal observations and episode records of the
envs that ended, and those of the others untouched).  The envs leave the last warp of a 16-lane group with one env.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from oracle import OracleEnv  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.config import SCENARIOS, QuadSimConfig  # noqa: E402
from test_gpu_parity import _sim, action_batch, run_parity  # noqa: E402
from test_gpu_scenarios import (SC_CTL, SC_FORMATION, SC_HIGHEST, SC_LOWEST, SC_SIZE, fast_timers,  # noqa: E402
                                near_turning_points)
from test_gpu_staggered import HOT_CAP, CheckedSim, assert_bitwise, assert_handles_equal, envs_per_tile, tile_counts  # noqa: E402

DYN_SAME, DYN_DIFF, SWAP, DYNFORM = (SCENARIOS[m] for m in ("dynamic_same_goal", "dynamic_diff_goal", "swap_goals", "dynamic_formations"))
LISSAJOUS, BEZIER, SWARM, RUN_AWAY = (SCENARIOS[m] for m in ("ep_lissajous3D", "ep_rand_bezier", "swarm_vs_swarm", "run_away"))
TIMED = (DYN_SAME, DYN_DIFF, SWAP, SWARM)               # goals change when tick % control_step_for_sec == 0
QF_SPHERE = 3                                           # QUADS_FORMATION_LIST index of the sphere (scenario_kernels.cuh)
DW = dict(use_downwash=True)


def case(mode, K, n_envs, steps, driver, ep_time=0.3, **kw):
    if K <= 3:
        kw.setdefault("neighbor_visible_num", K - 1)
    return dict(num_agents=K, quads_mode=mode, ep_time=ep_time, **kw), n_envs, steps, driver


def runaway(K, n_envs, **kw):
    return case("run_away", K, n_envs, 32, "runaway", ep_time=2.1, **kw)


def bezier(K, n_envs, **kw):
    return case("ep_rand_bezier", K, n_envs, 30, "bezier", ep_time=10.2, **kw)


def dynform(K, n_envs, **kw):
    return case("dynamic_formations", K, n_envs, 56, "dynform", ep_time=0.5, **kw)


# name: (config kwargs, envs, steps, event driver).  dw = use_downwash (feature set 6, else 4).  Lane groups of 16 hold two envs
# per warp (odd envs: the last warp holds one), of 32 one.
SCENARIO_WIDTH_CASES = {
    # 2 lanes (16 envs per warp): swarm halves of one drone and dynamic_diff_goal / dynamic_formations with K = 2 evaluate the
    # sphere with its 3 rows
    "swarm_k2": case("swarm_vs_swarm", 2, 27, 45, "timer"),
    "dyndiff_k2": case("dynamic_diff_goal", 2, 27, 45, "timer"),
    "dynform_k2_dw": dynform(2, 27, **DW),
    "dynsame_k2_dw": case("dynamic_same_goal", 2, 27, 45, "forced", **DW),
    "lissajous_k2": case("ep_lissajous3D", 2, 27, 40, "perstep"),
    "bezier_k2_dw": bezier(2, 27, **DW),
    # 4 and 8 lanes: the event scenarios test_gpu_scenarios.py has no case for at these widths
    "runaway_k3_dw": runaway(3, 21, **DW),
    "dynform_k4": dynform(4, 21, neighbor_visible_num=2),
    "mix_k4_dw": case("mix", 4, 21, 70, "timer", neighbor_visible_num=2, **DW),
    "dynsame_k6": case("dynamic_same_goal", 6, 11, 45, "forced", neighbor_visible_num=2),
    "dyndiff_k7_dw": case("dynamic_diff_goal", 7, 11, 45, "timer", neighbor_visible_num=2, **DW),
    "lissajous_k8_dw": case("ep_lissajous3D", 8, 11, 40, "perstep", neighbor_visible_num=2, **DW),
    "bezier_k5": bezier(5, 11, neighbor_visible_num=2),
    # 16 lanes
    "dynsame_k12": case("dynamic_same_goal", 12, 13, 45, "forced"),       # circle 8 + 4, grid 3 x 4
    "swap_k13_dw": case("swap_goals", 13, 13, 45, "timer", **DW),         # prime K: 12 swaps in 3 draws
    "swap_k16": case("swap_goals", 16, 13, 45, "timer"),                  # no padding lanes
    "swarm_k15": case("swarm_vs_swarm", 15, 15, 45, "timer"),             # halves 7 / 8: cube floor dims 1 / 2
    "dyndiff_k16_dw": case("dynamic_diff_goal", 16, 13, 45, "timer", **DW),   # no padding lanes; circle of two whole layers
    "dynform_k16_dw": dynform(16, 13, **DW),                               # two whole circle layers, 4 x 4 grid
    "lissajous_k12_dw": case("ep_lissajous3D", 12, 13, 40, "perstep", **DW),
    "bezier_k13": bezier(13, 13),
    "runaway_k12_dw": runaway(12, 13, **DW),
    "runaway_k16": runaway(16, 13),
    "mix_k12": case("mix", 12, 15, 70, "timer"),
    "mix_k14_dw": case("mix", 14, 13, 70, "timer", **DW),
    # 32 lanes
    "dynsame_k27_dw": case("dynamic_same_goal", 27, 9, 45, "forced", **DW),   # cube: int(27 ** (1/3)) == 2, 27 rows; circle 8+8+8+3
    "dyndiff_k17": case("dynamic_diff_goal", 17, 9, 45, "timer"),             # 15 padding lanes; prime grid 1 x 17
    "dyndiff_k32_dw": case("dynamic_diff_goal", 32, 9, 45, "timer", **DW),    # no padding lanes; circle of four whole layers
    "swap_k32": case("swap_goals", 32, 9, 45, "timer"),                       # 31 swaps: 8 draws
    "swap_k29_dw": case("swap_goals", 29, 9, 45, "timer", **DW),              # 3 padding lanes, prime
    "swarm_k27_dw": case("swarm_vs_swarm", 27, 9, 45, "timer", **DW),         # halves 13 / 14
    "swarm_k32": case("swarm_vs_swarm", 32, 9, 45, "timer"),                  # halves 16 / 16: two whole circle layers each
    "dynform_k27": dynform(27, 9),
    "lissajous_k32_dw": case("ep_lissajous3D", 32, 9, 40, "perstep", **DW),
    "bezier_k27_dw": bezier(27, 9, **DW),
    "runaway_k29": runaway(29, 9),
    "runaway_k32_dw": runaway(32, 9, **DW),
    "mix_k27": case("mix", 27, 9, 70, "timer"),
    "mix_k32_dw": case("mix", 32, 9, 70, "timer", **DW),
}


def formation_limits(formation, low, high, n):
    """(lowest, highest) formation size of update_formation_and_relate_param (scen_update_formation, scenario_kernels.cuh)."""
    if formation <= 2:
        return 0.5 * low / 0.3826834323650898, 0.5 * high / 0.3826834323650898
    if formation == 3:
        ratio = (1.75388487222762 - 0.0920858134405214) / (1.0 + (n / 10.3632729642351) ** 0.860487305801679) + 0.0920858134405214
        return low / ratio, high / ratio
    return low, high


def force_formations(row, fresh, K, breathing):
    """Envs `fresh` (just reset) evaluate formation e % 8.  dynamic_formations keeps the drawn size as a fraction of its range
    (QUADS_PARAMS_DICT: 0 .. 1.0); dynamic_same_goal (a point, size 0, in the reference) gets the middle of static_diff_goal's
    range (0.25 .. 0.5), so that the rows are distinct goals."""
    for e in np.flatnonzero(fresh):
        f = e % 8
        lo, hi = formation_limits(f, 0.0, 1.0, K) if breathing else formation_limits(f, 0.25, 0.5, K)
        frac = row[e, SC_SIZE] / row[e, SC_HIGHEST] if breathing else 0.5
        row[e, [SC_FORMATION, SC_LOWEST, SC_HIGHEST, SC_SIZE]] = (f, lo, hi, lo + frac * (hi - lo))


def goal_tolerance(cfg, *rows):
    """Goal tolerance per drone: 3e-6, and for a sphere the error of its fp32 spiral.  sphere_point (scenario_kernels.cuh) turns
    point r of m about the axis by t * x radians, t = -1 + 1 / (m - 1) + r * inc in [-1, 1] and x = 0.1 + 1.2 m (38.5 at m = 32):
    t carries a few ulps of 1 from its approximate divisions, each worth x * 2^-23 rad, so the goal moves by size * x * 2^-23 per
    ulp of t -- 7e-6 m at 27 drones and dynamic_formations' largest sphere, where the float64 reference has none.  Bound: 8 ulps."""
    K = cfg.num_agents
    n = np.full(len(rows[0]), float(K))
    tol = np.full(len(rows[0]), 3e-6)
    for row in rows:
        sphere = row[:, SC_FORMATION] == QF_SPHERE
        swarm = row[:, 0] == SWARM
        m = np.maximum(np.where(swarm, K - K // 2, n), 3)
        tol = np.maximum(tol, np.where(sphere, 3e-6 + np.abs(row[:, SC_SIZE]) * (0.1 + 1.2 * m) * 8 * 2.0 ** -23, 0.0))
    return np.repeat(tol, K)


class EventSim(CheckedSim):
    """CheckedSim over the whole batch that also counts, from the rows and clocks before each step, the envs in which the
    scenario's goal-changing code ran: `fired` (scenario_event, or a turning point of dynamic_formations) and goal moves."""

    def __init__(self, sim):
        super().__init__(sim, np.arange(sim.N), seed=1)
        N, cfg = sim.N, sim.cfg
        self.freq = int(round(cfg.sim_freq / cfg.sim_steps))
        self.fired, self.resampled, self.moved = np.zeros(N, int), np.zeros(N, int), np.zeros(N, int)
        self.mixed_pairs = 0                    # (step, warp) pairs of a 16-lane group in which exactly one env fired
        self.scen_seen, self.scen_events, self.formations = set(), {}, set()

    def step(self, a_small):
        sim, N, K = self.sim, self.sim.N, self.K
        st0 = {k: v.cpu().numpy() for k, v in sim.get_state(("tick", "scenario", "goal")).items()}
        out = super().step(a_small)
        st1 = {k: v.cpu().numpy() for k, v in sim.get_state(("scenario", "goal")).items()}
        row0, row1, t1 = st0["scenario"], st1["scenario"], st0["tick"].astype(np.int64) + 1
        scen, ctl = row0[:, 0].astype(int), row0[:, SC_CTL].astype(int)
        ended = t1 > self.ep_len                # scenario.step() ran before the reset: its goals are overwritten
        timer = np.isin(scen, TIMED) & (ctl > 0) & (t1 % np.maximum(ctl, 1) == 0)
        run_away = (scen == RUN_AWAY) & (t1 % self.freq == 0)
        resample = (scen == BEZIER) & ((t1 % (5 * self.freq) == 0) | (t1 == 1))
        turn = (scen == DYNFORM) & ((row0[:, SC_SIZE] <= -row0[:, SC_HIGHEST]) | (row0[:, SC_SIZE] >= row0[:, SC_HIGHEST]))
        fired = timer | run_away | resample | turn
        moved = (np.abs(st1["goal"] - st0["goal"]).max(axis=1) > 0).reshape(N, K).any(axis=1) & ~ended
        self.fired += fired
        self.resampled += resample & (t1 > 1)
        self.moved += moved
        if self.gpw == 2:
            f = fired[: N - N % 2].reshape(-1, 2)
            self.mixed_pairs += int((f[:, 0] != f[:, 1]).sum())
        event = fired | (moved & np.isin(scen, (DYNFORM, LISSAJOUS)))
        for s in np.unique(scen):
            self.scen_seen.add(int(s))
            self.scen_events[int(s)] = self.scen_events.get(int(s), 0) + int(event[scen == s].sum())
        # formations evaluated: dynamic_same_goal's at its event, the new draw of dynamic_diff_goal / swarm_vs_swarm, and
        # dynamic_formations' on every step
        same = ((scen == DYN_SAME) & fired | (scen == DYNFORM)) & ~ended
        drawn = np.isin(scen, (DYN_DIFF, SWARM)) & fired & ~ended
        self.formations |= set(row0[same, SC_FORMATION].astype(int)) | set(row1[drawn, SC_FORMATION].astype(int))
        return out


def run_case(name):
    kw, N, steps, driver = SCENARIO_WIDTH_CASES[name]
    cfg = QuadSimConfig(seed=61, num_envs=N, **kw)
    K, L = cfg.num_agents, cfg.ep_len
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(N)]
    sim.reset()
    for o in oracles:
        o.reset()
    wrap = EventSim(sim)
    e = np.arange(N)
    jumps = {"runaway": {2: 95 + e % 4, 12: 195 + e % 4, 22: L - 4 + e % 4},
             "bezier": {3: 496 + e % 3, 11: 996 + e % 3, 19: L - 3 + e % 3}}.get(driver, {})

    def hook(s):
        if s in jumps:
            wrap.set_ticks(jumps[s])
        if driver not in ("timer", "forced", "dynform"):
            return
        row = sim.get_state(("scenario",))["scenario"]
        changed = driver != "dynform" and fast_timers(row)
        if driver in ("forced", "dynform"):
            fresh = sim.get_state(("tick",))["tick"].cpu().numpy() == 0
            if fresh.any():
                r = row.cpu().numpy()
                force_formations(r, fresh, K, driver == "dynform")
                row = torch.from_numpy(r).to(row.device)
                changed = True
        if driver == "dynform" and s % 25 == 3:
            near_turning_points(row)
            changed = True
        if changed:
            sim.set_state(scenario=row)

    worst, cnt = run_parity("width_" + name, cfg, wrap, oracles, "hover", steps, hook, record_envs=wrap.comparable,
                            goal_atol=lambda pre, post: goal_tolerance(cfg, pre["scenario"], post["scenario"]))
    return cfg, wrap, worst, cnt


@pytest.mark.parametrize("name", list(SCENARIO_WIDTH_CASES))
def test_scenario_events_at_width(name):
    kw, N, steps, driver = SCENARIO_WIDTH_CASES[name]
    cfg, wrap, worst, cnt = run_case(name)
    scen = cfg.scenario_id()
    print(f"[width_{name}] fired per env {wrap.fired.tolist()} 5 s resamples {wrap.resampled.tolist()} mixed (step, warp) pairs "
          f"{wrap.mixed_pairs} formations {sorted(wrap.formations)} scenarios {wrap.scen_events} records {cnt.get('records', 0)}")
    if scen == SCENARIOS["mix"]:
        assert len(wrap.scen_seen) >= 7, wrap.scen_seen
        quiet = {s for s in wrap.scen_seen if s not in (SCENARIOS["static_same_goal"], SCENARIOS["static_diff_goal"])
                 and wrap.scen_events[s] == 0}
        assert not quiet, f"scenarios drawn whose goal events never ran: {quiet}"
    elif driver in ("timer", "forced"):
        assert (wrap.fired >= 2).all(), wrap.fired
    elif driver == "runaway":
        assert (wrap.fired >= 2).all(), wrap.fired
    elif driver == "bezier":
        assert (wrap.resampled >= 2).all(), wrap.resampled
    else:
        assert (wrap.moved >= steps // 2).all(), wrap.moved
        if driver == "dynform":
            assert (wrap.fired[::2] >= 1).all(), wrap.fired            # the even envs turned
    if driver in ("forced", "dynform"):
        assert wrap.formations == set(range(8)), wrap.formations
    elif cfg.num_agents == 2 and scen in (DYN_DIFF, SWARM):
        assert QF_SPHERE in wrap.formations, wrap.formations            # drawn at an event: 3 rows for 2 drones
    if wrap.gpw == 2 and driver != "perstep":
        # every warp with two envs had steps on which one env's scenario_event ran and the other's did not
        assert wrap.mixed_pairs >= N // 2, wrap.mixed_pairs
    if driver in ("runaway", "bezier"):
        assert cnt["done"] >= N                                         # every env ended its moved episode and was reset


# ------------------------------------------------------------------------------------------------------------------
# bitwise: the launch shape and the reset-first scheduling are not part of the result
# ------------------------------------------------------------------------------------------------------------------
def fast_timers_on(pair):
    """The fast timers of test_gpu_scenarios on identical handles: one rewritten row goes to both."""
    row = pair[0].get_state(("scenario",))["scenario"]
    if fast_timers(row):
        for s in pair:
            s.set_state(scenario=row)


BLOCK_CASES = {"mix_k12": dict(num_agents=12), "mix_k27_dw": dict(num_agents=27, use_downwash=True)}


@pytest.mark.parametrize("name", list(BLOCK_CASES))
def test_scenario_events_block_64_and_128_are_bitwise_identical(name, monkeypatch):
    """test_gpu_parity.test_block_64_and_128_are_bitwise_identical for the formation variants at 16 and 32 lanes, with the timer
    events firing every 5..11 steps: every output and the whole state (goals, scenario rows) compared after every step."""
    cfg = QuadSimConfig(seed=23, num_envs=301, quads_mode="mix", ep_time=0.3, **BLOCK_CASES[name])
    sims = []
    for blk in ("64", "128"):
        monkeypatch.setenv("QS_BLOCK", blk)
        sims.append(_sim(cfg))
    monkeypatch.delenv("QS_BLOCK")
    a_sim, b_sim = sims
    assert torch.equal(a_sim.reset(), b_sim.reset())
    rs = np.random.RandomState(6)
    n_events = 0
    for s in range(40):
        fast_timers_on(sims)
        st = a_sim.get_state(("tick", "scenario"))
        ctl, t1 = st["scenario"][:, SC_CTL].long(), st["tick"].long() + 1
        n_events += int(((ctl > 0) & (ctl <= 50) & (t1 % ctl.clamp(min=1) == 0)).sum())
        a = torch.from_numpy(action_batch(rs, cfg.num_envs * cfg.num_agents, "uniform" if s % 2 else "hover")).cuda()
        o1, r1, d1 = (x.clone() for x in a_sim.step(a))
        o2, r2, d2 = b_sim.step(a)
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2), f"step {s}"
        assert torch.equal(a_sim.terminal_obs, b_sim.terminal_obs), f"step {s}"
        assert_handles_equal(a_sim, b_sim, f"step {s}")
    assert n_events >= cfg.num_envs


HOT_SCENARIO_CASES = {"mix_k12": dict(num_agents=12, quads_mode="mix"), "swarm_k15": dict(num_agents=15, quads_mode="swarm_vs_swarm")}


@pytest.mark.parametrize("name", list(HOT_SCENARIO_CASES))
def test_scenario_events_reset_first_scheduling_is_bitwise_invisible(name, monkeypatch):
    """QS_HOT=0 against the default handle (test_gpu_staggered.test_reset_first_scheduling_is_bitwise_invisible) at 16 lanes, with
    fast timers and staggered clocks: goal events, episode ends and resets on different steps in the two envs of a warp, a few
    dozen listed warp-tiles per step and then more than the hot list holds."""
    cfg = QuadSimConfig(seed=53, num_envs=8192, ep_time=0.4, **HOT_SCENARIO_CASES[name])
    N, K, L, gpw = cfg.num_envs, cfg.num_agents, cfg.ep_len, envs_per_tile(cfg.num_agents)
    monkeypatch.setenv("QS_HOT", "0")
    plain = _sim(cfg)
    monkeypatch.delenv("QS_HOT")
    hot = _sim(cfg)
    pair = (plain, hot)
    rs = np.random.RandomState(8)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(9)
    o1, o2 = plain.reset().clone(), hot.reset()
    assert_bitwise(o1, o2, "reset obs")

    def set_ticks(t):
        for s in pair:
            s.set_state(tick=np.asarray(t, np.int32))
        assert_handles_equal(plain, hot, "set_state(tick)")

    listed = []                                 # per step: warp-tiles with an env that ends in it

    def device_steps(n):
        for i in range(n):
            fast_timers_on(pair)
            end = plain.get_state(("tick",))["tick"].cpu().numpy() + 1 > L
            listed.append(int(tile_counts(end, gpw)[0].sum()))
            a = torch.rand((N * K, 4), device="cuda", generator=gen) * 2.0 - 1.0
            (o1, r1, d1), (o2, r2, d2) = (tuple(x.clone() for x in s.step(a)) for s in pair)
            assert_bitwise(o1, o2, "obs"); assert_bitwise(r1, r2, "rew"); assert_bitwise(d1, d2, "done")
            assert_bitwise(plain.terminal_obs, hot.terminal_obs, "terminal_obs")
            assert_bitwise(plain.reset_success, hot.reset_success, "reset_success")
            assert_handles_equal(plain, hot, f"device step {i}")

    t = rs.randint(0, L - 24, N)                                        # under the cap: ~30 warp-tiles end per step
    for j in range(14):
        for w in rs.choice(-(-N // gpw), 30, replace=False):
            t[min(N - 1, w * gpw + rs.randint(gpw))] = L - j
    set_ticks(t)
    device_steps(16)
    set_ticks(rs.randint(0, L, N))                                      # over the cap
    device_steps(12)
    print(f"[hot_{name}] warp-tiles with an ending env per step: {listed}")
    assert max(listed) > HOT_CAP and any(0 < n <= HOT_CAP for n in listed), listed
    assert plain.episode_stats()["episodes"] > N // 4
