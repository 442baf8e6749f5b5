"""The step kernel in steady state: staggered episode clocks, as bench.py's make() sets them.

In the upstream modes an episode ends on its clock only (tick > ep_len).  When every env starts from one reset(), every env of a
warp-tile ends on the same step, and the divergent part of the step kernel -- one lane group resetting (obstacle map, scenario
draw, spawn) while the other groups of its warp have finished their step, the terminal-observation copy selected by the done
ballot, the per-episode records, and the reset-first scheduling (QS_HOT, DESIGN.md) in the regime where a few dozen tiles are
listed per step -- never runs with a mix of ending and continuing envs.  This file staggers the clocks with set_state(tick=...):
  A. oracle parity of every feature instantiation and lane-group width, with deterministic tick patterns inside warp-tiles;
  B. the same at the benchmark's launch shapes, on whole sampled warp-tiles, over and under the 128-tile cap of the hot list;
  C. reset-first scheduling is bitwise invisible: QS_HOT=0 against the default, with host steps, masked and full resets and
     clock jumps between the device steps.
"""
import dataclasses

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from oracle import OracleEnv  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402
from test_gpu_parity import WIDTH_CELLS, SubsetSim, _sim, run_parity  # noqa: E402

OBST = dict(use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor")
HOT_CAP = 128                       # listed warp-tiles per step (qs_create: e->hot_cap)


def envs_per_tile(K):
    return 32 // (1 << (K - 1).bit_length())


def unit_size(K):
    """Envs that run side by side: the warp-tile, or for one env per warp (K > 16) the two warps of a 64-thread block."""
    return max(envs_per_tile(K), 2)


def tile_counts(ending, unit):
    """(units with an ending env, units with some but not all of their valid envs ending) of a bool vector over envs."""
    n = len(ending)
    pad = -n % unit
    e = np.concatenate([ending, np.zeros(pad, bool)]).reshape(-1, unit)
    v = np.concatenate([np.ones(n, bool), np.zeros(pad, bool)]).reshape(-1, unit)
    ne, nv = e.sum(axis=1), v.sum(axis=1)
    return (ne > 0), (ne > 0) & (ne < nv)


class CheckedSim(SubsetSim):
    """SubsetSim (the compared envs of a batch behind QuadSwarmSim's interface) whose step() also checks, over the WHOLE batch:
      1. rows of terminal_obs of envs that did not end still hold the NaN written before the step, and no row of an env that
         ended does;
      2. episode records of envs that did not end are bitwise unchanged, those of envs that ended advanced their sequence number
         by one; reset_success (filled with a canary byte before the step) reads 0 for envs that ended (upstream reset() reports
         no success) and the canary elsewhere;
      3. done == (tick before the step + 1 > ep_len), the only way an upstream episode ends short of a non-finite state
         (`ended()`; the fork env overrides it with its own rule).
    It counts the mixed units (some but not all valid envs of a warp-tile end on a step) among the compared envs, and per step the
    warp-tiles of the whole batch with an ending env (what the reset-first scheduling lists).

    Records: the kernel fills the 5-sample distance ring and the distance windows by the episode clock (`tick >= 5`, windows of
    the last 100/300/500 ticks divided by min(n, tick)); the oracle by its own count of steps since its reset.  The two agree for
    every episode that starts at tick 0, i.e. every episode started by a reset -- but not for an episode whose clock was moved by
    set_state(tick=...), whose first steps were never run.  `comparable()` excludes exactly those shortened first episodes."""

    CANARY = 0x5A

    def __init__(self, sim, env_idx, seed=0):
        super().__init__(sim, env_idx, seed)
        self.ep_len = sim.cfg.to_c().ep_len
        self.unit, self.gpw = unit_size(self.K), envs_per_tile(self.K)
        self.idx_np = np.asarray(env_idx)
        self.units = np.unique(self.idx_np // self.unit)
        self.mixed, self.ending_tiles, self.first_records = 0, [], 0
        self.first_ep = np.zeros(sim.N, bool)
        self._comparable = np.ones(len(self.idx_np), bool)

    def set_ticks(self, ticks):
        ticks = np.asarray(ticks, dtype=np.int32)
        self.sim.set_state(tick=ticks)
        self.first_ep |= ticks != 0

    def comparable(self):
        return self._comparable

    def ended(self, tick0, rec1):
        """The envs that ended in the step just taken [N] bool, after checking the done mask and reset_success of the ended envs
        against the rule that ends an episode."""
        sim, N, K = self.sim, self.sim.N, self.K
        end = tick0 + 1 > self.ep_len
        assert torch.equal(sim.done.view(N, K), end[:, None].expand(N, K)), "done differs from the episode clocks"
        assert bool((sim.reset_success[end] == 0).all()), "reset_success"
        return end

    def step(self, a_small):
        sim, N, K = self.sim, self.sim.N, self.K
        tick0 = sim.get_state(("tick",))["tick"]
        rec0 = sim.episode_records()
        sim.terminal_obs.fill_(float("nan"))
        sim.reset_success.fill_(self.CANARY)
        out = super().step(a_small)
        rec1 = sim.episode_records()
        end = self.ended(tick0, rec1)
        keep = ~end
        keep_rows = keep.repeat_interleave(K)
        assert bool(torch.isnan(sim.terminal_obs[keep_rows]).all()), "terminal_obs written for an env that did not end"
        assert not bool(torch.isnan(sim.terminal_obs[~keep_rows]).any()), "terminal_obs incomplete for an env that ended"
        assert bool((sim.reset_success[keep] == self.CANARY).all()), "reset_success written for an env that did not end"
        assert torch.equal(rec1["env"][keep], rec0["env"][keep]), "episode record of an env that did not end changed"
        assert torch.equal(rec1["agent"][keep_rows].view(torch.int32), rec0["agent"][keep_rows].view(torch.int32)), \
            "per-drone episode record of an env that did not end changed"
        assert torch.equal(rec1["env"][end, 0], rec0["env"][end, 0] + 1), "episode sequence number of an env that ended"
        e = end.cpu().numpy()
        self.mixed += int(tile_counts(e, self.unit)[1][self.units].sum())
        self.ending_tiles.append(int(tile_counts(e, self.gpw)[0].sum()))
        self._comparable = ~self.first_ep[self.idx_np]
        self.first_records += int((e & self.first_ep)[self.idx_np].sum())
        self.first_ep &= ~e
        return out


def staggered_ticks(N, unit, L, rs):
    """Deterministic clock patterns per unit (ticks 0..L; tick t ends on step L - t), cycling over:
    one env apart from the others (exactly one ends, then all but one), first and last env apart, envs ending on consecutive
    steps, random ticks, and a synchronized unit.  The last (partial) unit always gets the first/last pattern."""
    t = np.zeros(N, np.int32)
    n_units = -(-N // unit)
    for u in range(n_units):
        lo, hi = u * unit, min(N, (u + 1) * unit)
        n = hi - lo
        kind = "first_last" if u == n_units - 1 else ("one", "first_last", "consecutive", "random", "sync")[u % 5]
        if kind == "one":
            t[lo:hi] = 0
            t[lo + u % n] = L - 3
        elif kind == "first_last":
            t[lo:hi] = L - 9
            t[lo] = t[hi - 1] = L - 1
        elif kind == "consecutive":
            t[lo:hi] = (L - 4 - np.arange(n)) % (L + 1)
        elif kind == "random":
            t[lo:hi] = rs.randint(0, L + 1, n)
        else:
            t[lo:hi] = L - 6
    return t


def oracle_stats(oracles):
    tot = {}
    for o in oracles:
        for k, v in o.stats().items():
            tot[k] = tot.get(k, 0) + v
    return tot


# name: (config kwargs, envs, action kind).  ep_time 0.2 s = 20 control steps; envs chosen so that the last warp-tile is partial.
STAGGER = {
    "feat0_k8": (dict(num_agents=8), 27, "uniform"),
    "feat1_obst_k6": (dict(num_agents=6, quads_mode="o_random", neighbor_visible_num=3, **OBST), 27, "hover"),
    "feat2_downwash_k8": (dict(num_agents=8, use_downwash=True), 27, "uniform"),
    # obstacle reset on its shared-memory fast path: the group's tile rows hold 8 x 40 floats >= obst_scratch_floats(12, 8) = 100
    "feat3_obst_downwash_k8": (dict(num_agents=8, quads_mode="mix", use_downwash=True, neighbor_visible_num=2, **OBST), 27, "hover"),
    "feat4_mix_k8": (dict(num_agents=8, quads_mode="mix"), 27, "hover"),
    "feat4_mix_k1": (dict(num_agents=1, quads_mode="mix", neighbor_obs_type="none", neighbor_visible_num=0), 167, "hover"),
    "feat6_mix_downwash_k8": (dict(num_agents=8, quads_mode="mix", use_downwash=True), 27, "hover"),
    "feat0_k3": (dict(num_agents=3, neighbor_visible_num=1), 53, "uniform"),
    "feat0_k16": (dict(num_agents=16), 13, "uniform"),
    "feat0_k32": (dict(num_agents=32), 9, "uniform"),
    # ... and on its sequential fallback: one drone's tile row is 28 floats < obst_scratch_floats(12, 1) = 84
    "feat1_obst_k1_fallback": (dict(num_agents=1, quads_mode="mix", neighbor_obs_type="none", neighbor_visible_num=0, **OBST), 137, "hover"),
    **WIDTH_CELLS,                      # every feature variant at the widths 2, 4, 16 and 32 (test_gpu_parity.py)
}


@pytest.mark.parametrize("name", list(STAGGER))
def test_staggered_parity(name):
    """Every env ends its (shortened) first episode at its own step and then a full one; the oracle checks every step and every
    full episode's record, the wrapper the rows of the envs that went on; the summed episode statistics of the full episodes
    agree with the oracle's."""
    kw, n_envs, kind = STAGGER[name]
    cfg = QuadSimConfig(seed=29, num_envs=n_envs, ep_time=0.2, **kw)
    L, K, N = cfg.to_c().ep_len, cfg.num_agents, n_envs
    steps = 2 * L + 6                           # every env ends its first episode by step L and its second by step 2 L + 1
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(N)]
    sim.reset()
    for o in oracles:
        o.reset()                               # same draws as the GPU reset (the formation scenarios' first episode)
    wrap = CheckedSim(sim, np.arange(N), seed=1)
    wrap.set_ticks(staggered_ticks(N, wrap.unit, L, np.random.RandomState(7)))
    snap = {}

    def hook(s):
        if s == L + 1:                          # every shortened first episode has ended: count the full episodes from here
            sim.episode_stats(reset=True)
            snap.update(oracle_stats(oracles))

    worst, cnt = run_parity("stagger_" + name, cfg, wrap, oracles, kind, steps, hook, record_envs=wrap.comparable)
    n_units = -(-N // wrap.unit)
    print(f"[stagger_{name}] mixed units {wrap.mixed} over {n_units} units, shortened first-episode records skipped "
          f"{wrap.first_records}, records compared {cnt.get('records', 0)}")
    assert wrap.mixed >= n_units, "the tick patterns no longer give warp-tiles with ending and continuing envs"
    assert cnt["done"] >= 2 * N and cnt.get("records", 0) >= N // 2
    gs, ref = sim.episode_stats(), oracle_stats(oracles)
    ref = {k: v - snap[k] for k, v in ref.items()}
    assert gs["episodes"] == ref["episodes"] >= N, (gs["episodes"], ref["episodes"])
    for k in ("num_collisions", "num_collisions_with_floor", "num_collisions_with_wall", "num_collisions_with_ceiling",
              "num_collisions_with_room", "num_collisions_after_settle", "num_collisions_obst_quad"):
        assert abs(gs[k] - ref[k]) <= max(2, 0.02 * ref[k]), (k, gs[k], ref[k])
    for k in ("distance_to_goal_1s", "distance_to_goal_3s", "distance_to_goal_5s"):
        assert abs(gs[k] - ref[k]) <= 1e-3 * abs(ref[k]), (k, gs[k], ref[k])
    assert gs["agents_success"] + gs["agents_deadlock"] + gs["agents_collided"] == gs["episodes"] * K
    assert gs["nonfinite_resets"] == 0


# ------------------------------------------------------------------------------------------------------------------
# B. the benchmark's launch shapes (128-thread blocks, full grids), whole sampled warp-tiles
# ------------------------------------------------------------------------------------------------------------------
CFG3 = dict(num_agents=8, quads_mode="mix", use_downwash=True, neighbor_visible_num=2, **OBST)
BIG = {
    # name: (config kwargs, envs, action kind, regime)
    "cfg2_65536x8": (dict(num_agents=8), 65536, "uniform", "over"),
    "cfg3_65536x8_over": (CFG3, 65536, "hover", "over"),
    "cfg3_65536x8_under": (CFG3, 65536, "hover", "under"),
    "mix_65536x8_over": (dict(num_agents=8, quads_mode="mix"), 65536, "hover", "over"),
    "mix_65536x8_under": (dict(num_agents=8, quads_mode="mix"), 65536, "hover", "under"),
    "cfg4_16384x32": (dict(num_agents=32), 16384, "uniform", "over"),
}
BIG_STEPS = 32


def undercap_ticks(N, gpw, L, steps, tiles, rs, per_step=30):
    """Most envs far from their end for the whole window; one env of each compared tile ends, at a step of its own; `per_step`
    further tiles get one env that ends on each step -- a few dozen listed tiles per step, as in bench's steady state."""
    t = rs.randint(0, L - steps - 1, N).astype(np.int32)
    for i, w in enumerate(tiles):
        n = min(gpw, N - w * gpw)
        t[w * gpw + i % n] = L - i % steps
    others = np.setdiff1d(np.arange(-(-N // gpw)), tiles)
    for j in range(steps):
        for w in rs.choice(others, per_step, replace=False):
            t[w * gpw + rs.randint(min(gpw, N - w * gpw))] = L - j
    return t


@pytest.mark.parametrize("name", list(BIG))
def test_staggered_parity_at_benchmarked_launch_shape(name, monkeypatch):
    kw, n_envs, kind, regime = BIG[name]
    ep_time = 0.2 if regime == "over" else 2.0          # 20 control steps; 200 for the clocks far from their end
    cfg = QuadSimConfig(seed=41, num_envs=n_envs, ep_time=ep_time, **kw)
    L, K, gpw = cfg.to_c().ep_len, cfg.num_agents, envs_per_tile(cfg.num_agents)
    monkeypatch.setenv("QS_BLOCK", "128")
    sim = _sim(cfg)
    monkeypatch.delenv("QS_BLOCK")
    n_tiles = -(-n_envs // gpw)
    rs = np.random.RandomState(3)
    tiles = np.sort(rs.choice(np.arange(1, n_tiles - 1), 256 // max(gpw, 4) - 2, replace=False))
    tiles = np.concatenate([[0], tiles, [n_tiles - 1]])                 # first and last warp-tile of the grid
    idx = (tiles[:, None] * gpw + np.arange(gpw)[None, :]).reshape(-1)
    idx = idx[idx < n_envs]
    oracles = [OracleEnv(cfg, int(i)) for i in idx]
    sim.reset()
    for o in oracles:
        o.reset()
    wrap = CheckedSim(sim, idx, seed=5)
    if regime == "over":                                                # uniform over [0, ep_len), as bench.py's make()
        gen = torch.Generator(device=sim.device)
        gen.manual_seed(1234)
        wrap.set_ticks(torch.randint(0, L, (n_envs,), generator=gen, device=sim.device, dtype=torch.int32).cpu().numpy())
    else:
        wrap.set_ticks(undercap_ticks(n_envs, gpw, L, BIG_STEPS, tiles, rs))
    small = dataclasses.replace(cfg, num_envs=len(idx))
    worst, cnt = run_parity("stagger_" + name, small, wrap, oracles, kind, BIG_STEPS, record_envs=wrap.comparable)
    lt = np.array(wrap.ending_tiles)
    print(f"[stagger_{name}] mixed tiles {wrap.mixed} over {len(tiles)} compared tiles; warp-tiles with an ending env per step: "
          f"min {lt.min()} median {int(np.median(lt))} max {lt.max()}; records compared {cnt.get('records', 0)}")
    assert wrap.mixed >= len(tiles) // (2 if gpw == 1 else 1)
    if regime == "over":
        assert cnt["done"] >= len(idx)
        if gpw > 1:
            # more than the hot list holds on every step but two: clocks drawn from [0, ep_len) leave no env ending on step 0,
            # and so none on step ep_len + 1
            assert (lt > HOT_CAP).sum() >= BIG_STEPS - 2, lt
    else:
        assert 8 <= lt.min() and lt.max() <= HOT_CAP, lt               # a few dozen per step, all of them listed


# ------------------------------------------------------------------------------------------------------------------
# C. reset-first scheduling is bitwise invisible
# ------------------------------------------------------------------------------------------------------------------
def bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def assert_bitwise(a, b, what):
    assert a.shape == b.shape and torch.equal(bits(a), bits(b)), what


def assert_handles_equal(a, b, what):
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert_bitwise(sa[k], sb[k], f"{what}: state {k}")
    ra, rb = a.episode_records(), b.episode_records()
    for k in ra:
        assert_bitwise(ra[k], rb[k], f"{what}: episode records {k}")
    ga, gb = a.episode_stats(), b.episode_stats()
    for k in ga:
        if isinstance(ga[k], float):
            # double atomicAdd sums: the hot blocks change the ORDER in which the episodes' terms arrive, which moves the last
            # bits; the terms themselves are the per-drone records compared bitwise above
            assert abs(ga[k] - gb[k]) <= 1e-12 * max(1.0, abs(ga[k])), (what, k, ga[k], gb[k])
        else:
            assert ga[k] == gb[k], (what, k, ga[k], gb[k])


HOT_CASES = {
    # name: (config kwargs, envs, QS_BLOCK).  feat 1 / 3 take the flag through shared memory (no prefetch, PFM == 0), feat 4 / 6
    # with the prefetched prologue; 64-thread blocks give 64 hot blocks, 128-thread blocks 32.
    "feat1_k8_b64": (dict(num_agents=8, quads_mode="o_random", neighbor_visible_num=2, **OBST), 8192, 64),
    "feat1_k3_b128": (dict(num_agents=3, quads_mode="o_random", neighbor_visible_num=1, **OBST), 8192, 128),
    "feat3_k8_b128": (CFG3, 8192, 128),
    "feat3_k1_b64": (dict(num_agents=1, quads_mode="mix", use_downwash=True, neighbor_obs_type="none", neighbor_visible_num=0, **OBST),
                     16384, 64),
    "feat4_k8_b64": (dict(num_agents=8, quads_mode="mix"), 8192, 64),
    "feat4_k16_b128": (dict(num_agents=16, quads_mode="mix"), 8192, 128),
    "feat4_k1_b128": (dict(num_agents=1, quads_mode="mix", neighbor_obs_type="none", neighbor_visible_num=0), 16384, 128),
    "feat6_k8_b128": (dict(num_agents=8, quads_mode="mix", use_downwash=True), 8192, 128),
    "feat6_k3_b64": (dict(num_agents=3, quads_mode="mix", use_downwash=True, neighbor_visible_num=1), 8192, 64),
    "feat4_k32_compiled_out": (dict(num_agents=32, quads_mode="mix"), 2048, 128),
}


@pytest.mark.parametrize("name", list(HOT_CASES))
def test_reset_first_scheduling_is_bitwise_invisible(name, monkeypatch):
    """Two handles, QS_HOT=0 and the default, same actions and clocks; every output and the whole state compared bitwise after
    every call.  Between the device steps: a chunked host step (lists off, hot_phase not advanced), a masked reset, clock jumps
    into and out of the next step's end, over-cap clocks, a full reset followed by steps in which no env ends."""
    kw, n_envs, block = HOT_CASES[name]
    cfg = QuadSimConfig(seed=53, num_envs=n_envs, ep_time=0.4, **kw)
    L, N, K, gpw = cfg.to_c().ep_len, n_envs, cfg.num_agents, envs_per_tile(cfg.num_agents)
    monkeypatch.setenv("QS_BLOCK", str(block))
    monkeypatch.setenv("QS_HOT", "0")
    plain = _sim(cfg)
    monkeypatch.delenv("QS_HOT")
    hot = _sim(cfg)
    monkeypatch.delenv("QS_BLOCK")
    pair = (plain, hot)
    rs = np.random.RandomState(8)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(9)
    listed = []                                # per device step: warp-tiles with an env that ends in it

    def both(fn, what):
        outs = [fn(s) for s in pair]
        assert_handles_equal(plain, hot, what)
        return outs

    def set_ticks(t):
        both(lambda s: s.set_state(tick=np.asarray(t, np.int32)), "set_state(tick)")

    def ticks():
        return plain.get_state(("tick",))["tick"].cpu().numpy()

    def device_steps(n):
        for _ in range(n):
            end = ticks() + 1 > L
            listed.append(int(tile_counts(end, gpw)[0].sum()))
            a = torch.rand((N * K, 4), device="cuda", generator=gen) * 2.0 - 1.0
            (o1, r1, d1), (o2, r2, d2) = both(lambda s: tuple(x.clone() for x in s.step(a)), f"device step {len(listed)}")
            assert_bitwise(o1, o2, "obs"); assert_bitwise(r1, r2, "rew"); assert_bitwise(d1, d2, "done")
            assert_bitwise(plain.terminal_obs, hot.terminal_obs, "terminal_obs")
            assert_bitwise(plain.reset_success, hot.reset_success, "reset_success")

    def undercap():
        t = rs.randint(0, L - 24, N)
        for j in range(14):
            for w in rs.choice(-(-N // gpw), 30, replace=False):
                t[min(N - 1, w * gpw + rs.randint(gpw))] = L - j
        return t

    o1, o2 = both(lambda s: s.reset().clone(), "reset")
    assert_bitwise(o1, o2, "reset obs")
    set_ticks(undercap())
    device_steps(6)
    monkeypatch.setenv("QS_HOST_CHUNKS", "3")
    a = (torch.rand((N * K, 4), device="cuda", generator=gen) * 2.0 - 1.0).cpu().numpy()
    host = []
    for s in pair:
        term, succ = np.full((N * K, cfg.obs_dim), np.nan, np.float32), np.full(N, 0x5A, np.uint8)
        host.append(tuple(x.copy() for x in s.step_host(a, terminal_obs=term, reset_success=succ)) + (term, succ))
    monkeypatch.delenv("QS_HOST_CHUNKS")
    for x, y in zip(*host):
        assert np.array_equal(x.view(np.int32) if x.dtype == np.float32 else x, y.view(np.int32) if y.dtype == np.float32 else y)
    assert host[0][2].any(), "no env ended in the host step"
    assert_handles_equal(plain, hot, "chunked host step")
    device_steps(3)
    t = ticks()
    mask = torch.from_numpy((rs.rand(N) < 0.1) | ((t == L) & (rs.rand(N) < 0.5)))
    o1, o2 = both(lambda s: s.reset(mask).clone(), "masked reset")
    assert_bitwise(o1, o2, "masked reset obs")
    device_steps(2)
    t = ticks()
    going = np.flatnonzero(t == L)
    t[going[: len(going) // 2]] = 0                                     # out of the next step's end (their tiles are listed)
    t[rs.choice(np.flatnonzero(t < L - 10), 40, replace=False)] = L     # into it (their tiles are not)
    set_ticks(t)
    device_steps(3)
    set_ticks(rs.randint(0, L, N))                                      # over the cap
    device_steps(6)
    o1, o2 = both(lambda s: s.reset().clone(), "full reset")
    assert_bitwise(o1, o2, "full reset obs")
    device_steps(4)                                                     # nothing ends: empty lists are consumed
    set_ticks(undercap())
    device_steps(4)
    print(f"[hot_{name}] warp-tiles with an ending env per device step: {listed}")
    if gpw > 1:
        assert max(listed) > HOT_CAP and any(0 < n <= HOT_CAP for n in listed)
        assert any(listed[i] == listed[i + 1] == 0 for i in range(len(listed) - 1))
    assert plain.episode_stats()["episodes"] > N // 10
