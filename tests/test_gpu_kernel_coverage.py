"""Every compiled program of the simulator is compared with the oracle by some case.

kernels_kg.cu builds the step, reset and fork kernels once per lane-group width KG (the lanes of one env), and the upstream step
kernel once more per feature set; group_obs_tail<KG, OBST> picks one of four neighbour-selection paths from (KG, obstacles, V), and
fork_neighbor_obs<KG> ranks the neighbours or takes all of them in index order.  Each combination is its own code, so a table of
oracle-compared cases can leave one of them untested without any test failing.  This test maps every case of those tables to the
program it runs and fails when a reachable program has no case -- when a case is removed, or when the width rule or the selection
branches change without the tables following.
"""
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from quad_swarm_rl_stable_baselines3_b200.config import SCENARIOS, QuadSimConfig, cube_floor_dim  # noqa: E402
from test_gpu_fork import FORK_CONFIGS  # noqa: E402
from test_gpu_parity import CONFIGS  # noqa: E402
from test_gpu_scenario_widths import SCENARIO_WIDTH_CASES  # noqa: E402
from test_gpu_scenarios import SCENARIO_CONFIGS  # noqa: E402
from test_gpu_staggered import STAGGER  # noqa: E402


def lane_group(K):
    """qs_create (quadsim.cu): e->KG = pow2_at_least(K)."""
    return 1 << (K - 1).bit_length()


def feature_set(K, obst, downwash, scen):
    """qs_create (quadsim.cu): feat = obstacles | downwash (K > 1) << 1 | formation scenario (never with obstacles) << 2."""
    return int(obst) | (2 if downwash and K > 1 else 0) | (4 if scen and not obst else 0)


def selection_path(K, V, obst):
    """group_obs_tail (quadsim_kernels.cuh), position/velocity neighbour rows with KG > 1: the branch that orders them."""
    KG = lane_group(K)
    if KG == 1 or V == 0:
        return None
    if V >= K - 1:
        return "all in index order"
    if (KG >= 16 or (obst and KG >= 4)) and 3 * V < 2 * (KG - 1):
        return "first minimum"
    if KG <= 8:
        return "packed rank count"
    return "all-pairs rank count"


def fork_path(K, V):
    """fork_neighbor_obs (fork_kernels.cuh): no rows for KG == 1 or V == 0, ranked rows for V < K - 1."""
    if lane_group(K) == 1 or V == 0:
        return None
    return "ranked" if V < K - 1 else "all in index order"


def program(cfg):
    """(KG, FEAT or "fork", neighbour-selection path, obstacles) of the kernels a config runs."""
    K = cfg.num_agents
    if cfg.env_mode == "fork":
        return lane_group(K), "fork", fork_path(K, cfg.visible), False
    scen = cfg.scenario_id() != SCENARIOS["static_same_goal"]
    path = selection_path(K, cfg.visible, cfg.use_obstacles) if cfg.neighbor_obs_type == "pos_vel" else None
    return lane_group(K), feature_set(K, cfg.use_obstacles, cfg.use_downwash, scen), path, cfg.use_obstacles


def covered():
    cfgs = [QuadSimConfig(**kw) for kw in CONFIGS.values()]
    cfgs += [QuadSimConfig(**kw) for kw, _, _ in STAGGER.values()]
    cfgs += [QuadSimConfig(**kw) for kw, _, _ in SCENARIO_CONFIGS.values()]
    cfgs += [QuadSimConfig.fork_default(**kw) for kw in FORK_CONFIGS.values()]
    return {program(c) for c in cfgs}


def test_every_kernel_instantiation_and_selection_path_is_oracle_compared():
    progs = covered()
    cells = {(kg, f) for kg, f, _, _ in progs}
    paths = {(kg, f == "fork", p, obst) for kg, f, p, obst in progs if p is not None}
    want_cells, want_paths = set(), set()
    for K in range(1, 33):
        KG = lane_group(K)
        want_cells.add((KG, "fork"))
        for V in range(K):
            if fork_path(K, V) is not None:
                want_paths.add((KG, True, fork_path(K, V), False))
        for obst in (False, True):
            for downwash in (False, True):
                for scen in (False, True):
                    if not (obst and scen):
                        want_cells.add((KG, feature_set(K, obst, downwash, scen)))
            for V in range(K):
                if selection_path(K, V, obst) is not None:
                    want_paths.add((KG, False, selection_path(K, V, obst), obst))
    assert len(want_cells) == 3 + 5 * 6 + 6          # KG = 1: feat 0, 1, 4; KG >= 2: all six; the fork kernel at every width
    assert not want_cells - cells, f"kernel instantiations no oracle-compared case runs: {sorted(want_cells - cells, key=str)}"
    # (KG, fork kernel, path, obstacles): group_obs_tail is instantiated apart for the obstacle variants
    assert not want_paths - paths, f"neighbour-selection paths no oracle-compared case reaches: {sorted(want_paths - paths, key=str)}"


EVENT_SCENARIOS = ("dynamic_same_goal", "dynamic_diff_goal", "swap_goals", "swarm_vs_swarm", "run_away", "dynamic_formations",
                   "ep_lissajous3D", "ep_rand_bezier", "mix")


def min_agents(mode):
    """QuadSimConfig.scenario_id (config.py): swap_goals and mix (which draws swap_goals) need K >= 3 on the device,
    swarm_vs_swarm and run_away K >= 2; dynamic_* take two halves / a formation of K >= 2 rows in the reference."""
    return 3 if mode in ("swap_goals", "mix") else (1 if mode in ("ep_lissajous3D", "ep_rand_bezier") else 2)


def event_edges(mode, K):
    """The K-dependent paths of a mode's goal-changing code (scenario_event and formation_scenario_step, scenario_kernels.cuh).
    formation_goal: circles stack layers of 8 (whole = n / 8 layers of 8, then one of n % 8), grid_dims(n) of a prime n is 1 x n,
    the sphere has max(n, 3) rows; swarm_vs_swarm builds its halves of K / 2 and K - K / 2 drones (swarm_goal: rows1 from the
    first) with cube floor dims cube_dim[1] and [2]; scen_shuffle_perm draws four uniforms per rng_u4, so more than 9 rows take
    more than two draws; swap_goals, run_away and dynamic_diff_goal index their group's lanes of the exchange buffer or the
    permutation, with KG - K padding lanes."""
    halves = [K // 2, K - K // 2]
    formed = {"dynamic_same_goal": [K], "dynamic_diff_goal": [K], "dynamic_formations": [K], "swarm_vs_swarm": halves}.get(mode, [])
    shuffled = {"dynamic_diff_goal": [K], "swap_goals": [K], "swarm_vs_swarm": halves}.get(mode, [])
    edges = set()
    circle = "circle of a swarm half" if mode == "swarm_vs_swarm" else "circle"
    for n in formed:
        if n > 8:
            edges.add(f"{circle}: a partial top layer" if n % 8 else f"{circle}: whole layers only")
        if n > 16:
            edges.add(f"{circle}: three or more layers")
        if n > 3 and all(n % a for a in range(2, n)):
            edges.add("grid: 1 x n for a prime n")
        if n < 3:
            edges.add("sphere: 3 rows for fewer than 3 drones")
    if mode == "swarm_vs_swarm" and K % 2:
        edges.add("swarm: halves of different sizes")
    if mode == "swarm_vs_swarm" and cube_floor_dim(K // 2) != cube_floor_dim(K - K // 2):
        edges.add("swarm: halves of different cube floor dims")
    if max(shuffled, default=0) > 9:
        edges.add("shuffle: more than two draws")
    if mode in ("swap_goals", "run_away", "dynamic_diff_goal") and K > 8:
        edges.add(f"{mode}: padding lanes" if K < lane_group(K) else f"{mode}: no padding lanes")
    return edges


def event_cases():
    """(config, mode) of every oracle-compared case whose goal events run: test_gpu_scenarios.py's with fast timers, run_away
    with ep_time > 1 s (the events come every second), the per-step modes; every case of SCENARIO_WIDTH_CASES."""
    out = []
    for kw, _, fast_timer in SCENARIO_CONFIGS.values():
        mode = kw["quads_mode"]
        if fast_timer or mode in ("dynamic_formations", "ep_lissajous3D", "ep_rand_bezier") or (mode == "run_away" and kw["ep_time"] > 1.0):
            out.append((QuadSimConfig(**kw), mode))
    out += [(QuadSimConfig(num_envs=n, **kw), kw["quads_mode"]) for kw, n, _, _ in SCENARIO_WIDTH_CASES.values()]
    return out


def test_every_scenario_event_runs_at_every_width():
    """Every (KG, event mode) the config rules allow has a case whose events fire (KG = 1, where only mix_k1 runs, aside); at 16
    and 32 lanes each of the feature sets 4 (scenarios) and 6 (scenarios + downwash) runs at least four event modes, mix among
    them (the upstream training recipe); and every (KG, K-dependent path of the event code) reachable at 2, 16 or 32 lanes is
    reached."""
    have, feats, edges = set(), {}, set()
    for cfg, mode in event_cases():
        K = cfg.num_agents
        KG, feat = lane_group(K), program(cfg)[1]
        have.add((KG, mode))
        feats.setdefault((KG, feat), set()).add(mode)
        edges |= {(KG, e) for e in event_edges(mode, K)}
    want, want_edges = set(), set()
    for K in range(2, 33):
        for mode in EVENT_SCENARIOS:
            if K >= min_agents(mode):
                want.add((lane_group(K), mode))
                if lane_group(K) in (2, 16, 32):
                    want_edges |= {(lane_group(K), e) for e in event_edges(mode, K)}
    assert len(want) == 7 + 4 * 9
    assert not want - have, f"(lane group, mode) whose goal events no oracle-compared case runs: {sorted(want - have)}"
    for KG in (16, 32):
        for feat in (4, 6):
            modes = feats.get((KG, feat), set())
            assert len(modes) >= 4 and "mix" in modes, (KG, feat, sorted(modes))
    assert not want_edges - edges, f"K-dependent paths of the event code no case reaches: {sorted(want_edges - edges)}"
