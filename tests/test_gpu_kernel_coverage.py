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

from quad_swarm_rl_stable_baselines3_b200.config import SCENARIOS, QuadSimConfig  # noqa: E402
from test_gpu_fork import FORK_CONFIGS  # noqa: E402
from test_gpu_parity import CONFIGS  # noqa: E402
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
