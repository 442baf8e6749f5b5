"""GPU parity: the CUDA simulator (through the C-ABI) against the CPU oracle on identical seeds and actions.

Tolerances (BASELINE.json north_star): fp32 kernel vs float64 oracle, relative error <= 1e-5 on pos/vel/rot/omega after
one step; collision flags, neighbour choices and reset masks bit-exact away from threshold ties; drift over 100
free-running steps is reported and bounded.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import OracleEnv, philox  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.config import OBS_REPR_DIM, QuadSimConfig  # noqa: E402

REL_TOL = 1e-5          # north_star tolerance on pos/vel/rot/omega after one step
PHYS = ("pos", "vel", "rot", "omega", "rot_damp", "cmds_damp", "ou")

# "Bit-exact away from threshold ties" is PROVEN per event, not budgeted: the oracle records, for every threshold decision of a
# step, how far (float64) the decided quantity was from its threshold, in fp32 ulps of the operands' magnitude
# (OracleEnv.margins()).  A discrete disagreement (flag bit, collision row, spawn yaw, neighbour choice) is accepted only if a
# decision of a class that can produce it was within the bound below; anything else fails the test.
#   positions: two sub-steps of p += dt*v round by 0.5 ulp(p) each -> 1 ulp per coordinate; wall / ceiling / floor / obstacle
#   decisions see one drone (<= sqrt(2) ulp), pair distances two drones (<= 2 sqrt(3) = 3.5 ulp): bound 4.
#   lift-off of a resting drone compares thrust/m with g: four motors x (lag, approximate sqrt, clamp, polynomial) -> bound 32.
#   spawn yaw (cos t hx + sin t hy vs 0.5, approximate division + sincospi) and neighbour ranking (sum of six squares): bound 8.
TIE_ULPS = dict(pair=4.0, obst=4.0, floor=4.0, wall=4.0, ceil=4.0, liftoff=32.0, yaw=8.0, rank=8.0)
FLAG_CLASSES = ("pair", "obst", "floor", "wall", "ceil", "liftoff")


def tie_proven(oracle, classes):
    """(proved, margins): some decision of `classes` in the oracle's last step was within its ulp bound of the threshold."""
    m = oracle.margins()
    return any(m[c] <= TIE_ULPS[c] for c in classes), {c: float(m[c]) for c in classes}


def _sim(cfg):
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    return QuadSwarmSim(cfg, device="cuda:0")


def relerr(a, b, floor):
    """max |a-b| / max(|b|, floor) -- `floor` is the natural scale of the quantity (1 m, 1 m/s, ...)."""
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


CONFIGS = {
    "cfg2_k8": dict(num_envs=48, num_agents=8, ep_time=0.4),
    "cfg3_obst_k8": dict(num_envs=32, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                         obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, ep_time=0.4,
                         rew_coeff=dict(quadcol_bin_smooth_max=4.0)),
    "cfg4_k32": dict(num_envs=10, num_agents=32, ep_time=0.3),
    "smallroom_k8": dict(num_envs=32, num_agents=8, room_dims=(3.0, 3.0, 3.0), ep_time=0.5),
    "crowd_k16": dict(num_envs=12, num_agents=16, room_dims=(4.0, 4.0, 6.0), ep_time=0.5),
    "nonoise_wall_k4": dict(num_envs=33, num_agents=4, sense_noise=None, neighbor_visible_num=-1,
                            obs_repr="xyz_vxyz_R_omega_wall", ep_time=0.3),
    "single_k1": dict(num_envs=70, num_agents=1, neighbor_obs_type="none", neighbor_visible_num=0, ep_time=0.3),
    "odd_k3": dict(num_envs=21, num_agents=3, neighbor_visible_num=1, ep_time=0.3),
    "single_k1_obst": dict(num_envs=40, num_agents=1, quads_mode="mix", use_obstacles=True, neighbor_obs_type="none", neighbor_visible_num=0,
                           obs_repr="xyz_vxyz_R_omega_floor", ep_time=0.3),
    "odd_k6_obst": dict(num_envs=9, num_agents=6, quads_mode="o_random", use_obstacles=True, neighbor_visible_num=3,
                        obs_repr="xyz_vxyz_R_omega_floor", ep_time=0.3),
}

# Every feature variant of the step and reset kernels at the lane-group widths 2, 4, 16 and 32 (KG = the power of two >= K, the
# lanes of one env), with K below the width wherever it can be so that padding lanes exist, and the neighbour-selection paths of
# the obstacle variants that no other case reaches.  The path of group_obs_tail (quadsim_kernels.cuh) that each case reaches is
# noted with V: "first minimum" when (KG >= 16 or obstacles and KG >= 4) and 3 V < 2 (KG - 1); else the packed rank count for
# KG <= 8; else the all-pairs rank count; "all" when V = K - 1.
# Run by test_reset_parity (explicit and masked reset) here and test_staggered_parity (step) in test_gpu_staggered.py.
# name: (config kwargs, envs, action kind); the envs leave the last warp-tile partial.
_OBST = dict(use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor")
WIDTH_CELLS = {
    "feat0_k2": (dict(num_agents=2, neighbor_visible_num=1), 27, "uniform"),                                    # all
    "feat1_obst_k2": (dict(num_agents=2, quads_mode="o_random", neighbor_visible_num=1, **_OBST), 27, "hover"),  # all
    "feat2_downwash_k2": (dict(num_agents=2, use_downwash=True, neighbor_visible_num=1), 27, "uniform"),         # all
    "feat3_obst_downwash_k2": (dict(num_agents=2, quads_mode="mix", use_downwash=True, neighbor_visible_num=1, **_OBST), 27, "hover"),
    "feat6_runaway_downwash_k2": (dict(num_agents=2, quads_mode="run_away", use_downwash=True, neighbor_visible_num=1), 27, "hover"),
    "feat1_obst_k3_v1": (dict(num_agents=3, quads_mode="o_random", neighbor_visible_num=1, **_OBST), 21, "hover"),      # first minimum
    "feat2_downwash_k3": (dict(num_agents=3, use_downwash=True, neighbor_visible_num=1), 21, "uniform"),                # packed
    "feat3_obst_downwash_k3": (dict(num_agents=3, quads_mode="mix", use_downwash=True, neighbor_visible_num=2, **_OBST), 21, "hover"),
    "feat6_mix_downwash_k3": (dict(num_agents=3, quads_mode="mix", use_downwash=True, neighbor_visible_num=1), 21, "hover"),  # packed
    "feat0_k16_v12": (dict(num_agents=16, neighbor_visible_num=12), 13, "uniform"),                          # all-pairs: 36 >= 30
    "feat1_obst_k13_v10": (dict(num_agents=13, quads_mode="o_random", neighbor_visible_num=10, **_OBST), 13, "hover"),  # all-pairs: 30 >= 30
    "feat2_downwash_k12_vall": (dict(num_agents=12, use_downwash=True, neighbor_visible_num=-1), 13, "uniform"),         # all
    "feat3_obst_downwash_k13": (dict(num_agents=13, quads_mode="mix", use_downwash=True, **_OBST), 13, "hover"),        # first minimum
    "feat6_mix_downwash_k12": (dict(num_agents=12, quads_mode="mix", use_downwash=True), 13, "hover"),                 # first minimum
    "feat0_k29_v24": (dict(num_agents=29, neighbor_visible_num=24), 9, "uniform"),                           # all-pairs: 72 >= 62
    "feat1_obst_k27": (dict(num_agents=27, quads_mode="o_random", **_OBST), 9, "hover"),                               # first minimum
    "feat2_downwash_k27_vall": (dict(num_agents=27, use_downwash=True, neighbor_visible_num=-1), 9, "uniform"),         # all
    "feat3_obst_downwash_k29_v22": (dict(num_agents=29, quads_mode="mix", use_downwash=True, neighbor_visible_num=22, **_OBST), 9,
                                    "hover"),                                                                          # all-pairs: 66 >= 62
    "feat6_mix_downwash_k27": (dict(num_agents=27, quads_mode="mix", use_downwash=True), 9, "hover"),                  # first minimum
    "feat1_obst_k4_v2": (dict(num_agents=4, quads_mode="o_random", neighbor_visible_num=2, **_OBST), 21, "hover"),     # packed: 6 >= 6
    "feat1_obst_k7_v5": (dict(num_agents=7, quads_mode="o_random", neighbor_visible_num=5, **_OBST), 11, "hover"),     # packed: 15 >= 14
    "feat3_obst_downwash_k6_vall": (dict(num_agents=6, quads_mode="mix", use_downwash=True, neighbor_visible_num=-1, **_OBST), 11,
                                    "hover"),                                                                          # all
    "feat1_obst_k12_vall": (dict(num_agents=12, quads_mode="o_random", neighbor_visible_num=-1, **_OBST), 13, "hover"),  # all
    "feat1_obst_k29_vall": (dict(num_agents=29, quads_mode="o_random", neighbor_visible_num=-1, **_OBST), 9, "hover"),   # all
}
CONFIGS.update({name: dict(num_envs=n, ep_time=0.3, **kw) for name, (kw, n, _) in WIDTH_CELLS.items()})


def make_pair(name, seed=3):
    cfg = QuadSimConfig(seed=seed, **CONFIGS[name])
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(cfg.num_envs)]
    return cfg, sim, oracles


def push_state(sim, oracles, cfg):
    """Teacher forcing: copy the GPU state (fp32 values are exact in float64) into the oracle envs."""
    st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
    K = cfg.num_agents
    # a drone resting on the floor sits at z == fp32(arm) on the GPU and at z == arm (float64) in the oracle: the same
    # state in each one's own representation (fp32(arm) is 1.7e-9 m above arm, which the oracle would read as airborne)
    arm = cfg.to_c().arm
    resting = ((st["flags"] & 1) == 1) & (st["pos"][:, 2] == np.float32(arm))
    pos64 = st["pos"].astype(np.float64)
    pos64[resting, 2] = arm
    st = dict(st, pos64=pos64)
    for e, o in enumerate(oracles):
        sl = slice(e * K, (e + 1) * K)
        o.set_state(**{k: (st["pos64"][sl] if k == "pos" else st[k][sl].astype(np.float64)) for k in PHYS},
                    goal=st["goal"][sl].astype(np.float64),
                    flags=st["flags"][sl] & 0xFF, col_mask=st["col_mask"][sl].astype(np.uint32),
                    tick=int(st["tick"][e]), svd_ctr=int(st["svd_ctr"][e]), step_ctr=int(st["step_ctr"][e]),
                    obst_xy=st["obst_xy"][e, :cfg.num_obstacles].astype(np.float64) if cfg.use_obstacles else None)
        if "scenario" in st:                      # formation scenarios: the scenario object's state (QS_SC_* row)
            o.set_scenario(st["scenario"][e].astype(np.float64))
    return st


def oracle_state(oracles):
    sts = [o.get_state() for o in oracles]
    out = {k: np.concatenate([s[k].reshape(len(s["flags"]), -1) for s in sts]) for k in PHYS + ("goal",)}
    out["flags"] = np.concatenate([s["flags"] for s in sts])
    out["col_mask"] = np.concatenate([s["col_mask"] for s in sts])
    out["tick"] = np.array([s["tick"] for s in sts])
    return out


def action_batch(rs, n, kind):
    if kind == "uniform":
        return rs.uniform(-1.0, 1.0, (n, 4)).astype(np.float32)
    if kind == "high":
        return rs.uniform(-0.2, 1.3, (n, 4)).astype(np.float32)
    return (0.05 + rs.uniform(-0.15, 0.15, (n, 4))).astype(np.float32)


def test_philox_contract_bit_exact():
    """The device generator and the oracle's are the same function of (counter, key)."""
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    L = _capi.lib()
    rs = np.random.RandomState(0)
    for _ in range(16):
        c = [int(x) for x in rs.randint(0, 2 ** 32, 6, dtype=np.uint64)]
        out = (C.c_uint32 * 4)()
        f = (C.c_float * 6)()
        assert L.qs_philox_probe(*c, out, f) == 0
        ref = philox(*c)
        assert list(out) == [int(x) for x in ref]
        u = lambda x: ((x >> 9) + 0.5) / 2 ** 23
        assert f[0] == np.float32(u(int(ref[0]))) and f[1] == np.float32(u(int(ref[1])))
        for p in range(2):
            u1, u2 = u(int(ref[2 * p])), u(int(ref[2 * p + 1]))
            rad, ang = np.sqrt(-2 * np.log(u1)), 2 * np.pi * u2
            np.testing.assert_allclose([f[2 + 2 * p], f[3 + 2 * p]], [rad * np.cos(ang), rad * np.sin(ang)], atol=2e-6)


def check_reset(cfg, obs, st, oracles, envs):
    """The reset envs `envs` of the kernel's observations `obs` and state `st` (host arrays) against their oracles, just reset."""
    K = cfg.num_agents
    rows = (envs[:, None] * K + np.arange(K)[None, :]).reshape(-1)
    ref = np.concatenate([oracles[e].reset() for e in envs])
    os_ = oracle_state([oracles[e] for e in envs])
    # a yaw-rejection tie (cos >= 0.5 in fp32 vs fp64) may flip one drone's accepted attempt: allow a handful
    bad = np.abs(st["rot"][rows] - os_["rot"]).max(axis=1) > 1e-5
    for i in np.unique(np.flatnonzero(bad) // K):
        proved, m = tie_proven(oracles[envs[i]], ("yaw",))
        assert proved, f"env {envs[i]}: spawn yaw differs without a rejection tie (margins in fp32 ulps: {m})"
    ok = ~bad
    np.testing.assert_allclose(st["pos"][rows][ok], os_["pos"][ok], atol=2e-6)
    np.testing.assert_allclose(st["goal"][rows], os_["goal"], atol=1e-6)
    okrows = np.repeat(ok.reshape(len(envs), K).all(axis=1), K)
    np.testing.assert_allclose(obs[rows][okrows], ref[okrows], atol=2e-5)
    if cfg.use_obstacles:
        for e in envs:
            np.testing.assert_allclose(st["obst_xy"][e, :cfg.num_obstacles], oracles[e].get_state()["obst_xy"], atol=1e-6)
    assert (st["tick"][envs] == 0).all()


@pytest.mark.parametrize("name", list(CONFIGS))
def test_reset_parity(name):
    """A full reset, then a masked one: the envs it names (one of them in the partial last warp-tile) against a second oracle
    reset, the others' observation rows and state bitwise unchanged."""
    cfg, sim, oracles = make_pair(name)
    N, K = cfg.num_envs, cfg.num_agents
    obs = sim.reset().cpu().numpy()
    assert obs.shape == (N * K, cfg.obs_dim)
    st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
    check_reset(cfg, obs, st, oracles, np.arange(N))
    assert (st["step_ctr"] == 1).all()

    mask = np.zeros(N, bool)
    mask[[1, N // 2, N - 1]] = True
    obs2 = sim.reset(torch.from_numpy(mask)).cpu().numpy()
    st2 = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
    check_reset(cfg, obs2, st2, oracles, np.flatnonzero(mask))     # the oracles' second reset draws from the same counter
    keep_rows = np.repeat(~mask, K)
    assert np.array_equal(obs2[keep_rows].view(np.int32), obs[keep_rows].view(np.int32)), "masked-out observation rows changed"
    for k, v in st.items():
        if k == "step_ctr":                                         # the handle's launch counter, reported per env
            continue
        sel = keep_rows if v.shape[0] == N * K else ~mask
        assert np.array_equal(st2[k][sel].view(np.uint8), v[sel].view(np.uint8)), f"state {k} of a masked-out env changed"


def run_parity(name, cfg, sim, oracles, kind, steps, hook=None, check_records=True, record_envs=None, goal_atol=None):
    """Every step: copy the GPU state into the oracle, step both with the same actions, compare everything.
    `record_envs`, if given, is called after each step and returns a bool mask [N]: the envs whose just-finished episode record
    is compared (default: every env that finished).  `goal_atol`, if given, is called with the state before and after the step
    and returns the goal tolerance per drone [N*K] (default 3e-6 for every drone)."""
    K, N = cfg.num_agents, cfg.num_envs
    rs = np.random.RandomState(11)
    worst = dict(pos=0.0, vel=0.0, rot=0.0, omega=0.0, obs=0.0, rew=0.0)
    cnt = dict(done=0, impulse=0, flag_mismatch=0, rows=0, env_skipped=0, tie_envs=0, proven_ties=0, unproven=0)
    for s in range(steps):
        if hook is not None:
            hook(s)
        pre = push_state(sim, oracles, cfg)
        a = action_batch(rs, N * K, kind)
        obs, rew, done = sim.step(torch.from_numpy(a).cuda())
        obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
        term = sim.terminal_obs.cpu().numpy()
        st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
        ref_obs, ref_rew, ref_done, ref_term = [], [], [], []
        for e, o in enumerate(oracles):
            ob, rw, dn, tm = o.step(a[e * K:(e + 1) * K].astype(np.float64), want_terminal=True)
            ref_obs.append(ob); ref_rew.append(rw); ref_done.append(dn); ref_term.append(tm)
            cnt["impulse"] += o.diag()["impulse_flag"]
        ref_obs, ref_rew, ref_done = np.concatenate(ref_obs), np.concatenate(ref_rew), np.concatenate(ref_done)
        ref_term = np.concatenate(ref_term)
        os_ = oracle_state(oracles)
        assert np.array_equal(done, ref_done), f"step {s}: done mask"
        assert np.array_equal(st["tick"], os_["tick"]), f"step {s}: tick"
        # discrete flags / collision rows must agree except at fp32-vs-fp64 threshold ties: an env where they differ
        # (rare) is dropped from the value comparison of this step and counted
        flag_ok = ((st["flags"] & 0xFF) == (os_["flags"] & 0xFF)) & (st["col_mask"].astype(np.uint32) == os_["col_mask"])
        env_ok = flag_ok.reshape(N, K).all(axis=1)
        if (~flag_ok).any() and cnt["flag_mismatch"] < 6:
            i = int(np.argmax(~flag_ok))
            import os
            if os.path.isdir("gpurun_out") and cnt["flag_mismatch"] == 0:
                sl = slice((i // K) * K, (i // K + 1) * K)
                np.savez(f"gpurun_out/mismatch_{name}.npz", env=i // K, drone=i % K, step=s, actions=a[sl],
                         **{"pre_" + k: v[sl] for k, v in pre.items() if v.shape[0] == N * K},
                         **{"gpu_" + k: v[sl] for k, v in st.items() if v.shape[0] == N * K},
                         **{"ora_" + k: v[sl] for k, v in os_.items() if v.shape[0] == N * K},
                         pre_tick=pre["tick"][i // K], pre_svd=pre["svd_ctr"][i // K], pre_step=pre["step_ctr"][i // K])
            print(f"[{name}] step {s}: flags of env {i // K} drone {i % K}: gpu {st['flags'][i] & 0xFF:#x}/{st['col_mask'][i]:#x} oracle "
                  f"{os_['flags'][i] & 0xFF:#x}/{os_['col_mask'][i]:#x} pos {st['pos'][i]} vs {os_['pos'][i]}")
        # threshold ties that the final flags cannot show: (i) a floor touch/lift-off inside a sub-step (z within 3e-5 m of
        # the arm height), (ii) a drone lying exactly on a wall plane with |v| below float64 resolution of dt*v (only
        # arises when drones are spawned outside a too-small room)
        arm = cfg.to_c().arm
        near_floor = (np.abs(os_["pos"][:, 2] - arm) < 3e-5) & ((os_["flags"] & 1) == 0)
        hx, hy = cfg.room_dims[0] / 2, cfg.room_dims[1] / 2
        on_wall = ((np.abs(pre["pos"][:, 0]) == hx) & (np.abs(pre["vel"][:, 0]) < 1e-6)) | \
                  ((np.abs(pre["pos"][:, 1]) == hy) & (np.abs(pre["vel"][:, 1]) < 1e-6))
        tie = (near_floor | on_wall).reshape(N, K).any(axis=1)
        env_ok &= ~tie
        # a reset inside the step draws a spawn yaw by rejection; a tie there shows up as a different rotation
        rot_far = (np.abs(st["rot"] - os_["rot"]).max(axis=1) > 1e-3).reshape(N, K).any(axis=1)
        env_ok &= ~(rot_far & done.reshape(N, K).any(axis=1))
        flag_env_bad = ~flag_ok.reshape(N, K).all(axis=1)
        yaw_env_bad = rot_far & done.reshape(N, K).any(axis=1)
        for e in np.flatnonzero(flag_env_bad | yaw_env_bad):
            classes = (FLAG_CLASSES if flag_env_bad[e] else ()) + (("yaw",) if yaw_env_bad[e] else ())
            proved, m = tie_proven(oracles[e], classes)
            cnt["proven_ties"] += int(proved)
            if not proved:
                cnt["unproven"] += 1
                print(f"[{name}] step {s}: env {e} disagrees with the oracle and NO decision was near its threshold (fp32 ulps): {m}")
        cnt["flag_mismatch"] += int(((~flag_ok) & ~np.repeat(tie, K)).sum()); cnt["rows"] += flag_ok.size
        cnt["env_skipped"] += int((~env_ok & ~tie).sum()); cnt["tie_envs"] += int(tie.sum())
        rows = np.repeat(env_ok, K)
        if not rows.any():
            continue
        for k in ("pos", "vel", "rot", "omega"):
            e_ = np.abs(st[k] - os_[k]).max(axis=1) / np.maximum(np.abs(os_[k]).max(axis=1), 1.0)
            e_[~rows] = 0
            if e_.max() > REL_TOL:
                i = int(np.argmax(e_))
                print(f"[{name}] step {s}: {k} of env {i // K} drone {i % K} off by {e_.max():.3e}: gpu {st[k][i]} oracle {os_[k][i]} "
                      f"flags {st['flags'][i]:#x} pos {st['pos'][i]} diag {oracles[i // K].diag()['new_pairs']}")
        worst["pos"] = max(worst["pos"], relerr(st["pos"][rows], os_["pos"][rows], 1.0))
        worst["vel"] = max(worst["vel"], relerr(st["vel"][rows], os_["vel"][rows], 1.0))
        worst["rot"] = max(worst["rot"], relerr(st["rot"][rows], os_["rot"][rows], 1.0))
        worst["omega"] = max(worst["omega"], relerr(st["omega"][rows], os_["omega"][rows], 1.0))
        if "scenario" in st:
            ref_rows = np.stack([o.get_scenario() for o in oracles])
            gtol = 3e-6 if goal_atol is None else goal_atol(pre, st)[rows][:, None]
            gbad = ~(np.abs(st["goal"][rows] - os_["goal"][rows]) <= gtol + 1e-7 * np.abs(os_["goal"][rows]))   # assert_allclose's rule
            assert not gbad.any(), f"step {s}: goals of drones {np.flatnonzero(rows)[gbad.any(axis=1)]} differ by more than the tolerance"
            assert np.array_equal(st["scenario"][env_ok][:, [0, 1, 9, 10]], ref_rows[env_ok][:, [0, 1, 9, 10]]), f"step {s}: scenario ids / timers"
            np.testing.assert_allclose(st["scenario"][env_ok], ref_rows[env_ok], atol=3e-6, err_msg=f"step {s}: scenario rows")
            worst["goal"] = max(worst.get("goal", 0.0), float(np.abs(st["goal"][rows] - os_["goal"][rows]).max()))
            cnt["goal_moves"] = cnt.get("goal_moves", 0) + int((np.abs(st["goal"] - pre["goal"]).max(axis=1) > 0).reshape(N, K).any(axis=1).sum())
        # neighbour rows chosen by rank (V < K - 1): a different choice or order is a discrete disagreement, accepted for an env
        # only when the oracle's ranking had two candidates within the rank bound; that env's neighbour columns are then skipped
        obs_c = obs
        if cfg.neighbor_obs_type == "pos_vel" and 0 < cfg.visible < K - 1:
            nb = slice(OBS_REPR_DIM[cfg.obs_repr], OBS_REPR_DIM[cfg.obs_repr] + 6 * cfg.visible)
            d_nb = np.abs(obs[:, nb] - ref_obs[:, nb]) / np.maximum(np.abs(ref_obs[:, nb]), 1.0)
            for e in np.flatnonzero(((d_nb > 5e-5).any(axis=1).reshape(N, K).any(axis=1)) & env_ok):
                proved, m = tie_proven(oracles[e], ("rank",))
                cnt["rank_ties"] = cnt.get("rank_ties", 0) + int(proved)
                if not proved:
                    cnt["unproven"] += 1
                    print(f"[{name}] step {s}: neighbour rows of env {e} differ and NO ranking was near a tie (fp32 ulps): {m}")
                    continue
                if obs_c is obs:
                    obs_c = obs.copy()
                obs_c[e * K:(e + 1) * K, nb] = ref_obs[e * K:(e + 1) * K, nb]
        worst["obs"] = max(worst["obs"], relerr(obs_c[rows], ref_obs[rows], 1.0))
        worst["rew"] = max(worst["rew"], float(np.abs(rew[rows] - ref_rew[rows]).max()))
        drows = rows & done
        if drows.any():
            np.testing.assert_allclose(term[drows], ref_term[drows], atol=5e-5, err_msg=f"step {s}: terminal obs")
        if done.any() and check_records:
            # per-episode records (infos[i]['episode_extra_stats']) of the envs that just finished
            env_rec, agent_rec = sim.episode_records_host()
            sel = done.reshape(N, K)[:, 0] & env_ok
            if record_envs is not None:
                sel = sel & record_envs()
            for e in np.flatnonzero(sel):
                ref_env, ref_agent = oracles[e].record()
                same = np.array_equal(env_rec[e, 1:19], ref_env[1:19])
                cnt["record_mismatch"] = cnt.get("record_mismatch", 0) + int(not same)
                if not same and cnt["record_mismatch"] <= 3:
                    print(f"[{name}] step {s}: episode record of env {e}: gpu {env_rec[e]} oracle {ref_env}")
                np.testing.assert_allclose(agent_rec[e * K:(e + 1) * K, :3], ref_agent[:, :3], rtol=2e-4, atol=1e-5, equal_nan=True,
                                           err_msg=f"step {s}: distance_to_goal windows of env {e}")
                cnt["records"] = cnt.get("records", 0) + 1
        cnt["done"] += int(done.reshape(N, K).any(axis=1).sum())
    print(f"\n[{name}] worst one-step rel err {worst}  {cnt}")
    for k in ("pos", "vel", "rot", "omega"):
        assert worst[k] <= REL_TOL, (k, worst[k])
    assert worst["obs"] <= 5e-5 and worst["rew"] <= 5e-6
    assert cnt["unproven"] == 0, "discrete state differs from the oracle away from any threshold tie"
    assert cnt["env_skipped"] <= max(2, (steps * N) // 200)
    assert cnt["tie_envs"] <= (steps * N) // 10
    # counters and agent tallies of the finished episodes agree (a tie earlier in the episode may flip one flag for good)
    assert cnt.get("record_mismatch", 0) <= max(1, cnt.get("records", 0) // 50), cnt
    return worst, cnt


@pytest.mark.parametrize("name,kind,steps", [
    ("cfg2_k8", "uniform", 60), ("cfg3_obst_k8", "hover", 60), ("cfg4_k32", "uniform", 40),
    ("smallroom_k8", "high", 70), ("crowd_k16", "hover", 60), ("nonoise_wall_k4", "uniform", 45),
    ("single_k1", "uniform", 45), ("odd_k3", "uniform", 45), ("odd_k6_obst", "hover", 45), ("single_k1_obst", "hover", 45)])
def test_single_step_parity(name, kind, steps):
    cfg, sim, oracles = make_pair(name)
    sim.reset()
    for o in oracles:
        o.reset()          # same draws as the GPU reset: the oracle learns which scenario (approach metric) its first episode runs
    worst, cnt = run_parity(name, cfg, sim, oracles, kind, steps)
    assert cnt["done"] >= cfg.num_envs          # every env went through at least one auto-reset
    if name in ("smallroom_k8", "crowd_k16"):
        assert cnt["impulse"] > 0


def test_forced_events_parity():
    """Hand-placed drones so that every impulse type fires in every env on known steps: obstacle hit, downwash,
    new drone-drone pair (incl. one drone in two new pairs), wall and ceiling bounce, upside-down touchdown."""
    cfg = QuadSimConfig(seed=21, num_envs=16, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                        obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, ep_time=2.0)
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(cfg.num_envs)]
    sim.reset()
    K, N = cfg.num_agents, cfg.num_envs

    def hook(s):
        if s not in (3, 9):
            return
        st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
        pos, vel, rot = st["pos"].reshape(N, K, 3).copy(), st["vel"].reshape(N, K, 3).copy(), st["rot"].reshape(N, K, 9).copy()
        for e in range(N):
            ox, oy = st["obst_xy"][e, 0]
            pos[e, 0] = (ox + 0.3 + 0.046 + 0.015, oy, 2.0); vel[e, 0] = (-2.5, 0.0, 0.0)          # obstacle hit
            pos[e, 1] = (4.2, -4.2, 6.0); vel[e, 1] = 0.0
            pos[e, 2] = (4.2, -4.2, 6.3); vel[e, 2] = 0.0                                             # 2 above 1: downwash
            pos[e, 3] = (-4.0, 4.0, 5.0); pos[e, 4] = (-4.0, 4.06, 5.04); pos[e, 5] = (-4.0, 3.94, 4.96)  # 3 in two pairs
            vel[e, 3] = (0.0, 0.0, 0.0); vel[e, 4] = (0.0, -1.0, 0.0); vel[e, 5] = (0.0, 1.0, 0.0)
            pos[e, 6] = (4.995, 1.0, 9.995); vel[e, 6] = (3.0, 0.5, 3.0)                              # wall + ceiling
            pos[e, 7] = (-3.0, -3.0, 0.05); vel[e, 7] = (0.3, 0.0, -1.0)                              # touchdown, inverted
            rot[e, 7] = (1, 0, 0, 0, -1, 0, 0, 0, -1)
        sim.set_state(pos=pos.reshape(-1, 3), vel=vel.reshape(-1, 3), rot=rot.reshape(-1, 9))

    worst, cnt = run_parity("forced_events", cfg, sim, oracles, "hover", 16, hook)
    assert cnt["impulse"] >= 2 * N
    flags = sim.get_state(("flags",))["flags"].cpu().numpy().reshape(N, K)
    assert (flags[:, 7] & 1).all()              # drone 7 sits on the floor in every env


def test_free_running_drift_100_steps():
    """No teacher forcing: 100 control steps from the same reset.  Free flight stays within 1e-3; once drones slide on the
    floor the friction chatter is chaotic (errors grow ~6x per sub-step in float64 as well, see DESIGN.md), so drones that
    touched the floor are only required to stay bounded."""
    cfg = QuadSimConfig(seed=5, num_envs=32, num_agents=8, ep_time=15.0)
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(cfg.num_envs)]
    sim.reset()
    for o in oracles:
        o.reset()
    push_state(sim, oracles, cfg)          # identical fp32-representable start
    rs = np.random.RandomState(2)
    K, N = cfg.num_agents, cfg.num_envs
    touched = np.zeros(N * K, dtype=bool)
    drift = []
    for s in range(100):
        a = (0.1 + rs.uniform(-0.3, 0.3, (N * K, 4))).astype(np.float32)
        sim.step(torch.from_numpy(a).cuda())
        for e, o in enumerate(oracles):
            o.step(a[e * K:(e + 1) * K].astype(np.float64))
        st = {k: v.cpu().numpy() for k, v in sim.get_state(("pos", "vel", "flags")).items()}
        os_ = oracle_state(oracles)
        touched |= ((st["flags"] | os_["flags"]) & 1).astype(bool)
        err = np.abs(st["pos"] - os_["pos"]).max(axis=1)
        drift.append((float(err[~touched].max()) if (~touched).any() else 0.0, float(err.max())))
    free = max(d[0] for d in drift)
    print(f"\n[drift] 100 steps: free-flight max |dpos| = {free:.3e} m, all drones max |dpos| = {max(d[1] for d in drift):.3e} m, "
          f"{int(touched.sum())}/{N * K} drones touched the floor")
    assert (~touched).sum() > N * K // 4
    assert free < 1e-3
    assert max(d[1] for d in drift) < 1.0


def test_host_buffer_path_matches_device_path():
    cfg = QuadSimConfig(seed=9, num_envs=16, num_agents=8)
    a_sim, b_sim = _sim(cfg), _sim(cfg)
    o1 = a_sim.reset().cpu().numpy()
    o2 = b_sim.reset_host()
    assert np.array_equal(o1, o2)
    rs = np.random.RandomState(1)
    for _ in range(5):
        a = rs.uniform(-1, 1, (cfg.num_envs * cfg.num_agents, 4)).astype(np.float32)
        ob, rw, dn = a_sim.step(torch.from_numpy(a).cuda())
        hob, hrw, hdn = b_sim.step_host(a)
        assert np.array_equal(ob.cpu().numpy(), hob) and np.array_equal(rw.cpu().numpy(), hrw)
        assert np.array_equal(dn.cpu().numpy(), hdn)


def test_masked_reset_and_sharding_independence():
    """env_id_offset keys the RNG by GLOBAL env id: a shard [8,16) reproduces envs 8..15 of the full batch."""
    full = _sim(QuadSimConfig(seed=4, num_envs=16, num_agents=8))
    shard = _sim(QuadSimConfig(seed=4, num_envs=8, num_agents=8, env_id_offset=8))
    of, os_ = full.reset().cpu().numpy(), shard.reset().cpu().numpy()
    assert np.array_equal(of[64:], os_)
    rs = np.random.RandomState(0)
    for _ in range(20):
        a = rs.uniform(-1, 1, (128, 4)).astype(np.float32)
        of = full.step(torch.from_numpy(a).cuda())[0].cpu().numpy()
        os_ = shard.step(torch.from_numpy(a[64:]).cuda())[0].cpu().numpy()
        assert np.array_equal(of[64:], os_)
    # masked reset touches only the chosen envs
    before = full.get_state(("pos", "tick"))
    mask = torch.zeros(16, dtype=torch.bool)
    mask[[1, 5]] = True
    obs_before = full.obs.clone()
    full.reset(mask)
    after = full.get_state(("pos", "tick"))
    changed = (before["pos"] != after["pos"]).any(dim=1).reshape(16, 8).any(dim=1).cpu()
    assert changed.tolist() == mask.tolist()
    assert (after["tick"].cpu()[mask] == 0).all() and (after["tick"].cpu()[~mask] == 20).all()
    same_rows = (~mask).repeat_interleave(8)
    assert torch.equal(full.obs.cpu()[same_rows], obs_before.cpu()[same_rows])


def test_episode_stats_match_oracle():
    cfg = QuadSimConfig(seed=8, num_envs=24, num_agents=8, ep_time=0.5, room_dims=(4.0, 4.0, 4.0))
    sim = _sim(cfg)
    oracles = [OracleEnv(cfg, i) for i in range(cfg.num_envs)]
    sim.reset()
    rs = np.random.RandomState(3)
    K, N = cfg.num_agents, cfg.num_envs
    for s in range(110):
        push_state(sim, oracles, cfg)
        a = action_batch(rs, N * K, "high")
        sim.step(torch.from_numpy(a).cuda())
        for e, o in enumerate(oracles):
            o.step(a[e * K:(e + 1) * K].astype(np.float64))
    gs = sim.episode_stats()
    ref = {}
    for o in oracles:
        for k, v in o.stats().items():
            ref[k] = ref.get(k, 0) + v
    assert gs["episodes"] == ref["episodes"] == 2 * N
    for k in ("num_collisions", "num_collisions_with_floor", "num_collisions_with_wall", "num_collisions_with_ceiling",
              "num_collisions_with_room", "num_collisions_after_settle"):
        assert abs(gs[k] - ref[k]) <= max(2, 0.02 * ref[k]), (k, gs[k], ref[k])
    for k in ("distance_to_goal_1s", "distance_to_goal_3s", "distance_to_goal_5s"):
        assert abs(gs[k] - ref[k]) <= 1e-3 * abs(ref[k]), (k, gs[k], ref[k])
    assert gs["agents_success"] + gs["agents_deadlock"] + gs["agents_collided"] == 2 * N * K


# ------------------------------------------------------------------------------------------------------------------
# oracle parity AT THE BENCHMARKED LAUNCH SHAPES (BASELINE.json configs[1..4]): 128-thread blocks, full grids
# ------------------------------------------------------------------------------------------------------------------
class SubsetSim:
    """The rows of a sampled set of envs of a large batch behind QuadSwarmSim's interface: run_parity teacher-forces and compares
    these envs against one OracleEnv each (created with the env's GLOBAL index, which keys its RNG), while the kernel runs the full
    batch -- the launch shape bench.py times.  The other envs get i.i.d. U(-1,1) actions."""

    def __init__(self, sim, env_idx, seed=0):
        self.sim, self.K = sim, sim.K
        self.env_idx = torch.as_tensor(env_idx, device=sim.device, dtype=torch.long)
        self.rows = (self.env_idx[:, None] * self.K + torch.arange(self.K, device=sim.device)[None, :]).reshape(-1)
        self.gen = torch.Generator(device=sim.device)
        self.gen.manual_seed(seed)

    def step(self, a_small):
        full = torch.rand((self.sim.N * self.K, self.sim.A), device=self.sim.device, generator=self.gen) * 2.0 - 1.0
        full[self.rows] = a_small
        obs, rew, done = self.sim.step(full)
        return obs[self.rows], rew[self.rows], done[self.rows]

    @property
    def terminal_obs(self):
        return self.sim.terminal_obs[self.rows]

    def get_state(self, fields=None):
        st = self.sim.get_state(fields)
        return {k: (v[self.rows] if v.shape[0] == self.sim.N * self.K else v[self.env_idx]) for k, v in st.items()}

    def episode_records_host(self):
        env, agent = self.sim.episode_records_host()
        return env[self.env_idx.cpu().numpy()], agent[self.rows.cpu().numpy()]


BIG = {
    "cfg2_4096x8": (dict(num_envs=4096, num_agents=8, ep_time=0.25), "uniform"),
    "cfg3_obst_4096x8": (dict(num_envs=4096, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                              obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, ep_time=0.25), "hover"),
    "cfg4_1024x32": (dict(num_envs=1024, num_agents=32, ep_time=0.25), "uniform"),
    "cfg5_65536x8": (dict(num_envs=65536, num_agents=8, ep_time=0.25), "uniform"),
    "cfg3_obst_65536x8": (dict(num_envs=65536, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                               obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, ep_time=0.25), "hover"),
    "cfg4_16384x32": (dict(num_envs=16384, num_agents=32, ep_time=0.25), "uniform"),
}


@pytest.mark.parametrize("name", list(BIG))
def test_parity_at_benchmarked_launch_shape(name, monkeypatch):
    """>= 256 sampled envs of the full-size batch against the oracle, teacher-forced, 32 steps (every env auto-resets once), with
    the 128-thread blocks the benchmark launches (forced for the 4096 / 1024-env points, whose default is 64)."""
    import dataclasses
    kw, kind = BIG[name]
    cfg = QuadSimConfig(seed=13, **kw)
    monkeypatch.setenv("QS_BLOCK", "128")
    sim = _sim(cfg)
    monkeypatch.delenv("QS_BLOCK")
    n_sample = 256 if cfg.num_agents <= 8 else 64              # 64 x 32 = 2048 drones for the 32-quad envs
    rs = np.random.RandomState(5)
    idx = np.sort(rs.choice(cfg.num_envs, n_sample, replace=False))
    idx[0], idx[-1] = 0, cfg.num_envs - 1                       # first and last warp-tile of the grid
    sub = SubsetSim(sim, idx, seed=3)
    oracles = [OracleEnv(cfg, int(i)) for i in idx]
    sim.reset()
    for o in oracles:
        o.reset()
    small = dataclasses.replace(cfg, num_envs=n_sample)
    worst, cnt = run_parity(name, small, sub, oracles, kind, 32)
    assert cnt["done"] >= n_sample


FEATS = {
    "feat0_plain": dict(num_agents=8),
    "feat1_obst": dict(num_agents=8, quads_mode="o_random", use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2),
    "feat2_downwash": dict(num_agents=8, use_downwash=True),
    "feat3_obst_downwash": dict(num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True, obs_repr="xyz_vxyz_R_omega_floor",
                                neighbor_visible_num=2),
    "feat4_scenarios": dict(num_agents=8, quads_mode="mix"),
    "feat6_scenarios_downwash": dict(num_agents=8, quads_mode="mix", use_downwash=True),
    "k32": dict(num_agents=32),
    "k3": dict(num_agents=3, neighbor_visible_num=1),
    "fork_k4": dict(env_mode="fork", num_agents=4, capture_radius=2.6),
    "fork_k12_sangle_v5": dict(env_mode="fork", num_agents=12, capture_radius=2.2, obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot",
                               neighbor_obs_type="dist_sangle", neighbor_visible_num=5),
}


@pytest.mark.parametrize("name", list(FEATS))
def test_block_64_and_128_are_bitwise_identical(name, monkeypatch):
    """The launch shape is not part of the result: 64- and 128-thread blocks (the small-batch and the large-batch default) produce
    the same bits in every feature variant of the step kernel and in the fork kernel, including partial last blocks and auto-resets."""
    make = QuadSimConfig.fork_default if FEATS[name].get("env_mode") == "fork" else QuadSimConfig
    cfg = make(seed=23, num_envs=301, ep_time=0.15, **FEATS[name])
    sims = []
    for blk in ("64", "128"):
        monkeypatch.setenv("QS_BLOCK", blk)
        sims.append(_sim(cfg))
    monkeypatch.delenv("QS_BLOCK")
    a_sim, b_sim = sims
    assert torch.equal(a_sim.reset(), b_sim.reset())
    rs = np.random.RandomState(6)
    n_done = 0
    for s in range(40):
        a = action_batch(rs, cfg.num_envs * cfg.num_agents, "uniform" if s % 2 else "hover")
        a = torch.from_numpy(np.ascontiguousarray(a[:, :a_sim.A])).cuda()
        o1, r1, d1 = a_sim.step(a)
        o2, r2, d2 = b_sim.step(a)
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2), f"step {s}"
        assert torch.equal(a_sim.terminal_obs, b_sim.terminal_obs)
        n_done += int(d1.any())
    assert n_done >= 2
    s1, s2 = a_sim.get_state(), b_sim.get_state()
    for k in s1:
        assert torch.equal(s1[k], s2[k]), k
    assert a_sim.episode_stats() == b_sim.episode_stats()


def test_two_handles_share_kernel_attributes():
    """Train env + eval env on one device (how sb_train.py runs): the dynamic shared-memory limit of a kernel instantiation is a
    per-device attribute, so a second, smaller handle must not lower it under the first one (K=32 with all 31 neighbours
    visible needs ~108 KB per 128-thread block at large N and ~54 KB per 64-thread block at small N)."""
    big = _sim(QuadSimConfig(seed=1, num_envs=2048, num_agents=32, neighbor_visible_num=-1, ep_time=0.1))
    big.reset()
    small = _sim(QuadSimConfig(seed=2, num_envs=8, num_agents=32, neighbor_visible_num=-1, ep_time=0.1))
    small.reset()
    gen = torch.Generator(device="cuda"); gen.manual_seed(0)
    for s in range(15):
        ob, _, _ = big.step(torch.rand((2048 * 32, 4), device="cuda", generator=gen) * 2 - 1)
        os_, _, _ = small.step(torch.rand((8 * 32, 4), device="cuda", generator=gen) * 2 - 1)
        torch.cuda.synchronize()
        assert bool(torch.isfinite(ob).all()) and bool(torch.isfinite(os_).all())
    big.reset(); small.reset()
    torch.cuda.synchronize()
