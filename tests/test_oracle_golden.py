"""The CPU oracle (oracle/quadsim_oracle.c) against outputs of the reference itself.

Fixtures are produced by tests/golden/make_golden.py from the unmodified reference in /root/reference
(SURVEY.md 8c: the reference's own tests hold no usable golden vectors for this path).
"""
import ast
import os

import numpy as np
import pytest

from oracle import OracleEnv
from quad_swarm_rl_stable_baselines3_b200 import quad_model
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig, episode_extra_stats

PHYS = ("pos", "vel", "rot", "omega", "rot_damp", "cmds_damp", "ou")


def cfg_from_kwargs(kw):
    kw = dict(kw)
    rew = kw.pop("rew_coeff", None) or {}
    rew = {k: v for k, v in rew.items()}
    return QuadSimConfig(num_envs=1, rew_coeff=rew, **kw)


def test_constants_match_reference(golden_dir):
    """quad_model.py vs the reference's QuadLink / update_model (inertia.py:182-310, quadrotor_dynamics.py:106-168)."""
    g = np.load(os.path.join(golden_dir, "dyn_jit.npz"))
    q = quad_model.crazyflie_constants()
    mine = np.array([q.mass, *q.inertia, *q.thrust_max, *q.torque_max, q.arm, q.motor_tau_up,
                     *np.array(q.prop_cross).reshape(-1)])
    np.testing.assert_allclose(mine, g["consts"], rtol=1e-12, atol=1e-18)
    assert quad_model.svd_period(0.005) == 100          # SURVEY.md 8a row a2 (probe)


def test_survey_known_answer_dynamics():
    """SURVEY.md Appendix A.1: one control step of QuadrotorDynamics.step from a hand-made state.
    (set_state rounds omega to float32, quadrotor_dynamics.py:190, hence 1e-8 rather than 1e-13 on what omega feeds.)"""
    o = OracleEnv(QuadSimConfig(num_envs=1, num_agents=1, neighbor_obs_type="none", neighbor_visible_num=0))
    rot = [0.9541425672790118, -0.29881057511918196, -0.018005596439997374,
           0.2951508833549871, 0.9490892608907772, -0.11007057243681952,
           0.04997916927067833, 0.09970865087213879, 0.9937606691655043]
    rd = np.array([0.7, 0.72, 0.68, 0.71])
    o.set_state(pos=[0.3, -0.2, 2.0], vel=[0.1, -0.2, 0.3], rot=rot, omega=[0.5, -0.4, 0.3], rot_damp=rd,
                cmds_damp=rd ** 2, ou=np.zeros(4), flags=[0])
    o.dynamics_only(0, [0.6, 0.5, 0.55, 0.45])
    s = o.get_state()
    np.testing.assert_allclose(s["pos"][0], [0.3009955565579763, -0.2020262077779446, 2.002985078884568], rtol=1e-13)
    np.testing.assert_allclose(s["vel"][0], [0.09815374185664064, -0.21064167712385498, 0.2943324935913465], rtol=1e-8)
    np.testing.assert_allclose(s["omega"][0], [0.3368657149955732, -0.42912022001622524, 0.3058370554945566], rtol=1e-7)
    np.testing.assert_allclose(s["rot"][0], [0.9531554796985265, -0.30178470374268573, -0.02050912254609862,
                                              0.2975597188776914, 0.9476714420573863, -0.11565920460691105,
                                              0.05434008853600427, 0.10413851590940512, 0.9930771995580635], rtol=1e-8)
    np.testing.assert_allclose(s["rot_damp"][0], [0.7185661671889045, 0.7167910409603038, 0.6953364007391983,
                                                   0.7002486915741181], rtol=1e-13)
    np.testing.assert_allclose(s["cmds_damp"][0], [0.5163373366285527, 0.5137893964009559, 0.48349271019294304,
                                                    0.4903482300512643], rtol=1e-13)


def test_reference_unit_test_known_answer_obstacle_normal():
    """The one meaningful known answer in the reference's own tests (collisions/test/unit_test/obstacles.py:6-18):
    pos (0,0,0), vel (1,0,0), obstacle at (0.5,0.5,5) -> vnew = -sqrt(2)/2, collision normal (-sqrt(2)/2, -sqrt(2)/2, 0)."""
    from oracle import col_norm_and_new_vel_obst
    vnew, n = col_norm_and_new_vel_obst([0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.5, 0.5, 5.0])
    assert round(vnew, 6) == round(-np.sqrt(2) / 2.0, 6)
    np.testing.assert_allclose(n, [-np.sqrt(2) / 2.0, -np.sqrt(2) / 2.0, 0.0], atol=1e-15)


def test_dynamics_jit_on(golden_dir):
    """JIT-ON reference QuadrotorDynamics.step: free flight, SVD at sub-step 100, floor touch and sliding.
    One-step teacher-forced comparison (floor friction chatter is chaotic, so free-running traces are only
    compared until first floor contact)."""
    g = np.load(os.path.join(golden_dir, "dyn_jit.npz"))
    cfg = QuadSimConfig(num_envs=1, num_agents=1, neighbor_obs_type="none", neighbor_visible_num=0)
    cfg.motor.thrust_noise_ratio = 0.0
    for r in range(int(g["n_runs"])):
        T = g[f"r{r}_cmds"].shape[0]
        o = OracleEnv(cfg)
        worst = 0.0
        for s in range(T):
            fl = int(g[f"r{r}_on_floor"][s])
            o.set_state(pos=g[f"r{r}_pos"][s], vel=g[f"r{r}_vel"][s], rot=g[f"r{r}_rot"][s], omega=g[f"r{r}_omega"][s],
                        rot_damp=g[f"r{r}_rot_damp"][s], cmds_damp=g[f"r{r}_cmds_damp"][s], ou=np.zeros(4), flags=[fl],
                        svd_ctr=(2 * s) % 100)
            a = 2.0 * g[f"r{r}_cmds"][s] - 1.0           # RawControl maps [-1,1] -> [0,1]
            o.step(a[None, :])
            st = o.get_state()
            first_touch = (not g[f"r{r}_on_floor"][s]) and g[f"r{r}_on_floor"][s + 1]
            for k in ("pos", "vel", "rot", "omega", "rot_damp", "cmds_damp"):
                err = np.abs(st[k][0] - g[f"r{r}_{k}"][s + 1]).max()
                if k == "rot" and first_touch and err > 2e-9:
                    # touched down upside-down: the reference draws a random yaw from numba's private RNG
                    # (quadrotor_dynamics.py:623-626), which cannot be taped -> both must be pure yaw rotations
                    for R in (st[k][0], g[f"r{r}_rot"][s + 1]):
                        assert abs(R[8] - 1.0) < 1e-12 and abs(R[0] - R[4]) < 1e-12 and abs(R[1] + R[3]) < 1e-12
                    continue
                worst = max(worst, err)
                assert err < 2e-9, (r, s, k, err)
            assert (st["flags"][0] & 1) == int(g[f"r{r}_on_floor"][s + 1]), (r, s)
            assert ((st["flags"][0] >> 1) & 1) == int(g[f"r{r}_crashed_floor"][s + 1]), (r, s)
        assert g[f"r{r}_on_floor"].sum() > 50           # the run does include floor contact


TRACE_NAMES = ["cfg2_k8", "smallroom_k8", "crowd_k16", "cfg3_obst_k8", "cfg4_k32", "nonoise_k4", "obst_k1"]
# formation scenarios (SURVEY.md 8 f2): compact fixtures -- float32 observations / actions, bit-packed flags, and the
# reference scenario object's own state per step (QS_SC_* row)
SCENARIO_TRACE_NAMES = ["scen_static_diff_k8", "scen_static_diff_k12", "scen_dyn_same_k3", "scen_dyn_diff_k4", "scen_swap_k3",
                        "scen_swarm_k6", "scen_swarm_k4", "scen_dynform_k5", "scen_lissajous_k3", "scen_bezier_k3",
                        "scen_mix_k4", "scen_mix_k1", "scen_runaway_k5"]
SCENARIO_IDS = {"static_same_goal": 0, "static_diff_goal": 5, "dynamic_same_goal": 6, "dynamic_diff_goal": 7, "swap_goals": 8,
                "dynamic_formations": 9, "ep_lissajous3D": 11, "ep_rand_bezier": 12, "swarm_vs_swarm": 13, "run_away": 14}


def load_trace(golden_dir, name):
    g = dict(np.load(os.path.join(golden_dir, f"trace_{name}.npz")))
    if "flag_shape" in g:
        shape = tuple(int(v) for v in g["flag_shape"])
        for k in ("on_floor", "crashed_floor", "crashed_wall", "crashed_ceiling"):
            g["s_" + k] = np.unpackbits(g["s_" + k])[:int(np.prod(shape))].reshape(shape).astype(bool)
        g["actions"] = g["actions"].astype(np.float64)
    return g


def test_formation_goals(golden_dir):
    """QuadrotorScenario.generate_goals (scenarios/base.py:42-116) for all 8 formations x 16 swarm sizes, incl. the quirks:
    a sphere of n < 3 drones has 3 rows, int(27 ** (1/3)) == 2, the cube's x uses formation_center[2]."""
    from oracle import generate_goals
    g = np.load(os.path.join(golden_dir, "formations.npz"))
    for i, (n, fi, size, layer, cx, cy, cz, rows) in enumerate(g["index"]):
        mine = generate_goals(int(fi), size, int(n), [cx, cy, cz], layer)
        assert mine.shape[0] == int(rows), (n, fi)
        np.testing.assert_allclose(mine, g[f"g{i}"], rtol=0, atol=1e-12, err_msg=f"n={n} formation={fi}")


@pytest.mark.parametrize("name", TRACE_NAMES + SCENARIO_TRACE_NAMES)
def test_env_trace(golden_dir, name):
    """QuadrotorEnvMulti.reset/step traces (JIT off, every draw taped): the oracle replays the reference's own draws.
    The physical state is re-synchronised to the reference before every step (teacher forcing; contact dynamics are
    chaotic), while collision / room / episode bookkeeping free-runs across the whole trace."""
    g = load_trace(golden_dir, name)
    files = tuple(g.keys())
    compact = "sc_row" in g
    obs_tol = 2e-6 if compact else 1e-9          # compact fixtures keep observations in float32
    kw = ast.literal_eval(str(g["env_kwargs"]))
    cfg = cfg_from_kwargs(kw)
    K = cfg.num_agents
    o = OracleEnv(cfg)
    on, ou_, oc = np.cumsum(np.r_[0, g["n_tn"]]), np.cumsum(np.r_[0, g["n_tu"]]), np.cumsum(np.r_[0, g["n_tc"]])

    def tape(i):
        o.set_tape(g["tn"][on[i]:on[i + 1]], g["tu"][ou_[i]:ou_[i + 1]], g["tc"][oc[i]:oc[i + 1]])

    def check_tape(i, what):
        assert o.tape_pos() == (g["n_tn"][i], g["n_tu"][i], g["n_tc"][i]), (what, o.tape_pos(), g["n_tn"][i], g["n_tu"][i], g["n_tc"][i])

    def check_state(i, what):
        st = o.get_state()
        for k in PHYS:
            ref = g["s_" + k][i].reshape(K, -1)
            np.testing.assert_allclose(st[k].reshape(K, -1), ref, rtol=0, atol=5e-9, err_msg=f"{what} {k}")
        np.testing.assert_allclose(st["goal"], g["s_goal"][i], atol=1e-12, err_msg=f"{what} goal")
        for bit, key in enumerate(("on_floor", "crashed_floor", "crashed_wall", "crashed_ceiling")):
            assert np.array_equal((st["flags"] >> bit) & 1, g["s_" + key][i].astype(np.int32)), (what, key)
        assert st["tick"] == g["tick"][i], what
        if "obst_xy" in files:
            np.testing.assert_allclose(st["obst_xy"], g["obst_xy"][i], atol=1e-12, err_msg=f"{what} obstacles")
        if compact:
            # the scenario object itself: which scenario this episode runs, formation, sizes, centre, timers
            row, ref = o.get_scenario(), g["sc_row"][i]
            assert int(row[0]) == SCENARIO_IDS[str(g["scenario"][i])], (what, row[0], g["scenario"][i])
            n_cmp = 18 if str(g["scenario"][i]) == "swarm_vs_swarm" else 12
            np.testing.assert_allclose(row[1:n_cmp], ref[1:n_cmp], rtol=0, atol=1e-12, err_msg=f"{what} scenario state")

    tape(0)
    obs = o.reset()
    check_tape(0, "reset")
    np.testing.assert_allclose(obs, g["obs"][0], rtol=0, atol=obs_tol)
    check_state(0, "reset")
    n_done = n_impulse = 0
    T = g["actions"].shape[0]
    ep_rows = {int(st_): row for st_, row in zip(g["ep_step"], g["ep_stats"])} if "ep_step" in files else {}
    STAT_KEYS = ("num_collisions", "num_collisions_after_settle", "num_collisions_final_5s", "num_collisions_with_room",
                 "num_collisions_with_floor", "num_collisions_with_wall", "num_collisions_with_ceiling",
                 "num_collisions_obst_quad", "num_collisions_obst_quad_after_settle", "agents_success", "agents_deadlock",
                 "agents_collided", "distance_to_goal_1s", "distance_to_goal_3s", "distance_to_goal_5s")
    prev_stats = o.stats()
    for s in range(T):
        # teacher forcing of the physical state only
        st = o.get_state()
        fl = (st["flags"] & ~0xF)
        for bit, key in enumerate(("on_floor", "crashed_floor", "crashed_wall", "crashed_ceiling")):
            fl |= g["s_" + key][s].astype(np.int32) << bit
        o.set_state(flags=fl, **{k: g["s_" + k][s] for k in PHYS})
        tape(s + 1)
        obs, rew, done = o.step(g["actions"][s])
        check_tape(s + 1, f"step {s}")
        check_state(s + 1, f"step {s}")
        np.testing.assert_allclose(rew, g["rew"][s], rtol=0, atol=1e-9, err_msg=f"step {s} reward")
        assert np.array_equal(done, g["done"][s]), f"step {s} done"
        np.testing.assert_allclose(obs, g["obs"][s + 1], rtol=0, atol=max(obs_tol, 1e-8), err_msg=f"step {s} obs")
        n_done += int(done.any())
        n_impulse += o.diag()["impulse_flag"]
        if done.any() and ep_rows:
            # infos[i]['episode_extra_stats'] of the reference (quadrotor_multi.py:739-831) vs what this episode added to qs_stats
            cur = o.stats()
            delta = np.array([cur[k] - prev_stats[k] for k in STAT_KEYS], dtype=np.float64)
            np.testing.assert_allclose(delta[:12], ep_rows[s][:12], rtol=0, atol=0, err_msg=f"step {s} episode counters")
            np.testing.assert_allclose(delta[12:], ep_rows[s][12:], rtol=1e-9, atol=1e-9, err_msg=f"step {s} distance_to_goal windows")
            assert cur["episodes"] - prev_stats["episodes"] == 1
            prev_stats = cur
            # the per-episode record -> the dict the VecEnv layer hands out as infos[i]['episode_extra_stats']
            env_rec, agent_rec = o.record()
            ep_i = list(ep_rows).index(s)
            assert env_rec[0] == ep_i + 1 and env_rec[16] == cfg.ep_len + 1
            np.testing.assert_array_equal(env_rec[2:14], ep_rows[s][:12].astype(np.int32))
            np.testing.assert_allclose(agent_rec[:, :3].sum(axis=0), ep_rows[s][12:], rtol=1e-9, atol=1e-9)
            if compact:
                det, sname = g["ep_detail"][ep_i], str(g["ep_scenario"][ep_i])
                for i in range(K):
                    d = episode_extra_stats(env_rec, agent_rec[i], K, cfg.use_obstacles)
                    assert sorted(k.replace(sname, "<scenario>") for k in d) == list(g["ep_keys"]), sorted(d)
                    ref_vals = dict(zip(("distance_to_goal_1s", "distance_to_goal_3s", "distance_to_goal_5s",
                                         "metric/agent_neighbor_col_rate", "metric/agent_obst_col_rate",
                                         f"{sname}/distance_to_goal_3s", f"{sname}/num_collisions"), det[i]))
                    for k, v in ref_vals.items():
                        assert abs(d[k] - v) <= 1e-9 * max(1.0, abs(v)), (s, i, k, d[k], v)
    assert n_done >= 1
    assert not ep_rows or len(ep_rows) == n_done
    if name in ("smallroom_k8", "crowd_k16", "cfg3_obst_k8"):
        assert n_impulse >= 1


# ------------------------------------------------------------------------------------------------------------------
# fork mode (quadrotor_multi_rewards.py: PID pre-controller, 8 control steps per call, capture task)
# ------------------------------------------------------------------------------------------------------------------
FORK_TRACE_NAMES = ["fork_k4", "fork_k1", "fork_k8_sangle", "fork_k4_cam", "fork_k6_cam_v2", "fork_k4_heading", "fork_k5_sheading_v3", "fork_k3_nself"]


def fork_cfg_from_kwargs(kw):
    kw = dict(kw)
    m = dict(num_agents=kw.pop("num_agents"), ep_time=kw.pop("episode_duration", 30.0))
    if "initial_capture_radius" in kw:
        m["capture_radius"] = kw.pop("initial_capture_radius")
    cam = {}
    if "pixel_noise_cam" in kw:
        cam["cam_pixel_noise"] = kw.pop("pixel_noise_cam")
    if "n_cameras" in kw:
        cam["cam_num"] = kw.pop("n_cameras")
    if cam:
        m["camera"] = cam
    m.update(kw)          # obs_repr / neighbor_obs_type / neighbor_visible_num carry the reference's names
    return QuadSimConfig.fork_default(num_envs=1, **m)


def test_fork_constants_match_survey_known_answers():
    """SURVEY.md Appendix A.2: mixer allocation and controller inertia of the reference."""
    from quad_swarm_rl_stable_baselines3_b200.fork_model import ForkParams
    p = ForkParams()
    s = 0.7071067811865476
    np.testing.assert_allclose(p.model.mixer(), [[-s, -s, -1, 1], [s, s, -1, 1], [s, -s, 1, 1], [-s, s, 1, 1]], atol=1e-12)
    np.testing.assert_allclose(p.model.inertia_diag(), [1.48072512e-05, 1.48072512e-05, 2.95725024e-05], rtol=1e-8)


@pytest.mark.parametrize("name", FORK_TRACE_NAMES)
def test_fork_env_trace(golden_dir, name):
    """QuadrotorEnvMulti.step (fork) + the VecEnv worker's auto-reset, every draw taped.  The full state (dynamics,
    12 PIDs, heading, evader) is re-synchronised to the reference before every call; the 8 control sub-steps inside a
    call, the episode bookkeeping and the capture-radius schedule free-run."""
    g = np.load(os.path.join(golden_dir, f"trace_{name}.npz"))
    cfg = fork_cfg_from_kwargs(ast.literal_eval(str(g["env_kwargs"])))
    K = cfg.num_agents
    o = OracleEnv(cfg)
    assert o.D == g["obs"].shape[2] and o.A == 2
    on, ou_ = np.cumsum(np.r_[0, g["n_tn"]]), np.cumsum(np.r_[0, g["n_tu"]])

    def tape(i):
        o.set_tape(g["tn"][on[i]:on[i + 1]], g["tu"][ou_[i]:ou_[i + 1]], None)

    def check(i, what):
        assert o.tape_pos()[:2] == (g["n_tn"][i], g["n_tu"][i]), (what, o.tape_pos(), g["n_tn"][i], g["n_tu"][i])
        st, fs = o.get_state(), o.get_fork_state()
        for k in PHYS:
            np.testing.assert_allclose(st[k].reshape(K, -1), g["s_" + k][i].reshape(K, -1), rtol=0, atol=2e-8, err_msg=f"{what} {k}")
        np.testing.assert_allclose(st["goal"], g["s_goal"][i], atol=1e-12, err_msg=f"{what} goal")
        np.testing.assert_allclose(fs["evader"], g["s_evader"][i], atol=1e-12, err_msg=f"{what} evader")
        np.testing.assert_allclose(fs["heading"][:, 0], g["s_angle"][i], atol=1e-12, err_msg=f"{what} angle")
        np.testing.assert_allclose(fs["heading"][:, 1], g["s_ang_vel"][i], atol=1e-12, err_msg=f"{what} ang_vel")
        np.testing.assert_allclose(fs["heading"][:, 2], g["s_heading"][i], atol=1e-12, err_msg=f"{what} self.heading")
        np.testing.assert_allclose(fs["pid"], g["s_pid"][i], rtol=1e-7, atol=1e-9, err_msg=f"{what} pid")
        assert st["tick"] == g["tick"][i], what

    def force(i):
        st = o.get_state()
        fl = st["flags"] & ~0xF
        for bit, key in enumerate(("on_floor", "crashed_floor", "crashed_wall", "crashed_ceiling")):
            fl |= g["s_" + key][i].astype(np.int32) << bit
        o.set_state(flags=fl, goal=g["s_goal"][i], **{k: g["s_" + k][i] for k in PHYS})
        o.set_fork_state(pid=g["s_pid"][i], heading=np.stack([g["s_angle"][i], g["s_ang_vel"][i], g["s_heading"][i]], axis=1),
                         evader=g["s_evader"][i])

    # the very first reset starts from the constructor state of the reference: drones at the origin, evader at (0, 0)
    tape(0)
    o.set_state(pos=np.zeros((K, 3)))
    obs = o.reset()
    check(0, "reset")
    np.testing.assert_allclose(obs, g["obs"][0], rtol=0, atol=1e-8)
    n_done = n_succ = 0
    for s in range(g["actions"].shape[0]):
        force(s)
        o.set_param(8, float(g["radius"][s]))                    # QS_PARAM_CAPTURE_RADIUS
        tape(s + 1)
        obs, rew, done, term = o.step(g["actions"][s], want_terminal=True)
        check(s + 1, f"step {s}")
        np.testing.assert_allclose(rew, g["rew"][s], rtol=0, atol=1e-9, err_msg=f"step {s} reward")
        assert np.array_equal(done, g["done"][s]), f"step {s} done"
        np.testing.assert_allclose(obs, g["obs"][s + 1], rtol=0, atol=2e-7, err_msg=f"step {s} obs")
        if done.any():
            np.testing.assert_allclose(term, g["term"][s], rtol=0, atol=2e-7, err_msg=f"step {s} terminal obs")
            assert o.last_reset_success == bool(g["success"][s]), f"step {s} reset_info['success']"
            n_done += 1
            n_succ += int(g["success"][s])
        else:
            assert o.last_reset_success is None and g["success"][s] == -1
    assert n_done >= 2 and n_succ == int((g["success"] == 1).sum())
    if name in ("fork_k4", "fork_k1", "fork_k8_sangle", "fork_k4_cam"):
        assert n_succ >= 1
    assert o.stats()["episodes"] == n_done and o.stats()["episodes_success"] == n_succ

