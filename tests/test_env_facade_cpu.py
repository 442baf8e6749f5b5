"""The `QuadrotorEnvMulti`-shaped drop-in (quad_swarm_rl_stable_baselines3_b200/env.py) and the SB3 VecEnv claim, on CPU through
the oracle-backed simulator of tests/oracle_sim.py."""
import importlib

import numpy as np
import pytest

import sb3_stub
from oracle_sim import OracleSim
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig
from quad_swarm_rl_stable_baselines3_b200.env import QuadrotorEnvMulti, SB3QuadrotorEnv, reward_info_dict

REW_KEYS = {"rew_main", "rew_pos", "rew_action", "rew_crash", "rew_orient", "rew_spin", "rewraw_main", "rewraw_pos", "rewraw_action",
            "rewraw_crash", "rewraw_orient", "rewraw_spin", "rew_quadcol", "rew_proximity", "rewraw_quadcol"}


def upstream_env(**kw):
    cfg = QuadSimConfig(num_envs=1, num_agents=kw.pop("num_agents", 8), ep_time=kw.pop("ep_time", 0.2), seed=5, **kw)
    return QuadrotorEnvMulti(cfg, sim=OracleSim(cfg)), cfg


def test_upstream_env_api_shape_and_reward_breakdown():
    env, cfg = upstream_env()
    K, D = 8, 54
    assert env.num_agents == K and env.observation_space.shape == (D,) and env.action_space.shape == (4,)
    obs, info = env.reset()
    assert isinstance(obs, np.ndarray) and obs.shape == (K, D) and obs.dtype == np.float64 and info == {}
    rs = np.random.RandomState(0)
    n_done = 0
    for t in range(45):
        a = rs.uniform(-1, 1, (K, 4))
        obs, rewards, dones, infos = env.step(a)
        assert obs.shape == (K, D) and isinstance(rewards, list) and isinstance(dones, list) and isinstance(infos, list)
        assert len(rewards) == len(dones) == len(infos) == K and all(isinstance(d, bool) for d in dones)
        assert len({id(i) for i in infos}) == K
        for i in range(K):
            r = infos[i]["rewards"]
            assert set(r) == REW_KEYS
            total = r["rew_pos"] + r["rew_action"] + r["rew_crash"] + r["rew_orient"] + r["rew_spin"] + r["rew_quadcol"] + r["rew_proximity"]
            assert abs(total - rewards[i]) < 1e-6, (total, rewards[i])
            assert r["rewraw_pos"] <= 0 and r["rew_main"] == r["rew_pos"] and r["rewraw_quadcol"] in (0.0, -1.0)
        if dones[0]:
            n_done += 1
            assert all(dones)
            st = infos[0]["episode_extra_stats"]
            assert "num_collisions" in st and "metric/agent_success_rate" in st and "static_same_goal/distance_to_goal_1s" in st
            assert env.envs[0].tick == 0                       # the upstream env has already reset itself (quadrotor_multi.py:836)
        else:
            assert "episode_extra_stats" not in infos[0]
    assert n_done == 2
    env.close()


def test_dynamics_views_and_set_state():
    env, cfg = upstream_env(num_agents=3, neighbor_visible_num=2)
    env.reset()
    d = env.envs[1].dynamics
    assert d.pos.shape == (3,) and d.vel.shape == (3,) and d.rot.shape == (3, 3) and d.omega.shape == (3,)
    assert len(env.all_dynamics()) == 3
    np.testing.assert_allclose(env.envs[1].goal, [0, 0, 2])
    d.set_state(np.array([0.5, -0.5, 3.0]), np.zeros(3), np.eye(3), np.zeros(3))     # raw_test.py:39-42
    np.testing.assert_allclose(env.envs[1].dynamics.pos, [0.5, -0.5, 3.0])
    p0 = env.envs[0].dynamics.pos.copy()
    env.step(np.zeros((3, 4)))
    assert not np.array_equal(env.envs[0].dynamics.pos, p0)                          # views are refreshed after a step
    assert abs(env.envs[1].dynamics.pos[2] - 3.0) < 0.01


def test_fork_env_episode_boundary_matches_the_worker_protocol():
    """step() on the last step returns the finished episode's last observation and does not reset; the reset() that the VecEnv
    worker issues next (subproc_vec_env_custom.py:43-46) returns the new episode's first observation with {"success": ...}."""
    cfg = QuadSimConfig.fork_default(num_envs=1, num_agents=4, ep_time=0.4, capture_radius=2.6, seed=3)
    sim = OracleSim(cfg)
    calls = dict(reset=0)
    orig = sim.reset_host
    sim.reset_host = lambda: (calls.__setitem__("reset", calls["reset"] + 1), orig())[1]
    env = SB3QuadrotorEnv(cfg, sim=sim)
    obs, info = env.reset(seed=1, options=None)
    assert obs.shape == (4, 12) and info == {"success": False} and calls["reset"] == 1
    rs = np.random.RandomState(0)
    finished = successes = 0
    for t in range(40):
        obs, rew, term, trunc, infos = env.step(rs.uniform(-1, 1, (4, 2)))
        assert term == trunc and len(infos) == 4
        if term[0]:
            finished += 1
            terminal = obs.copy()
            np.testing.assert_array_equal(terminal, sim_term(env))
            obs2, info = env.reset()
            successes += int(info["success"])
            assert set(info) == {"success"} and obs2.shape == (4, 12) and not np.array_equal(obs2, terminal)
            assert calls["reset"] == 1, "the kernel already reset the env inside the step: no second reset"
    assert finished >= 2 and successes >= 1
    env.set_capture_radius(0.3)
    assert env.env.capture_radius == 0.3


def sim_term(env):
    return env.env._term.astype(np.float64)


def test_constructor_accepts_the_upstream_keyword_arguments():
    """quadrotor_multi.py:27-45 as called by make_quadrotor_env_multi (quad_utils.py:36-66): rendering / numba / replay arguments
    are accepted and ignored."""
    import types
    sim_cfg = QuadSimConfig(num_envs=1, num_agents=4, neighbor_visible_num=2, ep_time=0.3)
    env = QuadrotorEnvMulti(
        cfg=types.SimpleNamespace(seed=0), sim=OracleSim(sim_cfg), num_agents=4, ep_time=0.3, rew_coeff=None, obs_repr="xyz_vxyz_R_omega",
        neighbor_visible_num=2, neighbor_obs_type="pos_vel", collision_hitbox_radius=2.0, collision_falloff_radius=4.0,
        use_obstacles=False, obst_density=0.2, obst_size=0.6, obst_spawn_area=[8.0, 8.0], use_downwash=False, use_numba=True,
        quads_mode="static_same_goal", room_dims=(10.0, 10.0, 10.0), use_replay_buffer=False, quads_view_mode=["topdown"],
        quads_render=False, dynamics_params="Crazyflie", raw_control=True, raw_control_zero_middle=True,
        dynamics_randomize_every=None, dynamics_change=None, dyn_sampler_1=None, sense_noise="default", init_random_state=False)
    assert env.num_agents == 4 and env.cfg.obs_dim == 18 + 12
    obs, _ = env.reset()
    assert obs.shape == (4, 30)


def test_reward_info_dict_weights():
    row = [-0.01, -0.005, -0.005, 0.004, -0.02, -1.0, -0.03, -1.0]
    rc = dict(pos=1.0, effort=0.05, crash=1.0, orient=1.0, spin=0.1, quadcol_bin=5.0, quadcol_bin_smooth_max=10.0, quadcol_bin_obst=5.0)
    r = reward_info_dict(row, rc, use_obstacles=True)
    assert r["rew_action"] == pytest.approx(0.05 * -0.005) and r["rew_quadcol"] == -5.0 and r["rew_quadcol_obstacle"] == -5.0
    assert r["rew_proximity"] == pytest.approx(-0.03) and r["rewraw_quadcol_obstacle"] == -1.0


def test_sb3_vec_env_abc_and_rollout_access_patterns():
    """`QuadSwarmVecEnv` under (a stand-in for) SB3's VecEnv ABC: it instantiates (no abstract method left), and the rollout /
    VecMonitor / curriculum access patterns of tests/sb3_stub.py run on it -- including in-place writes into infos[i]."""
    added = sb3_stub.install()
    import quad_swarm_rl_stable_baselines3_b200.vec_env as ve
    try:
        ve = importlib.reload(ve)
        assert ve._SB3VecEnv is sb3_stub.VecEnv and issubclass(ve.QuadSwarmVecEnv, sb3_stub.VecEnv)
        for cfg, act_dim in ((QuadSimConfig.fork_default(num_envs=5, num_agents=4, ep_time=0.4, capture_radius=2.6, seed=3), 2),
                             (QuadSimConfig(num_envs=3, num_agents=8, ep_time=0.15, seed=4), 4)):
            env = ve.QuadSwarmVecEnv(cfg, sim=OracleSim(cfg))
            policy = lambda obs, rng, A=act_dim: rng.uniform(-1.5, 1.5, (obs.shape[0], A)).astype(np.float32)   # noqa: E731
            buf, log = sb3_stub.collect_rollouts(env, 24, policy, np.random.RandomState(0))
            assert buf.pos == 24 and np.isfinite(buf.obs).all() and np.isfinite(buf.rewards).all()
            assert log["episodes"] >= cfg.num_envs * cfg.num_agents and log["terminal_obs"] == log["episodes"]
            assert log["reset_infos"] * cfg.num_agents == log["episodes"]
            assert env.get_attr("num_agents") == [cfg.num_agents] * cfg.num_envs and env.env_is_wrapped(object) == [False] * cfg.num_envs
            env.close()
    finally:
        sb3_stub.uninstall(added)
        importlib.reload(ve)
