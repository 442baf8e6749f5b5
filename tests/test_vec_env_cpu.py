"""Host-side logic of the VecEnv facade (the drop-in for SubprocVecEnvCustom), driven on CPU through the oracle-backed
simulator of tests/oracle_sim.py: shapes, row order, infos / terminal_observation, reset_infos, env_method, buffers."""
import numpy as np
import pytest

from oracle_sim import OracleSim
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig
from quad_swarm_rl_stable_baselines3_b200.vec_env import QuadSwarmVecEnv, make_spaces


def test_spaces_match_reference_bounds():
    obs, act = make_spaces(QuadSimConfig(num_envs=1, num_agents=8))                # cfg2: 18 + 6*6
    assert obs.shape == (54,) and act.shape == (4,)
    np.testing.assert_allclose(obs.high[:6], [10, 10, 10, 3, 3, 3])
    np.testing.assert_allclose(obs.high[18:24], [10, 10, 10, 6, 6, 6])            # rxyz, rvxyz (quadrotor_single.py:295-296)
    f_obs, f_act = make_spaces(QuadSimConfig.fork_default(num_envs=1))
    assert f_obs.shape == (12,) and f_act.shape == (2,)
    np.testing.assert_allclose(f_obs.low[:6], [0, -3, -7.5, -3, -np.pi, -40], rtol=1e-6)   # quadrotor_single_rewards.py:329-340
    np.testing.assert_allclose(f_obs.high[6:8], [7.5, np.pi], rtol=1e-6)


def test_fork_vec_env_contract():
    cfg = QuadSimConfig.fork_default(num_envs=6, num_agents=4, ep_time=0.4, capture_radius=2.6, seed=3)
    env = QuadSwarmVecEnv(cfg, sim=OracleSim(cfg))
    N, K = 6, 4
    assert env.num_envs == N * K and env.agents_per_env == K and env.batch == 0
    obs0 = env.reset()
    assert obs0.shape == (N * K, 12) and obs0.dtype == np.float32
    assert len(env.reset_infos) == N and all(r == {"success": False} for r in env.reset_infos)
    rs = np.random.RandomState(0)
    seen_done = seen_success = 0
    prev = obs0
    for t in range(12):
        prev_copy = prev.copy()
        a = rs.uniform(-1, 1, (N * K, 2)).astype(np.float32)
        env.step_async(a)
        assert env.waiting
        obs, rew, done, infos = env.step_wait()
        assert not env.waiting
        assert np.array_equal(prev, prev_copy), "the previous observation array must survive one step (SB3 _last_obs)"
        assert obs.shape == (N * K, 12) and rew.shape == (N * K,) and done.shape == (N * K,) and done.dtype == np.bool_
        assert len(infos) == N * K and len(env.reset_infos) == N
        d2 = done.reshape(N, K)
        assert (d2.all(axis=1) == d2.any(axis=1)).all()                          # all agents of an env finish together
        for e in range(N):
            if d2[e, 0]:
                seen_done += 1
                assert set(env.reset_infos[e]) == {"success"}
                seen_success += int(env.reset_infos[e]["success"])
                for k in range(K):
                    assert infos[e * K + k]["terminal_observation"].shape == (12,)
                    assert "TimeLimit.truncated" not in infos[e * K + k]           # subproc_vec_env_custom.py:40
            else:
                assert env.reset_infos[e] is None and "terminal_observation" not in infos[e * K]
        prev = obs
    assert seen_done >= 3 and seen_success >= 1
    assert env.env_method("set_capture_radius", 0.25) == [None] * N
    assert env.get_attr("capture_radius", indices=[0, 2]) == [0.25, 0.25]
    assert env.get_attr("num_agents") == [K] * N and env.env_is_wrapped(object) == [False] * N
    with pytest.raises(AttributeError):
        env.env_method("no_such_method")
    with pytest.raises(ValueError):
        env.step_async(np.zeros((3, 2), np.float32))
    env.close()
    assert env.closed and env.sim.closed


def test_upstream_vec_env_matches_direct_oracle():
    cfg = QuadSimConfig(num_envs=3, num_agents=8, ep_time=0.1, seed=4)
    env = QuadSwarmVecEnv(cfg, sim=OracleSim(cfg))
    ref = OracleSim(cfg)
    np.testing.assert_array_equal(env.reset(), ref.reset_host())
    rs = np.random.RandomState(1)
    n_done = 0
    for t in range(14):
        a = rs.uniform(-1, 1, (24, 4)).astype(np.float32)
        obs, rew, done, infos = env.step(a)
        o2, r2, d2 = ref.step_host(a)
        np.testing.assert_array_equal(obs, o2); np.testing.assert_array_equal(rew, r2); np.testing.assert_array_equal(done, d2)
        if done.any():
            n_done += 1
            assert all(r == {} for r in env.reset_infos)
            # infos[i]['episode_extra_stats'] with the reference's keys (quadrotor_multi.py:739-831)
            for i in (0, 7, 23):
                es = infos[i]["episode_extra_stats"]
                assert {"num_collisions", "num_collisions_after_settle", "static_same_goal/num_collisions", "distance_to_goal_1s",
                        "static_same_goal/distance_to_goal_5s", "metric/agent_success_rate", "metric/agent_col_rate",
                        "static_same_goal/agent_deadlock_rate", "metric/agent_neighbor_col_rate"} <= set(es)
                assert "num_collisions_obst_quad" not in es
                assert abs(es["metric/agent_success_rate"] + es["metric/agent_deadlock_rate"] + es["metric/agent_col_rate"] - 1.0) < 1e-12
                assert es["distance_to_goal_1s"] > 0 and es["distance_to_goal_1s"] == es["static_same_goal/distance_to_goal_1s"]
            assert infos[0]["episode_extra_stats"]["distance_to_goal_1s"] != infos[1]["episode_extra_stats"]["distance_to_goal_1s"]
    assert n_done >= 1
    # the per-episode records add up to the rollout aggregate
    tot = env.sim.episode_stats()
    assert tot["episodes"] == n_done * cfg.num_envs


def test_mix_vec_env_infos_name_the_scenario_of_the_episode():
    cfg = QuadSimConfig(num_envs=6, num_agents=4, quads_mode="mix", neighbor_visible_num=2, ep_time=0.05, seed=9)
    env = QuadSwarmVecEnv(cfg, sim=OracleSim(cfg))
    env.reset()
    names = set()
    for t in range(40):
        obs, rew, done, infos = env.step(np.zeros((24, 4), np.float32))
        for e in np.flatnonzero(done.reshape(6, 4)[:, 0]):
            es = infos[e * 4]["episode_extra_stats"]
            prefixed = [k.split("/")[0] for k in es if k.endswith("/agent_success_rate") and not k.startswith("metric/")]
            assert len(prefixed) == 1
            names.add(prefixed[0])
    assert len(names) >= 5 and names <= {"static_same_goal", "static_diff_goal", "ep_lissajous3D", "ep_rand_bezier", "dynamic_same_goal",
                                         "dynamic_diff_goal", "dynamic_formations", "swap_goals", "swarm_vs_swarm"}


def test_episode_extra_stats_keys_with_obstacles():
    """The obstacle env adds the obstacle counters and names the scenario the episode actually ran (mix -> o_random | o_static_same_goal)."""
    cfg = QuadSimConfig(num_envs=2, num_agents=4, quads_mode="mix", use_obstacles=True, use_downwash=True, neighbor_visible_num=2,
                        obs_repr="xyz_vxyz_R_omega_floor", ep_time=0.05, seed=3)
    env = QuadSwarmVecEnv(cfg, sim=OracleSim(cfg))
    env.reset()
    seen = set()
    for t in range(30):
        obs, rew, done, infos = env.step(np.zeros((8, 4), np.float32))
        for e in np.flatnonzero(done.reshape(2, 4)[:, 0]):
            es = infos[e * 4 + 1]["episode_extra_stats"]
            name = [k.split("/")[0] for k in es if k.endswith("/num_collisions_obst")][0]
            seen.add(name)
            assert {"num_collisions_obst_quad", "num_collisions_obst_quad_after_settle", f"{name}/num_collisions_obst_quad_3_5",
                    "num_collisions_obst_quad_5", "metric/agent_obst_col_rate", f"{name}/agent_obst_col_rate"} <= set(es)
    assert seen and seen <= {"o_random", "o_static_same_goal"}


def test_reward_coefficient_annealing_hook():
    """AnnealSchedule / anneal_reward_coefficients = the annealing branch of QuadsRewardShapingWrapper (reward_shaping.py:109-118)."""
    from quad_swarm_rl_stable_baselines3_b200.vec_env import AnnealSchedule
    cfg = QuadSimConfig(num_envs=1, num_agents=8, seed=4, rew_coeff=dict(quadcol_bin=0.0, quadcol_bin_smooth_max=0.0))
    env = QuadSwarmVecEnv(cfg, sim=OracleSim(cfg))
    env.reset()
    sched = [AnnealSchedule("quadcol_bin", 5.0, 1000.0), AnnealSchedule("quadcol_bin_smooth_max", 10.0, 1000.0)]
    assert env.anneal_reward_coefficients(250.0, sched) == {"z_anneal_quadcol_bin": 1.25, "z_anneal_quadcol_bin_smooth_max": 2.5}
    assert env.anneal_reward_coefficients(4000.0, sched) == {"z_anneal_quadcol_bin": 5.0, "z_anneal_quadcol_bin_smooth_max": 10.0}
    # the coefficients reach the simulator: drones spawn within the proximity fall-off of each other often enough that the
    # smooth penalty changes the reward of the very next step
    ref = OracleSim(cfg)
    ref.reset_host()
    a = np.zeros((8, 4), np.float32)
    r_env = env.step(a)[1]
    r_ref = ref.step_host(a)[1]
    assert (r_env <= r_ref + 1e-9).all()
