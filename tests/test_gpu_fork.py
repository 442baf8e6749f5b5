"""Fork mode (the env swarm_rl/sb_train.py trains on) on the GPU, through the C-ABI, against the CPU oracle.

One call = 8 control steps (PID cascade + mixer + dynamics + capture bookkeeping + evader motion), so the north-star
tolerance "relative error <= 1e-5 on pos/vel/rot/omega after one step" is applied per control step: <= 8e-5 after a
call with the natural scale (1 m, 1 m/s, 1, 1 rad/s) as floor -- measured values are printed.  Flags, dones,
reset_info["success"] and neighbour slots are exact away from threshold ties.
"""
import os
import re
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from oracle import OracleEnv  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402

QS_ER_EP_LEN, QS_ER_SUCCESS, QS_ER_NONFINITE = 16, 17, 18       # include/quadsim.h

PHYS = ("pos", "vel", "rot", "omega", "rot_damp", "cmds_damp", "ou")
FORK_CONFIGS = {
    "fork_k4": dict(num_envs=40, num_agents=4, ep_time=0.48, capture_radius=2.6),
    "fork_k1": dict(num_envs=50, num_agents=1, ep_time=0.4, capture_radius=2.4, neighbor_obs_type="none", neighbor_visible_num=0),
    "fork_k8_sangle": dict(num_envs=16, num_agents=8, ep_time=0.4, capture_radius=2.2,
                           obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot", neighbor_obs_type="dist_sangle",
                           neighbor_visible_num=3),
    "fork_k3_aw": dict(num_envs=11, num_agents=3, ep_time=0.4, capture_radius=0.3, obs_repr="aw_awdot_dist_distdot_angle_angledot"),
    # sb_train.py:122-137 (the author's current sweep): camera-model neighbour observations; pixel noise on here
    "fork_k4_cam": dict(num_envs=24, num_agents=4, ep_time=0.4, capture_radius=2.4, neighbor_obs_type="ndist_nsangle",
                        obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot"),
    "fork_k6_cam_v2": dict(num_envs=12, num_agents=6, ep_time=0.4, capture_radius=2.2, neighbor_obs_type="ndist_nsangle",
                           neighbor_visible_num=2, camera=dict(cam_pixel_noise=1.0, cam_num=4)),
    "fork_k3_nself": dict(num_envs=20, num_agents=3, ep_time=0.4, capture_radius=2.3, neighbor_obs_type="ndist_nsangle",
                          obs_repr="cdist_cdistdot_ndist_distdot_nsangle_angledot", camera=dict(cam_pixel_noise=0.7)),
    "fork_k4_heading": dict(num_envs=16, num_agents=4, ep_time=0.4, capture_radius=2.4, neighbor_obs_type="dist_angle_heading"),
    "fork_k5_sheading_v3": dict(num_envs=10, num_agents=5, ep_time=0.4, capture_radius=2.2, neighbor_obs_type="dist_sangle_sheading",
                                neighbor_visible_num=3, obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot"),
    # lane-group widths 2, 16 and 32 (K = 12 leaves padding lanes); ranked neighbour rows (V < K - 1) at 4, 16 and 32 lanes, rows
    # of all others at 8
    "fork_k2": dict(num_envs=30, num_agents=2, ep_time=0.4, capture_radius=2.4),
    "fork_k12_sangle_v5": dict(num_envs=8, num_agents=12, ep_time=0.4, capture_radius=2.2, obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot",
                               neighbor_obs_type="dist_sangle", neighbor_visible_num=5),
    "fork_k16_cam": dict(num_envs=6, num_agents=16, ep_time=0.4, capture_radius=2.2, neighbor_obs_type="ndist_nsangle",
                         obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot"),
    "fork_k32_v20": dict(num_envs=5, num_agents=32, ep_time=0.4, capture_radius=2.2, neighbor_visible_num=20),
    "fork_k32_all": dict(num_envs=5, num_agents=32, ep_time=0.4, capture_radius=2.2),
    "fork_k3_v1": dict(num_envs=16, num_agents=3, ep_time=0.4, capture_radius=2.4, neighbor_visible_num=1),
    "fork_k7": dict(num_envs=10, num_agents=7, ep_time=0.4, capture_radius=2.2),
}


def _sim(cfg):
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    return QuadSwarmSim(cfg, device="cuda:0")


def relerr(a, b, floor):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def make_pair(name, seed=5):
    cfg = QuadSimConfig.fork_default(seed=seed, **FORK_CONFIGS[name])
    return cfg, _sim(cfg), [OracleEnv(cfg, i) for i in range(cfg.num_envs)]


def ranking_tie(cfg, o):
    """True if the neighbour ranking of this env is decided below fp32 resolution: two candidates of some drone have
    ranking metrics (norm of the feature row, quadrotor_multi_rewards.py:455-457) within 2e-6 of each other.  Happens
    right after a reset when the chasers sit millimetres apart (dist_sangle rows have norm sqrt(d^2 + 1))."""
    K = cfg.num_agents
    if cfg.visible >= K - 1 or cfg.visible == 0:
        return False
    pos = o.get_state()["pos"]
    ang = o.get_fork_state()["heading"][:, 0]
    hsn = o.get_fork_state()["heading"][:, 2]
    return_camera = False
    for i in range(K):
        mets = []
        for j in range(K):
            if j == i:
                continue
            d = pos[j] - pos[i]
            dist = np.linalg.norm(d)
            a = (np.arctan2(d[1], d[0]) - ang[i] + np.pi) % (2 * np.pi) - np.pi
            hd = (hsn[j] - hsn[i] + np.pi) % (2 * np.pi) - np.pi
            t = cfg.neighbor_obs_type
            if t == "ndist_nsangle":
                return_camera = True
                row = [min(dist, 10.0), 1.0]         # |(l, cos, sin)| = sqrt(l^2 + 1); l ~ dist up to the pixel noise
            else:
                row = {"dist_angle": [dist, a], "dist_sangle": [dist, np.cos(a), np.sin(a)],
                       "dist_angle_heading": [dist, a, hd],
                       "dist_sangle_sheading": [dist, np.cos(a), np.sin(a), np.cos(hd), np.sin(hd)]}[t]
            mets.append(max(np.linalg.norm(row), 0.01))
        mets = np.sort(mets)
        # camera rows carry pixel noise (amplified ~dist^2/(r f) px) and the disc degenerates below its radius: only call
        # the ranking decided when the candidates are clearly separated
        tol = 5e-3 if return_camera else 2e-6
        if np.any(np.diff(mets) < tol * mets[1:]):
            return True
    return False


def push_state(sim, oracles, cfg):
    st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
    K = cfg.num_agents
    for e, o in enumerate(oracles):
        sl = slice(e * K, (e + 1) * K)
        o.set_state(**{k: st[k][sl].astype(np.float64) for k in PHYS}, goal=st["goal"][sl].astype(np.float64),
                    flags=st["flags"][sl] & 0xFF, col_mask=st["col_mask"][sl].astype(np.uint32),
                    tick=int(st["tick"][e]), svd_ctr=int(st["svd_ctr"][e]), step_ctr=int(st["step_ctr"][e]))
        o.set_fork_state(pid=st["pid"][sl].astype(np.float64), heading=st["heading"][sl].astype(np.float64),
                         evader=st["evader"][e].astype(np.float64))
    return st


@pytest.mark.parametrize("name", list(FORK_CONFIGS))
def test_fork_reset_parity(name):
    cfg, sim, oracles = make_pair(name)
    assert sim.A == 2 and sim.D == cfg.obs_dim == oracles[0].D
    obs = sim.reset().cpu().numpy()
    ref = np.concatenate([o.reset() for o in oracles])
    st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
    for k in ("pos", "goal", "rot"):
        np.testing.assert_allclose(st[k], np.concatenate([o.get_state()[k].reshape(cfg.num_agents, -1) for o in oracles]), atol=2e-6, err_msg=k)
    np.testing.assert_allclose(st["evader"], np.stack([o.get_fork_state()["evader"] for o in oracles]), atol=2e-6)
    np.testing.assert_allclose(st["heading"], np.concatenate([o.get_fork_state()["heading"] for o in oracles]), atol=2e-6)
    K = cfg.num_agents
    S = 7 if "sangle" in cfg.obs_repr else 6
    np.testing.assert_allclose(obs[:, :S], ref[:, :S], atol=5e-5)                      # self block: always
    ok = np.repeat([not ranking_tie(cfg, o) for o in oracles], K)
    assert ok.sum() >= len(ok) // 2 or cfg.neighbor_obs_type == "ndist_nsangle"       # (camera rows of mm-apart drones: all ties)
    np.testing.assert_allclose(obs[ok], ref[ok], atol=5e-4)      # bearings between drones millimetres apart, see test_fork_step_parity
    # second reset: the evader's first step now sees the chasers (dynamic_repulsive.py:44)
    obs = sim.reset().cpu().numpy()
    ref = np.concatenate([o.reset() for o in oracles])
    ok = np.repeat([not ranking_tie(cfg, o) for o in oracles], K)
    np.testing.assert_allclose(obs[ok], ref[ok], atol=5e-4)


def new_tally():
    return dict(worst=dict(pos=0.0, vel=0.0, rot=0.0, omega=0.0, pid=0.0, obs=0.0, nbr=0.0), done=0, succ=0, tie=0, rank_tie=0)


def compare_fork_call(cfg, oracles, a, out, st, s, t):
    """One call of the fork kernel against the oracles, which held the kernel's state before it (push_state): every oracle steps
    with its env's actions `a` and is compared with `out` = (obs, rew, done, terminal_obs, reset_success) and the state `st`
    after the call (host arrays over the compared envs).  Errors and events go into the tally `t` (new_tally())."""
    K, D = cfg.num_agents, cfg.obs_dim
    obs, rew, done, term, succ = out
    worst = t["worst"]
    S = 7 if "sangle" in cfg.obs_repr else 6
    for e, o in enumerate(oracles):
        sl = slice(e * K, (e + 1) * K)
        r_obs, r_rew, r_done, r_term = o.step(a[sl].astype(np.float64), want_terminal=True)
        os_, fs = o.get_state(), o.get_fork_state()
        if r_done.any() != done[sl].any():
            # capture-threshold tie: some |goal - pos| within fp32 round-off of the radius in one of the sub-steps
            t["tie"] += 1
            continue
        assert np.array_equal(done[sl], r_done), (s, e)
        np.testing.assert_allclose(rew[sl], r_rew, atol=1e-5, err_msg=f"step {s} env {e} reward")
        if r_done.any():
            t["done"] += 1
            assert bool(succ[e]) == bool(o.last_reset_success), (s, e)
            t["succ"] += int(succ[e])
            np.testing.assert_allclose(term[sl][:, :S], r_term[:, :S], atol=2e-4, err_msg=f"step {s} env {e} terminal obs")
            # camera-model distances l carry the fp32 round-off of the ray slopes amplified by l^2 / (2 r), see check_fork_tally
            np.testing.assert_allclose(term[sl][:, S:], r_term[:, S:], atol=5e-3 if cfg.neighbor_obs_type == "ndist_nsangle" else 2e-4,
                                       err_msg=f"step {s} env {e} terminal obs, neighbour block")
            # chasers respawn on a ring of radius U(0, 0.5): neighbour bearings atan2(dy, dx) of drones a few mm apart
            # amplify the fp32 rounding of the positions (1e-8 m) by 1/distance
            pp = o.get_state()["pos"]
            dmin = min([np.linalg.norm(pp[a_] - pp[b]) for a_ in range(K) for b in range(a_ + 1, K)], default=1.0)
            # bearing error ~ 1e-8 m / distance: compare the neighbour block only when the respawn ring is not degenerate
            cols = slice(0, S) if (ranking_tie(cfg, o) or dmin < 2e-3) else slice(0, D)
            np.testing.assert_allclose(obs[sl][:, cols], r_obs[:, cols], atol=5e-4, err_msg=f"step {s} env {e} reset obs")
            continue
        for k, floor in (("pos", 1.0), ("vel", 1.0), ("rot", 1.0), ("omega", 1.0)):
            worst[k] = max(worst[k], relerr(st[k][sl], os_[k].reshape(K, -1), floor))
        worst["pid"] = max(worst["pid"], relerr(st["pid"][sl], fs["pid"], 1.0))
        cols = slice(0, S) if ranking_tie(cfg, o) else slice(0, D)
        t["rank_tie"] += cols.stop != D
        worst["obs"] = max(worst["obs"], relerr(obs[sl][:, :S], r_obs[:, :S], 1.0))
        # Neighbour rows hold bearings atan2(dy, dx) (or their sin / cos) of the other chasers: fp32 round-off of the two
        # positions (<= 4 ulp at the room scale, ~1e-6 m) turns into 1e-6 / distance radians.  Episodes start with the chasers a few
        # millimetres apart, so the bound is conditioned on the closest pair of the env; at >= 5 mm it is the flat 2e-4.
        pp = os_["pos"].reshape(K, -1)
        dmin = min([np.linalg.norm(pp[a_, :2] - pp[b, :2]) for a_ in range(K) for b in range(a_ + 1, K)], default=1.0)
        err_nbr = relerr(obs[sl][:, cols], r_obs[:, cols], 1.0)
        if cfg.neighbor_obs_type != "ndist_nsangle":
            assert err_nbr <= 2e-4 + 1e-6 / max(dmin, 1e-9), (s, e, err_nbr, dmin)
            err_nbr = min(err_nbr, 2e-4) if dmin < 5e-3 else err_nbr
        worst["nbr"] = max(worst["nbr"], err_nbr)
        assert st["tick"][e] == os_["tick"], (s, e)
        np.testing.assert_allclose(st["evader"][e], fs["evader"], atol=5e-6)


def check_fork_tally(name, cfg, t):
    worst = t["worst"]
    print(f"\n[{name}] worst rel err after one call (8 control steps): {worst}  dones={t['done']} captures={t['succ']} ties={t['tie']} "
          f"ranking-tie env-steps={t['rank_tie']}")
    assert t["done"] >= 3 and t["tie"] <= 2
    assert max(worst[k] for k in ("pos", "vel", "rot", "omega")) <= 8e-5
    assert worst["obs"] <= 2e-4
    # neighbour block.  The camera model measures distance as l = r / sin(alpha / 2) from the angle alpha between two tangent
    # rays (r = 0.1 m): dl = l^2 / (2 r) d(alpha), i.e. fp32 round-off of the ray slopes (4e-7) becomes 2e-3 m at l = 10 m --
    # three orders of magnitude below what one pixel of the model's own noise does there (3 m).
    assert worst["nbr"] <= (5e-3 if cfg.neighbor_obs_type == "ndist_nsangle" else 2e-4)


@pytest.mark.parametrize("name,steps", [("fork_k4", 60), ("fork_k1", 40), ("fork_k8_sangle", 40), ("fork_k3_aw", 40),
                                        ("fork_k4_cam", 40), ("fork_k6_cam_v2", 40), ("fork_k4_heading", 40), ("fork_k5_sheading_v3", 40),
                                        ("fork_k2", 40), ("fork_k12_sangle_v5", 40), ("fork_k16_cam", 40), ("fork_k32_v20", 40),
                                        ("fork_k32_all", 40), ("fork_k3_v1", 40), ("fork_k7", 40)])
def test_fork_step_parity(name, steps):
    import torch
    cfg, sim, oracles = make_pair(name)
    N, K = cfg.num_envs, cfg.num_agents
    sim.reset()
    for o in oracles:
        o.reset()
    rs = np.random.RandomState(11)
    t = new_tally()
    for s in range(steps):
        if s == steps // 2:
            sim.set_capture_radius(0.9)
            for o in oracles:
                o.set_param(8, 0.9)
        if re.search(r"_v\d+$", name):
            # fewer than K-1 neighbours visible: spread the chasers of freshly reset envs over metres (they respawn within
            # millimetres of each other, where every ranking metric ties) so that the ranking is actually decided
            stt = sim.get_state(["tick", "pos"])
            fresh = np.repeat(stt["tick"].cpu().numpy() == 0, K)
            if fresh.any():
                pos = stt["pos"].cpu().numpy()
                pos[fresh, :2] = rs.uniform(-3.0, 3.0, (int(fresh.sum()), 2))
                sim.set_state(pos=pos)
        push_state(sim, oracles, cfg)
        a = rs.uniform(-1.0, 1.0, (N * K, 2)).astype(np.float32)
        out = tuple(x.cpu().numpy() for x in sim.step(torch.from_numpy(a).cuda())) + \
            (sim.terminal_obs.cpu().numpy(), sim.reset_success.cpu().numpy())
        st = {k: v.cpu().numpy() for k, v in sim.get_state().items()}
        compare_fork_call(cfg, oracles, a, out, st, s, t)
    check_fork_tally(name, cfg, t)
    gs, osum = sim.episode_stats(), [o.stats() for o in oracles]
    if t["tie"] == 0:
        for k in ("episodes", "episodes_success", "num_collisions", "num_collisions_with_floor", "num_collisions_with_wall"):
            assert gs[k] == sum(x[k] for x in osum), k


def test_fork_parity_at_benchmarked_launch_shape(monkeypatch):
    """The fork env at the launch shape `bench.py --workload fork` times (65536 envs x 4 chasers, 128-thread blocks): whole sampled
    warp-tiles, the first and the last of the grid among them, teacher-forced against one oracle each (keyed by the env's global
    index) for 40 calls, with the clocks staggered so that timeouts fall on every sub-step.  Over the whole batch, every call:
    done, terminal_obs, reset_success and the episode records are written for the envs that ended and only for those
    (ForkCheckedSim), and some warp-tiles had a group end on a sub-step before the last while others of the tile went on."""
    import dataclasses
    import torch
    from test_gpu_staggered import CheckedSim, envs_per_tile

    class ForkCheckedSim(CheckedSim):
        """The fork's done rule: an env ends on a capture (reset_success 1, recorded length = the sub-steps it ran) or on its clock
        (reset_success 0, recorded length ep_len + 1); an env that goes on ran all sub-steps of the call."""

        def ended(self, tick0, rec1):
            sim, N, K, sub = self.sim, self.sim.N, self.K, cfg.fork.substeps
            dn = sim.done.view(N, K)
            end = dn[:, 0]
            assert torch.equal(dn, end[:, None].expand(N, K)), "the agents of an env end together"
            tick1 = sim.get_state(("tick",))["tick"]
            assert bool((tick1[~end] == tick0[~end] + sub).all()) and bool((tick0[~end] + sub <= self.ep_len).all()), "env went on"
            assert bool((tick1[end] == 0).all())
            succ, rec = sim.reset_success[end].int(), rec1["env"][end]
            ran = rec[:, QS_ER_EP_LEN] - tick0[end]
            assert torch.equal(succ, rec[:, QS_ER_SUCCESS]), "reset_success differs from the episode record"
            caught, timed_out = succ == 1, succ == 0
            assert bool((caught | timed_out).all()) and int(rec[:, QS_ER_NONFINITE].sum()) == 0
            assert bool(((ran >= 1) & (ran <= sub)).all()), "recorded episode length"
            assert bool((rec[timed_out, QS_ER_EP_LEN] == self.ep_len + 1).all()), "an env ended neither captured nor on its clock"
            # warp-tiles in which a group ended on a sub-step before the last while another group went on
            early = torch.zeros(N, dtype=torch.bool, device=end.device)
            early[end] = ran < sub
            n_t = -(-N // self.gpw)
            pad = n_t * self.gpw - N
            e_t = torch.cat([early, early.new_zeros(pad)]).view(n_t, self.gpw).any(dim=1)
            c_t = torch.cat([~end, end.new_zeros(pad)]).view(n_t, self.gpw).any(dim=1)
            self.idle_tiles += int((e_t & c_t).sum())
            self.early_captures += int((caught & (ran < sub)).sum())
            return end

    cfg = QuadSimConfig.fork_default(num_envs=65536, ep_time=0.8, capture_radius=2.6, seed=37)
    N, K, L, gpw = cfg.num_envs, cfg.num_agents, cfg.ep_len, envs_per_tile(cfg.num_agents)
    monkeypatch.setenv("QS_BLOCK", "128")
    sim = _sim(cfg)
    monkeypatch.delenv("QS_BLOCK")
    n_tiles = -(-N // gpw)
    rs = np.random.RandomState(4)
    tiles = np.concatenate([[0], np.sort(rs.choice(np.arange(1, n_tiles - 1), 30, replace=False)), [n_tiles - 1]])
    idx = (tiles[:, None] * gpw + np.arange(gpw)[None, :]).reshape(-1)
    oracles = [OracleEnv(cfg, int(i)) for i in idx]
    sim.reset()
    for o in oracles:
        o.reset()
    wrap = ForkCheckedSim(sim, idx, seed=6)
    wrap.idle_tiles = wrap.early_captures = 0
    wrap.set_ticks(rs.randint(0, L, N))
    small = dataclasses.replace(cfg, num_envs=len(idx))
    t = new_tally()
    for s in range(40):
        push_state(wrap, oracles, small)
        a = rs.uniform(-1.0, 1.0, (len(idx) * K, 2)).astype(np.float32)
        out = tuple(x.cpu().numpy() for x in wrap.step(torch.from_numpy(a).cuda())) + \
            (wrap.terminal_obs.cpu().numpy(), sim.reset_success[wrap.env_idx].cpu().numpy())
        st = {k: v.cpu().numpy() for k, v in wrap.get_state().items()}
        compare_fork_call(small, oracles, a, out, st, s, t)
    print(f"[fork_65536x4] mixed tiles {wrap.mixed} over {len(tiles)} compared tiles; warp-tiles with a group that ended before the "
          f"last sub-step next to one that went on: {wrap.idle_tiles}; captures before the last sub-step {wrap.early_captures}")
    check_fork_tally("fork_65536x4", small, t)
    assert t["done"] >= len(idx) and t["succ"] > 0
    assert wrap.mixed >= len(tiles) and wrap.idle_tiles >= N // gpw and wrap.early_captures > 0


def test_fork_host_path_and_reset_info():
    """qs_step_host in fork mode: numpy in / numpy out incl. terminal observation and reset_info['success']."""
    import torch
    cfg = QuadSimConfig.fork_default(num_envs=64, num_agents=4, ep_time=0.24, capture_radius=3.0, seed=9)
    a_sim, b_sim = _sim(cfg), _sim(cfg)
    a_sim.reset(); b_sim.reset_host()
    rs = np.random.RandomState(2)
    n = cfg.num_envs * cfg.num_agents
    term = np.zeros((n, cfg.obs_dim), np.float32)
    succ = np.full(cfg.num_envs, 7, np.uint8)
    seen = 0
    for s in range(6):
        a = rs.uniform(-1, 1, (n, 2)).astype(np.float32)
        o1, r1, d1 = a_sim.step(torch.from_numpy(a).cuda())
        o2, r2, d2 = b_sim.step_host(a, terminal_obs=term, reset_success=succ)
        assert np.array_equal(o1.cpu().numpy(), o2) and np.array_equal(r1.cpu().numpy(), r2) and np.array_equal(d1.cpu().numpy(), d2)
        env_done = d2.reshape(cfg.num_envs, cfg.num_agents)[:, 0]
        if env_done.any():
            seen += int(env_done.sum())
            rows = np.repeat(env_done, cfg.num_agents)
            assert np.array_equal(term[rows], a_sim.terminal_obs.cpu().numpy()[rows])
            assert np.array_equal(succ[env_done], a_sim.reset_success.cpu().numpy()[env_done])
            assert set(np.unique(succ[env_done])) <= {0, 1}
    assert seen > 0
