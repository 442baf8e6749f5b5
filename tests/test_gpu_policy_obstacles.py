"""Fused tcgen05 policy forward with the obstacle encoder (csrc/policy_kernels.cu, variant OB; include/quadpolicy.h version 2) against the
torch module it replaces (`ppo.QuadEncoder` with `obstacle`: 9 SDF inputs -> 256 -> 256, tanh, feed-forward input [self | neighbour mean |
obstacle]; reference: swarm_rl/models/quad_multi_model.py:250-354).

Two references, both plain PyTorch, with the tolerances of tests/test_gpu_policy.py:
  * fp32: the module as it is;
  * bf16-emulated: the module with weights and layer inputs rounded to bf16 where the kernel rounds them, obstacle encoder included.
The obstacle columns are drawn at another scale than the rest of the row (positive, like the SDF distances), so a wrong column offset
cannot pass.
"""
import ctypes as C
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402

TOL_FP32_MAX = 3e-2
TOL_FP32_RMS = 6e-3
TOL_EMU_MAX = 3e-3


def cfg3(**kw):
    """BASELINE configs[2] / cfg3: the obstacle scenario (S 19, W 6, V 2, O 9, obs 40)."""
    args = dict(num_envs=64, num_agents=8, quads_mode="mix", use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2)
    args.update(kw)
    return QuadSimConfig(**args)


def bf16(x):
    import torch
    return x.to(torch.bfloat16).to(torch.float32)


def emulated_forward(pol, obs):
    """The module's forward with the kernel's rounding points, obstacle encoder included."""
    import torch

    def lin(layer, x):
        return bf16(x) @ bf16(layer.weight).t() + layer.bias

    def mlp2(seq, x):
        return torch.tanh(lin(seq[2], torch.tanh(lin(seq[0], x))))

    def tower(enc, head):
        parts = [mlp2(enc.self_encoder, obs[:, :enc.S])]
        if enc.kind == "mean_embed":
            nb = obs[:, enc.S:enc.S + enc.W * enc.V].reshape(-1, enc.V, enc.W)
            parts.append(sum(mlp2(enc.neighbor, nb[:, j]) for j in range(enc.V)) * (1.0 / enc.V))
        o0 = enc.S + enc.W * enc.V
        parts.append(mlp2(enc.obstacle, obs[:, o0:o0 + enc.O]))
        y = torch.tanh(bf16(torch.cat(parts, dim=1)) @ bf16(enc.feed_forward[0].weight).t() + enc.feed_forward[0].bias)
        return y @ head.weight.t() + head.bias                 # heads stay fp32 in the kernel

    return tower(pol.actor, pol.action_net), tower(pol.critic, pol.value_net).squeeze(-1)


def make_policy(cfg, seed):
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    torch.manual_seed(seed)
    pol = QuadActorCritic(cfg).to("cuda:0")
    with torch.no_grad():                                         # non-zero biases
        for m in pol.modules():
            if isinstance(m, torch.nn.Linear):
                m.bias.uniform_(-0.3, 0.3)
    return pol


def make_obs(pol, n, pad=0):
    import torch
    enc = pol.actor
    o0 = enc.S + enc.W * enc.V
    obs = torch.randn(n, o0 + enc.O + pad, device="cuda:0") * 0.8
    obs[:, o0:o0 + enc.O] = 0.5 + 2.5 * torch.rand(n, enc.O, device="cuda:0")
    return obs


def check_parity(pol, fp, obs, tag):
    import torch
    enc = pol.actor
    D = enc.S + enc.W * enc.V + enc.O
    mean, value = fp.forward(obs)
    torch.cuda.synchronize()
    torch.backends.cuda.matmul.allow_tf32 = False
    x = obs[:, :D].contiguous()
    with torch.no_grad():
        r_mean, r_value = pol.action_net(pol.actor(x)), pol.value(x)
        e_mean, e_value = emulated_forward(pol, x)
    assert torch.isfinite(mean).all() and torch.isfinite(value).all()
    d32 = torch.cat([(mean - r_mean).reshape(-1), (value - r_value).reshape(-1)])
    demu = torch.cat([(mean - e_mean).reshape(-1), (value - e_value).reshape(-1)])
    print(f"\n[{tag}] n={obs.shape[0]} S={fp.S} W={fp.W} V={fp.V} O={fp.O} A={fp.A}: vs fp32 max {float(d32.abs().max()):.2e}"
          f" rms {float(d32.pow(2).mean().sqrt()):.2e}; vs bf16-emulated max {float(demu.abs().max()):.2e}")
    assert float(demu.abs().max()) <= TOL_EMU_MAX
    assert float(d32.abs().max()) <= TOL_FP32_MAX
    assert float(d32.pow(2).mean().sqrt()) <= TOL_FP32_RMS
    return mean, value


CASES = {
    # name: (config, rows, extra obs columns behind the obstacle block)
    "cfg3": (lambda: cfg3(), 8192, 0),
    "ragged_rows": (lambda: cfg3(), 1000 + 37, 0),
    "tiny": (lambda: cfg3(num_envs=1), 5, 0),
    "one_tile_exact": (lambda: cfg3(num_envs=16), 128, 0),
    "many_tiles": (lambda: cfg3(), 148 * 128 * 2 + 77, 0),
    "v6": (lambda: QuadSimConfig(num_envs=8, num_agents=8, quads_mode="mix", use_obstacles=True, neighbor_visible_num=6), 3000, 0),
    "no_neighbours": (lambda: cfg3(num_envs=8, num_agents=1, neighbor_visible_num=0), 600, 0),
    "padded_stride": (lambda: cfg3(), 2048 + 3, 5),
}


@pytest.mark.parametrize("name", list(CASES))
def test_fused_forward_with_obstacles_matches_torch(name):
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy, supported
    make, n, pad = CASES[name]
    pol = make_policy(make(), 1234)
    assert supported(pol) and pol.actor.O == 9
    fp = FusedPolicy(pol, "cuda:0")
    obs = make_obs(pol, n, pad)
    l0 = fp.launch_count
    check_parity(pol, fp, obs, name)
    assert fp.launch_count == l0 + 1


def test_obstacle_weight_resync():
    """Only the obstacle encoder changes: the kernel keeps its packed copy until sync(), then follows the module."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy
    pol = make_policy(cfg3(), 7)
    fp = FusedPolicy(pol, "cuda:0")
    obs = make_obs(pol, 1500)
    m0, v0 = fp.forward(obs)
    with torch.no_grad():
        for enc in (pol.actor, pol.critic):
            for p in enc.obstacle.parameters():
                p.add_(0.1 * torch.randn_like(p))
    m_stale, _ = fp.forward(obs)
    assert torch.equal(m0, m_stale)
    fp.sync()
    m1, v1 = check_parity(pol, fp, obs, "resync")
    assert float((m1 - m0).abs().max()) > 0.02 and float((v1 - v0).abs().max()) > 0.02


def test_device_ppo_obstacle_config_uses_the_fused_rollout():
    import numpy as np
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    cfg = cfg3(num_envs=128, ep_time=0.3, seed=2)
    sim = QuadSwarmSim(cfg, device="cuda:0")
    sim.want_terminal_obs = False
    n_steps = 8
    ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=n_steps, batch_size=4096, n_epochs=1))
    assert ppo.fused is not None and ppo.fused.O == 9
    w0 = torch.cat([p.detach().reshape(-1).clone() for p in ppo.policy.parameters()])
    l0, s0 = ppo.fused.launch_count, sim.launch_count
    hist = ppo.learn(2)
    assert ppo.fused.launch_count - l0 == 2 * (n_steps + 1)          # one launch per env step + the bootstrap value
    assert sim.launch_count - s0 == 2 * n_steps                      # one simulator launch per env step
    for r in hist:
        assert all(np.isfinite(r[k]) for k in ("pg", "vf", "ent", "kl", "mean_reward"))
    w1 = torch.cat([p.detach().reshape(-1) for p in ppo.policy.parameters()])
    assert bool(torch.isfinite(w1).all()) and not torch.equal(w0, w1)
    obs = make_obs(ppo.policy, 700)
    m, _ = ppo.fused.forward(obs)                                    # the packed weights follow the optimiser
    with torch.no_grad():
        r = ppo.policy.action_net(ppo.policy.actor(obs))
    assert float((m - r).abs().max()) <= TOL_FP32_MAX


def test_abi_obstacle_checks_and_version_1_handle():
    """Version-2 checks (obst_dim bound, null obstacle pointers, obs_stride covering the obstacle block) and a handle created with the
    six-field version-1 struct, which still runs the plain kernel."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy, QpConfigC, QpTowerWeightsC
    lib = _capi.lib()
    dev = torch.device("cuda:0")
    h = C.c_void_p()
    assert lib.qp_create(C.byref(QpConfigC(2, 19, 6, 2, 256, 4, 25)), 0, C.byref(h)) == -2 and not h.value
    assert b"obst_dim" in lib.qp_last_error(None)
    assert lib.qp_create(C.byref(QpConfigC(2, 19, 6, 2, 256, 4, -1)), 0, C.byref(h)) == -2
    assert lib.qp_create(C.byref(QpConfigC(3, 19, 6, 2, 256, 4, 9)), 0, C.byref(h)) == -2

    pol = make_policy(cfg3(), 3)
    fp = FusedPolicy(pol, dev)
    w = QpTowerWeightsC()
    for name in QpTowerWeightsC.FIELDS:                           # non-null everywhere but one obstacle pointer: rejected before any packing
        setattr(w, name, fp._keep[0].data_ptr())
    w.obst_w2 = None
    s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    assert lib.qp_set_weights(fp._h, 0, C.byref(w), s) == -1
    assert b"obstacle" in lib.qp_last_error(fp._h)
    obs = make_obs(pol, 10)
    mean, value = torch.empty(10, 4, device=dev), torch.empty(10, device=dev)
    assert lib.qp_forward(fp._h, obs.data_ptr(), 10, 39, mean.data_ptr(), value.data_ptr(), s) == -2   # 19 + 2 * 6 + 9 = 40
    assert b"obs_stride" in lib.qp_last_error(fp._h)
    assert lib.qp_forward(fp._h, obs.data_ptr(), 10, 40, mean.data_ptr(), value.data_ptr(), s) == 0
    fp.close()

    # version 1: the struct ends before obst_dim (a C caller of the first release); the handle never reads the obst_* weight fields
    class QpConfigV1(C.Structure):
        _fields_ = [(n, C.c_int32) for n in ("api_version", "self_dim", "nbr_dim", "num_nbr", "hidden", "act_dim")]

    class QpTowerWeightsV1(C.Structure):
        _fields_ = [(n, C.c_void_p) for n in QpTowerWeightsC.FIELDS[:12]]

    cfg = QuadSimConfig(num_envs=64, num_agents=8)                 # cfg2: S 18, W 6, V 6, obs 54
    pol2 = make_policy(cfg, 11)
    ref = FusedPolicy(pol2, dev)                                   # version-2 handle, obst_dim 0
    h1 = C.c_void_p()
    assert lib.qp_create(C.byref(QpConfigV1(1, 18, 6, 6, 256, 4)), 0, C.byref(h1)) == 0 and h1.value
    try:
        keep = []
        for tower, (enc, head) in enumerate(((pol2.actor, pol2.action_net), (pol2.critic, pol2.value_net))):
            t = [enc.self_encoder[0].weight, enc.self_encoder[0].bias, enc.self_encoder[2].weight, enc.self_encoder[2].bias,
                 enc.neighbor[0].weight, enc.neighbor[0].bias, enc.neighbor[2].weight, enc.neighbor[2].bias,
                 enc.feed_forward[0].weight, enc.feed_forward[0].bias, head.weight, head.bias]
            t = [v.detach().float().contiguous() for v in t]
            keep += t
            w1 = QpTowerWeightsV1(*[v.data_ptr() for v in t])
            assert lib.qp_set_weights(h1, tower, C.byref(w1), s) == 0
        obs2 = torch.randn(4096, 54, device=dev) * 0.8
        m1, v1 = torch.empty(4096, 4, device=dev), torch.empty(4096, device=dev)
        assert lib.qp_forward(h1, obs2.data_ptr(), 4096, 54, m1.data_ptr(), v1.data_ptr(), s) == 0
        m2, v2 = ref.forward(obs2)
        torch.cuda.synchronize()
        assert torch.equal(m1, m2) and torch.equal(v1, v2)
        with torch.no_grad():
            assert float((m1 - pol2.action_net(pol2.actor(obs2))).abs().max()) <= TOL_FP32_MAX
    finally:
        lib.qp_destroy(h1)
        ref.close()
