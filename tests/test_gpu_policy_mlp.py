"""Fused tcgen05 policy forward with the MLP neighbour encoder (csrc/policy_kernels.cu, variant MLP; include/quadpolicy.h
qp_create_encoder(QP_NBR_MLP)) against the torch module it replaces (`ppo.QuadEncoder` with neighbor_encoder="mlp": the W * V neighbour
columns as one vector -> 256 -> 256 -> 256, tanh, feed-forward input [self | neighbour]; reference: swarm_rl/models/quad_multi_model.py:104-122).

Two references, both plain PyTorch, with the fp32 tolerances of tests/test_gpu_policy.py (the emulation's is wider, see TOL_EMU_MAX):
  * fp32: the module as it is;
  * bf16-emulated: the module with weights and layer inputs rounded to bf16 where the kernel rounds them.
Neighbour inputs 32-39 (the part of layer 1 that reads stream 0's x tile) are drawn at another scale than the rest of the row, so a wrong
slot for them cannot pass.  Every forward runs on NaN-filled outputs with rows to spare and NaN observation rows behind row n: nothing
behind row n may be written, and no live row may read them.
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
# tests/test_gpu_policy.py's 3e-3 plus a third: the emulation's tanh is exact, the kernel's tanh.approx (2^-11 relative) flips the bf16
# rounding of some activations, and the MLP tower rounds two more 256-wide layers than the deep-sets one and does not average its encoder
# output over V neighbours.  Measured on a B200: 1.9e-3 .. 2.6e-3 up to 8192 rows, 3.2e-3 on the 37965-row batch.
TOL_EMU_MAX = 4e-3
SPARE = 128                      # canary rows behind row n


def cfg2(**kw):
    """BASELINE configs[4] / cfg2: 8 quads, S 18, W 6, V 6 (W * V = 36)."""
    args = dict(num_envs=64, num_agents=8)
    args.update(kw)
    return QuadSimConfig(**args)


def bf16(x):
    import torch
    return x.to(torch.bfloat16).to(torch.float32)


def emulated_forward(pol, obs):
    """The module's forward with the kernel's rounding points."""
    import torch

    def lin(layer, x):
        return bf16(x) @ bf16(layer.weight).t() + layer.bias

    def tower(enc, head):
        h = torch.tanh(lin(enc.self_encoder[2], torch.tanh(lin(enc.self_encoder[0], obs[:, :enc.S]))))
        x = obs[:, enc.S:enc.S + enc.W * enc.V]
        for i in (0, 2, 4):
            x = torch.tanh(lin(enc.neighbor[i], x))
        y = torch.tanh(bf16(torch.cat([h, x], dim=1)) @ bf16(enc.feed_forward[0].weight).t() + enc.feed_forward[0].bias)
        return y @ head.weight.t() + head.bias                 # heads stay fp32 in the kernel

    return tower(pol.actor, pol.action_net), tower(pol.critic, pol.value_net).squeeze(-1)


def make_policy(cfg, seed):
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    torch.manual_seed(seed)
    pol = QuadActorCritic(cfg, neighbor_encoder="mlp").to("cuda:0")
    with torch.no_grad():                                         # non-zero biases
        for m in pol.modules():
            if isinstance(m, torch.nn.Linear):
                m.bias.uniform_(-0.3, 0.3)
    return pol


def make_obs(pol, n, pad=0):
    """[n + SPARE, D + pad]: rows behind n are NaN; neighbour inputs 32.. are positive and larger than the rest."""
    import torch
    enc = pol.actor
    D = enc.S + enc.W * enc.V
    obs = torch.randn(n + SPARE, D + pad, device="cuda:0") * 0.8
    if enc.W * enc.V > 32:
        obs[:, enc.S + 32:D] = 1.0 + 2.0 * torch.rand(n + SPARE, D - enc.S - 32, device="cuda:0")
    obs[n:] = float("nan")
    return obs


def fused_forward(fp, obs, n):
    """qp_forward on the first n rows into NaN-filled outputs with SPARE rows behind them."""
    import torch
    mean = torch.full((n + SPARE, fp.A), float("nan"), device=fp.device)
    value = torch.full((n + SPARE,), float("nan"), device=fp.device)
    l0 = fp.launch_count
    with torch.cuda.device(fp.device):
        rc = fp._lib.qp_forward(fp._h, obs.data_ptr(), n, obs.shape[1], mean.data_ptr(), value.data_ptr(), fp._stream())
    assert rc == 0, fp._lib.qp_last_error(fp._h)
    torch.cuda.synchronize()
    assert fp.launch_count == l0 + 1
    assert bool(mean[n:].isnan().all()) and bool(value[n:].isnan().all()), "rows behind n were written"
    return mean[:n], value[:n]


def check_parity(pol, fp, obs, n, tag):
    import torch
    enc = pol.actor
    D = enc.S + enc.W * enc.V
    mean, value = fused_forward(fp, obs, n)
    torch.backends.cuda.matmul.allow_tf32 = False
    x = obs[:n, :D].contiguous()
    with torch.no_grad():
        r_mean, r_value = pol.action_net(pol.actor(x)), pol.value(x)
        e_mean, e_value = emulated_forward(pol, x)
    assert torch.isfinite(mean).all() and torch.isfinite(value).all()
    d32 = torch.cat([(mean - r_mean).reshape(-1), (value - r_value).reshape(-1)])
    demu = torch.cat([(mean - e_mean).reshape(-1), (value - e_value).reshape(-1)])
    print(f"\n[{tag}] n={n} stride={obs.shape[1]} S={fp.S} W={fp.W} V={fp.V} A={fp.A}: vs fp32 max {float(d32.abs().max()):.2e}"
          f" rms {float(d32.pow(2).mean().sqrt()):.2e}; vs bf16-emulated max {float(demu.abs().max()):.2e}")
    assert float(demu.abs().max()) <= TOL_EMU_MAX
    assert float(d32.abs().max()) <= TOL_FP32_MAX
    assert float(d32.pow(2).mean().sqrt()) <= TOL_FP32_RMS
    return mean, value


CASES = {
    # name: (config, rows, extra obs columns behind the neighbour block)
    "cfg2": (lambda: cfg2(), 8192, 0),
    "ragged_rows": (lambda: cfg2(), 1000 + 37, 0),
    "one_row": (lambda: cfg2(num_envs=1), 1, 0),
    "one_tile_exact": (lambda: cfg2(num_envs=16), 128, 0),
    "many_tiles": (lambda: cfg2(), 148 * 128 * 2 + 77, 0),
    "padded_stride": (lambda: cfg2(), 2048 + 3, 5),
    "k32_v6": (lambda: QuadSimConfig(num_envs=4, num_agents=32, neighbor_visible_num=6), 3000, 0),
    "fork_act2": (lambda: QuadSimConfig.fork_default(num_envs=8), 900, 0),
    "fork_k8_sheading": (lambda: QuadSimConfig.fork_default(num_envs=8, num_agents=8, neighbor_obs_type="dist_sangle_sheading",
                                                            obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot"), 1500, 3),
}


@pytest.mark.parametrize("name", list(CASES))
def test_fused_forward_with_mlp_encoder_matches_torch(name):
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy, supported
    make, n, pad = CASES[name]
    pol = make_policy(make(), 1234)
    assert pol.actor.kind == "mlp" and supported(pol)
    fp = FusedPolicy(pol, "cuda:0")
    assert fp.V == pol.actor.V
    check_parity(pol, fp, make_obs(pol, n, pad), n, name)
    fp.close()


def test_mlp_weight_resync():
    """Only the neighbour encoder's third layer changes: the kernel keeps its packed copy until sync(), then follows the module."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy
    pol = make_policy(cfg2(), 7)
    fp = FusedPolicy(pol, "cuda:0")
    obs = make_obs(pol, 1500)
    m0, v0 = fused_forward(fp, obs, 1500)
    with torch.no_grad():
        for enc in (pol.actor, pol.critic):
            for p in enc.neighbor[4].parameters():
                p.add_(0.1 * torch.randn_like(p))
    m_stale, _ = fused_forward(fp, obs, 1500)
    assert torch.equal(m0, m_stale)
    fp.sync()
    m1, v1 = check_parity(pol, fp, obs, 1500, "resync")
    assert float((m1 - m0).abs().max()) > 0.02 and float((v1 - v0).abs().max()) > 0.02
    fp.close()


def test_abi_mlp_rejections():
    """qp_create_encoder rejects what the MLP variant does not build, by code and message; qp_set_weights rejects a null layer 3."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import QP_API_VERSION, FusedPolicy, QpConfigC, QpTowerWeightsC
    lib = _capi.lib()
    h = C.c_void_p()
    for cfg, kind, msg in ((QpConfigC(QP_API_VERSION, 18, 6, 7, 256, 4, 0), 1, b"<= 40"),          # W * V = 42
                           (QpConfigC(QP_API_VERSION, 19, 6, 2, 256, 4, 9), 1, b"obst_dim"),       # with the obstacle encoder
                           (QpConfigC(QP_API_VERSION, 18, 6, 0, 256, 4, 0), 1, b"num_nbr"),        # no neighbours
                           (QpConfigC(QP_API_VERSION, 18, 6, 6, 256, 4, 0), 2, b"nbr_encoder"),    # unknown kind
                           (QpConfigC(QP_API_VERSION, 18, 6, 6, 256, 4, 0), -1, b"nbr_encoder")):
        assert lib.qp_create_encoder(C.byref(cfg), kind, 0, C.byref(h)) == -2 and not h.value
        assert msg in lib.qp_last_error(None), lib.qp_last_error(None)
    assert lib.qp_create_encoder(C.byref(QpConfigC(QP_API_VERSION, 18, 8, 5, 256, 4, 0)), 1, 0, C.byref(h)) == 0 and h.value   # 40: the limit
    lib.qp_destroy(h)

    dev = torch.device("cuda:0")
    pol = make_policy(cfg2(), 3)
    fp = FusedPolicy(pol, dev)
    obs = make_obs(pol, 600)
    m0, v0 = fused_forward(fp, obs, 600)
    s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    for missing in ("nbr_w3", "nbr_b3"):                          # rejected before anything is packed: the outputs do not change
        w = QpTowerWeightsC()
        for name in QpTowerWeightsC.FIELDS:
            setattr(w, name, fp._keep[0].data_ptr())
        setattr(w, missing, None)
        assert lib.qp_set_weights(fp._h, 0, C.byref(w), s) == -1
        assert b"nbr_w3" in lib.qp_last_error(fp._h)
    m1, v1 = fused_forward(fp, obs, 600)
    assert torch.equal(m0, m1) and torch.equal(v0, v1)
    fp.close()


def test_supported_keeps_the_unbuilt_mlp_policies_on_torch():
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import supported
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    with_obstacles = QuadSimConfig(num_envs=8, num_agents=8, quads_mode="mix", use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor",
                                   neighbor_visible_num=2)
    wide = cfg2(num_envs=8, neighbor_visible_num=7)                # W * V = 42
    for cfg in (with_obstacles, wide):
        assert not supported(QuadActorCritic(cfg, neighbor_encoder="mlp"))
        assert supported(QuadActorCritic(cfg))                      # the deep-sets policy of the same config is built


@pytest.mark.parametrize("which", ["obstacles", "wide"])
def test_device_ppo_leaves_unbuilt_mlp_policies_on_torch(which):
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    extra = (dict(quads_mode="mix", use_obstacles=True, obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2) if which == "obstacles"
             else dict(neighbor_visible_num=7))
    cfg = QuadSimConfig(num_envs=16, num_agents=8, ep_time=0.3, seed=2, **extra)
    sim = QuadSwarmSim(cfg, device="cuda:0")
    ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=2, batch_size=256, n_epochs=1, neighbor_encoder="mlp"))
    assert ppo.fused is None


def test_device_ppo_mlp_config_uses_the_fused_rollout():
    """cfg2 (W * V = 36) and the fork env (W 2, V 3: its policy's first layers have 6 inputs and train through _FirstBiasTanh)."""
    import numpy as np
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    for cfg, V in ((cfg2(num_envs=128, ep_time=0.3, seed=2), 6), (QuadSimConfig.fork_default(num_envs=256, ep_time=1.0, seed=3), 3)):
        sim = QuadSwarmSim(cfg, device="cuda:0")
        sim.want_terminal_obs = False
        n_steps = 8
        ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=n_steps, batch_size=4096, n_epochs=1, neighbor_encoder="mlp"))
        assert ppo.fused is not None and ppo.fused.kind == "mlp" and ppo.fused.V == V
        w0 = torch.cat([p.detach().reshape(-1).clone() for p in ppo.policy.parameters()])
        l0, s0 = ppo.fused.launch_count, sim.launch_count
        hist = ppo.learn(2)
        assert ppo.fused.launch_count - l0 == 2 * (n_steps + 1)          # one launch per env step + the bootstrap value
        assert sim.launch_count - s0 == 2 * n_steps
        for r in hist:
            assert all(np.isfinite(r[k]) for k in ("pg", "vf", "ent", "kl", "mean_reward"))
        w1 = torch.cat([p.detach().reshape(-1) for p in ppo.policy.parameters()])
        assert bool(torch.isfinite(w1).all()) and not torch.equal(w0, w1)
        obs = make_obs(ppo.policy, 700)
        m, v = fused_forward(ppo.fused, obs, 700)                         # update() packed the optimiser's weights again
        with torch.no_grad():
            x = obs[:700]
            r_mean, r_value = ppo.policy.action_net(ppo.policy.actor(x)), ppo.policy.value(x)
        assert float((m - r_mean).abs().max()) <= TOL_FP32_MAX and float((v - r_value).abs().max()) <= TOL_FP32_MAX
        ppo.fused.close()
