"""Fused tcgen05 policy forward (csrc/policy_kernels.cu, include/quadpolicy.h) against the torch fp32 module it replaces
(`ppo.QuadActorCritic` = the reference's ActorCriticPolicyCustomSeparateWeights + QuadMultiEncoder,
swarm_rl/models/ActorCriticPolicyCustom.py:284-556, swarm_rl/models/quad_multi_model.py:16-41,250-354).

Two references, both plain PyTorch:
  * fp32: the module as it is.  The kernel multiplies in bf16 (fp32 accumulation), so the tolerance is the bf16 one, stated below.
  * bf16-emulated: the same module with weights and layer inputs rounded to bf16 at the points the kernel rounds them (everything
    else fp32).  This pins the kernel's arithmetic (layout of every weight image, bias, tanh, neighbour mean, heads) to 2e-3.
"""
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402

TOL_FP32_MAX = 3e-2        # |kernel - fp32 module|, absolute, outputs are O(1): bf16 operands through 4 layers
TOL_FP32_RMS = 6e-3
TOL_EMU_MAX = 3e-3         # |kernel - bf16-emulated module|: accumulation order + tanh.approx (2^-11) only


def bf16(x):
    import torch
    return x.to(torch.bfloat16).to(torch.float32)


def emulated_forward(pol, obs):
    """The module's forward with the kernel's rounding points."""
    import torch

    def lin(layer, x):
        return bf16(x) @ bf16(layer.weight).t() + layer.bias

    def tower(enc, head):
        s = obs[:, :enc.S]
        h = torch.tanh(lin(enc.self_encoder[2], torch.tanh(lin(enc.self_encoder[0], s))))
        if enc.kind == "mean_embed":
            nb = obs[:, enc.S:enc.S + enc.W * enc.V].reshape(-1, enc.V, enc.W)
            acc = 0
            for j in range(enc.V):
                acc = acc + torch.tanh(lin(enc.neighbor[2], torch.tanh(lin(enc.neighbor[0], nb[:, j]))))
            m = acc * (1.0 / enc.V)
        else:
            m = torch.zeros_like(h)
        w = enc.feed_forward[0].weight
        if w.shape[1] == 256:
            y = torch.tanh(bf16(h) @ bf16(w).t() + enc.feed_forward[0].bias)
        else:
            y = torch.tanh(bf16(torch.cat([h, m], dim=1)) @ bf16(w).t() + enc.feed_forward[0].bias)
        return y @ head.weight.t() + head.bias                 # heads stay fp32 in the kernel

    return tower(pol.actor, pol.action_net), tower(pol.critic, pol.value_net).squeeze(-1)


CASES = {
    # name: (config, rows, extra obs columns behind the neighbour block)
    "cfg2_k8": (lambda: QuadSimConfig(num_envs=64, num_agents=8), 8192, 0),
    "ragged_rows": (lambda: QuadSimConfig(num_envs=64, num_agents=8), 1000 + 37, 0),
    "tiny": (lambda: QuadSimConfig(num_envs=1, num_agents=8), 5, 0),
    "one_tile_exact": (lambda: QuadSimConfig(num_envs=16, num_agents=8), 128, 0),
    "many_tiles": (lambda: QuadSimConfig(num_envs=64, num_agents=8), 148 * 128 * 2 + 77, 0),
    "repr24_v2": (lambda: QuadSimConfig(num_envs=8, num_agents=8, obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2), 777, 0),
    "no_neighbours": (lambda: QuadSimConfig(num_envs=8, num_agents=1, neighbor_visible_num=0), 600, 0),
    "k32_v6_padded_stride": (lambda: QuadSimConfig(num_envs=4, num_agents=32, neighbor_visible_num=6), 2048 + 3, 5),
    "fork_act2": (lambda: QuadSimConfig.fork_default(num_envs=8), 900, 0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_fused_forward_matches_torch(name):
    import torch
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy, supported
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    make, n, pad = CASES[name]
    cfg = make()
    torch.manual_seed(1234)
    dev = torch.device("cuda:0")
    pol = QuadActorCritic(cfg).to(dev)
    with torch.no_grad():                                         # non-zero biases and a non-trivial head
        for m in pol.modules():
            if isinstance(m, torch.nn.Linear):
                m.bias.uniform_(-0.3, 0.3)
    if not supported(pol):
        pytest.skip("architecture outside the fused kernel (documented in include/quadpolicy.h)")
    fp = FusedPolicy(pol, dev)
    D = pol.actor.S + pol.actor.W * pol.actor.V
    obs = torch.randn(n, D + pad, device=dev) * 0.8
    l0 = fp.launch_count
    mean, value = fp.forward(obs)
    torch.cuda.synchronize()
    assert fp.launch_count == l0 + 1
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        r_mean = pol.action_net(pol.actor(obs[:, :D] if pad == 0 else obs[:, :D].contiguous()))
        r_value = pol.value(obs[:, :D].contiguous())
        e_mean, e_value = emulated_forward(pol, obs[:, :D].contiguous())
    assert torch.isfinite(mean).all() and torch.isfinite(value).all()
    d32 = torch.cat([(mean - r_mean).reshape(-1), (value - r_value).reshape(-1)])
    demu = torch.cat([(mean - e_mean).reshape(-1), (value - e_value).reshape(-1)])
    print(f"\n[{name}] n={n} S={fp.S} W={fp.W} V={fp.V} A={fp.A}: vs fp32 max {float(d32.abs().max()):.2e} rms {float(d32.pow(2).mean().sqrt()):.2e};"
          f" vs bf16-emulated max {float(demu.abs().max()):.2e}; |mean| rms {float(r_mean.pow(2).mean().sqrt()):.2f}")
    assert float(demu.abs().max()) <= TOL_EMU_MAX
    assert float(d32.abs().max()) <= TOL_FP32_MAX
    assert float(d32.pow(2).mean().sqrt()) <= TOL_FP32_RMS


def test_weight_resync_and_act():
    """`sync()` after an optimiser step re-packs the weights; `act` returns the Gaussian sample's log-probability."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import FusedPolicy
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    cfg = QuadSimConfig(num_envs=32, num_agents=8)
    dev = torch.device("cuda:0")
    torch.manual_seed(7)
    pol = QuadActorCritic(cfg).to(dev)
    fp = FusedPolicy(pol, dev)
    obs = torch.randn(512, 54, device=dev)
    m0, _ = fp.forward(obs)
    with torch.no_grad():
        for p in pol.parameters():
            p.add_(0.05 * torch.randn_like(p))
    m_stale, _ = fp.forward(obs)
    assert torch.equal(m0, m_stale)                              # the kernel runs on its packed copy until sync()
    fp.sync()
    m1, v1 = fp.forward(obs)
    with torch.no_grad():
        r = pol.action_net(pol.actor(obs))
    assert float((m1 - r).abs().max()) <= TOL_FP32_MAX and float((m1 - m0).abs().max()) > 0.05
    a, logp, v = fp.act(obs)
    d = torch.distributions.Normal(m1, pol.log_std.detach().exp().expand_as(m1))
    assert torch.allclose(logp, d.log_prob(a).sum(-1), atol=1e-4) and torch.equal(v, v1)


def test_gae_kernel_matches_the_recursion():
    """`qp_gae` against `ppo.compute_gae` (itself pinned against a numpy restatement of SB3's recursion in tests/test_ppo_cpu.py)."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import gae
    from quad_swarm_rl_stable_baselines3_b200.ppo import compute_gae
    torch.manual_seed(3)
    dev = torch.device("cuda:0")
    for T, n in ((1, 5), (7, 1000), (128, 4096 + 3)):
        rew, val = torch.randn(T, n, device=dev), torch.randn(T, n, device=dev)
        done = torch.rand(T, n, device=dev) < 0.05
        last = torch.randn(n, device=dev)
        a0, r0 = compute_gae(rew, val, done, last, 0.99, 0.95)
        a1, r1 = gae(rew, val, done, last, 0.99, 0.95)
        assert float((a0 - a1).abs().max()) <= 2e-5 * max(1.0, float(a0.abs().max())), (T, n)
        assert float((r0 - r1).abs().max()) <= 2e-5 * max(1.0, float(r0.abs().max())), (T, n)


def test_device_ppo_uses_the_fused_rollout():
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    cfg = QuadSimConfig(num_envs=256, num_agents=8, ep_time=0.3, seed=1)
    sim = QuadSwarmSim(cfg, device="cuda:0")
    sim.want_terminal_obs = False
    ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=8, batch_size=4096, n_epochs=1))
    assert ppo.fused is not None
    l0 = ppo.fused.launch_count
    hist = ppo.learn(2)
    assert ppo.fused.launch_count - l0 == 2 * (8 + 1)               # one launch per env step + the bootstrap value
    assert all(torch.isfinite(torch.tensor([r[k] for k in ("pg", "vf", "ent", "kl")])).all() for r in hist)
    obs = torch.randn(512, 54, device="cuda:0")
    m, _ = ppo.fused.forward(obs)                                  # the packed weights follow the optimiser
    with torch.no_grad():
        r = ppo.policy.action_net(ppo.policy.actor(obs))
    assert float((m - r).abs().max()) <= TOL_FP32_MAX


def test_two_policies_and_argument_checks():
    """Handles of every built variant alive at once (a training policy and an evaluation copy, as sb_train.py keeps them, of each
    encoder): deep-sets (cfg2 and the fork's), obstacle, MLP, and an MLP handle made from the six-field version-1 qp_config.  Their
    forwards interleave on the default stream and a second one, and each output equals, bit for bit, the same handle's forward run alone;
    repacking one handle's weights and then destroying another leave the remaining handles' outputs bitwise unchanged.  The C-ABI rejects
    bad shapes with a message instead of launching."""
    import ctypes as C
    import torch
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import QP_NBR, FusedPolicy
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    dev = torch.device("cuda:0")
    lib = _capi.lib()
    torch.manual_seed(5)
    fork_k8 = QuadSimConfig.fork_default(num_envs=8, num_agents=8, neighbor_obs_type="dist_sangle_sheading",
                                         obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot")           # MLP: 35 inputs
    pols = {"deepsets": QuadActorCritic(QuadSimConfig(num_envs=8, num_agents=8)),
            "fork": QuadActorCritic(QuadSimConfig.fork_default(num_envs=8)),
            "obstacles": QuadActorCritic(QuadSimConfig(num_envs=8, num_agents=8, quads_mode="mix", use_obstacles=True,
                                                       obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2)),
            "mlp": QuadActorCritic(QuadSimConfig(num_envs=8, num_agents=8), neighbor_encoder="mlp"),
            "mlp_v1": QuadActorCritic(fork_k8, neighbor_encoder="mlp")}
    rows = {"deepsets": 3000, "fork": 700, "obstacles": 1500, "mlp": 2100, "mlp_v1": 900}
    obs = {}
    for k, pol in pols.items():
        pol.to(dev)
        with torch.no_grad():                                     # non-zero biases
            for m in pol.modules():
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)
        enc = pol.actor
        obs[k] = torch.randn(rows[k], enc.S + enc.W * enc.V + enc.O, device=dev) * 0.8
    fps = {k: FusedPolicy(pol, dev) for k, pol in pols.items()}
    assert fps["obstacles"].O == 9 and fps["mlp"].kind == "mlp" and fps["mlp_v1"].kind == "mlp"

    # version 1: the struct ends before obst_dim (a C caller of the first release)
    class QpConfigV1(C.Structure):
        _fields_ = [(n, C.c_int32) for n in ("api_version", "self_dim", "nbr_dim", "num_nbr", "hidden", "act_dim")]

    f1, h1 = fps["mlp_v1"], C.c_void_p()
    assert lib.qp_create_encoder(C.byref(QpConfigV1(1, f1.S, f1.W, f1.V, 256, f1.A)), QP_NBR["mlp"], 0, C.byref(h1)) == 0 and h1.value
    lib.qp_destroy(f1._h)
    f1._h = h1                                                    # the same policy, packed into the version-1 handle
    f1.sync()

    alone = {}
    for k, fp in fps.items():
        alone[k] = fp.forward(obs[k])
        torch.cuda.synchronize()
        pol = pols[k]
        with torch.no_grad():
            assert float((alone[k][0] - pol.action_net(pol.actor(obs[k]))).abs().max()) <= TOL_FP32_MAX, k
            assert float((alone[k][1] - pol.value(obs[k])).abs().max()) <= TOL_FP32_MAX, k

    def interleaved():
        """Three rounds over the live handles; each round alternates them between the default stream and a second one."""
        main, side = torch.cuda.current_stream(dev), torch.cuda.Stream(dev)
        side.wait_stream(main)
        outs = []
        for r in range(3):
            for i, k in enumerate(fps):
                with torch.cuda.stream(side if (i + r) % 2 else main):
                    outs.append((k, fps[k].forward(obs[k])))
        torch.cuda.synchronize()
        for k, (m, v) in outs:
            assert torch.equal(m, alone[k][0]) and torch.equal(v, alone[k][1]), k

    interleaved()
    with torch.no_grad():                                         # new weights in one handle ...
        for p in pols["mlp"].parameters():
            p.add_(0.05 * torch.randn_like(p))
    fps["mlp"].sync()
    m, v = fps["mlp"].forward(obs["mlp"])
    torch.cuda.synchronize()
    assert float((m - alone["mlp"][0]).abs().max()) > 0.05
    with torch.no_grad():
        assert float((m - pols["mlp"].action_net(pols["mlp"].actor(obs["mlp"]))).abs().max()) <= TOL_FP32_MAX
    alone["mlp"] = (m, v)
    interleaved()                                                 # ... the others unchanged
    fps.pop("obstacles").close()                                  # one handle destroyed: the others unchanged
    interleaved()

    fa = fps["deepsets"]
    oa = obs["deepsets"]
    mean, value = torch.empty(10, 4, device=dev), torch.empty(10, device=dev)
    s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    assert lib.qp_forward(fa._h, oa.data_ptr(), 10, 40, mean.data_ptr(), value.data_ptr(), s) == -2      # stride shorter than S + V*W
    assert b"obs_stride" in lib.qp_last_error(fa._h)
    assert lib.qp_forward(fa._h, None, 10, 54, mean.data_ptr(), value.data_ptr(), s) == -1
    assert lib.qp_forward(fa._h, oa.data_ptr(), 0, 54, mean.data_ptr(), value.data_ptr(), s) == -2
    with pytest.raises(ValueError):
        fa.forward(oa.double())
    for fp in fps.values():
        fp.close()
