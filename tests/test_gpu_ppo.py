"""Device PPO loop over the real CUDA simulator: rollouts and updates stay on the GPU."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402


@pytest.mark.parametrize("make", [
    lambda: QuadSimConfig(num_envs=256, num_agents=8, ep_time=0.3, seed=1),
    lambda: QuadSimConfig(num_envs=128, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                          obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, ep_time=0.3, seed=2),
    lambda: QuadSimConfig.fork_default(num_envs=256, ep_time=1.0, seed=3),
])
def test_ppo_iterations_on_device(make):
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    cfg = make()
    sim = QuadSwarmSim(cfg, device="cuda:0")
    sim.want_terminal_obs = False
    ppo = DevicePPO(sim, cfg, PPOConfig(n_steps=16, batch_size=4096, n_epochs=2, hidden=64, neighbor_hidden=32))
    w0 = torch.cat([p.detach().reshape(-1).clone() for p in ppo.policy.parameters()])
    l0 = sim.launch_count
    hist = ppo.learn(3)
    n = cfg.num_envs * cfg.num_agents
    assert hist[-1]["agent_steps"] == 3 * 16 * n
    assert sim.launch_count - l0 == 3 * 16                      # one simulator launch per env step, nothing else
    for r in hist:
        assert all(np.isfinite(r[k]) for k in ("pg", "vf", "ent", "kl", "mean_reward"))
        assert r["minibatches"] == 2 * int(np.ceil(16 * n / 4096))
    w1 = torch.cat([p.detach().reshape(-1) for p in ppo.policy.parameters()])
    assert bool(torch.isfinite(w1).all()) and not torch.equal(w0, w1)
    assert ppo.obs_buf.is_cuda and ppo.adv.is_cuda
    assert sum(r["episodes"] for r in hist) > 0



@pytest.mark.parametrize("dtype_name", ["float32", "bfloat16"])
def test_fused_bias_tanh_layer_matches_autograd(dtype_name):
    """`TanhMLP` on CUDA (bias-free GEMM + `qp_bias_tanh` / `qp_bias_tanh_backward`) against the plain nn.Sequential it subclasses:
    outputs, input gradient, weight and bias gradients, with and without bf16 autocast."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import TanhMLP, _mlp
    torch.manual_seed(0)
    dev = torch.device("cuda:0")
    bf16 = dtype_name == "bfloat16"
    for sizes, n in (([24, 256, 256], 3001), ([6, 48, 48, 48], 517), ([512, 512], 1024)):
        a = _mlp(sizes).to(dev)
        assert isinstance(a, TanhMLP)
        b = torch.nn.Sequential(*[type(m)(m.in_features, m.out_features) if isinstance(m, torch.nn.Linear) else type(m)() for m in a]).to(dev)
        b.load_state_dict(a.state_dict())
        with torch.no_grad():
            for m in a:
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.5, 0.5)
            b.load_state_dict(a.state_dict())
        x = torch.randn(n, sizes[0], device=dev)
        xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        g = torch.randn(n, sizes[-1], device=dev)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            ya, yb = a(xa), b(xb)
        (ya.float() * g).sum().backward()
        (yb.float() * g).sum().backward()
        tol = 3e-2 if bf16 else 2e-5
        scale = lambda t: max(1.0, float(t.abs().max()))
        assert float((ya.float() - yb.float()).abs().max()) <= tol
        assert float((xa.grad - xb.grad).abs().max()) <= tol * scale(xb.grad)
        for (na, pa), (nb, pb) in zip(a.named_parameters(), b.named_parameters()):
            assert float((pa.grad - pb.grad).abs().max()) <= tol * scale(pb.grad), (sizes, na)
    a.fused = False                                                 # the switch gives the plain Sequential back
    with torch.no_grad():
        assert torch.equal(a(x), b(x))


FORK_K8 = dict(num_agents=8, neighbor_obs_type="dist_sangle_sheading", obs_repr="cdist_cdistdot_dist_distdot_sangle_angledot")
TRAINING_TOWERS = {
    # name: (config, hidden, neighbor_hidden, neighbour encoder)
    "cfg2": (lambda: QuadSimConfig(num_envs=2, num_agents=8), 256, 256, "mean_embed"),
    "k5_v3_narrow": (lambda: QuadSimConfig(num_envs=2, num_agents=5, neighbor_visible_num=3), 64, 48, "mean_embed"),
    "cfg2_mlp": (lambda: QuadSimConfig(num_envs=2, num_agents=8), 256, 256, "mlp"),                   # 36 neighbour inputs
    # S 6 and W * V 6: the self encoder's and the MLP's first layers take _FirstBiasTanh on a strided slice of the observation
    "fork_mlp": (lambda: QuadSimConfig.fork_default(num_envs=2), 256, 256, "mlp"),
    "fork_k8_sheading_mlp": (lambda: QuadSimConfig.fork_default(num_envs=2, **FORK_K8), 256, 256, "mlp"),   # S 7, 35 neighbour inputs
    "fork": (lambda: QuadSimConfig.fork_default(num_envs=2), 256, 256, "mean_embed"),
    "cfg3_obstacles": (lambda: QuadSimConfig(num_envs=2, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                                             obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2), 256, 256, "mean_embed"),
    "no_neighbours": (lambda: QuadSimConfig(num_envs=2, num_agents=1, neighbor_visible_num=0), 256, 256, "mean_embed"),
}


@pytest.mark.parametrize("autocast", [False, True])
def test_fused_encoder_training_path_matches_plain_autograd(autocast):
    """The whole tower on CUDA with gradients (TanhMLP pairs, `_FirstBiasTanh` on first layers of at most 8 inputs, the fused layer-2 /
    neighbour-mean tail `qp_bias_tanh_mean[_backward]`) against the same module with the fused path switched off: output and every
    parameter gradient, for every neighbour encoder the kernels serve (deep-sets, MLP, none) and the obstacle encoder."""
    import torch
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadEncoder, TanhMLP
    dev = torch.device("cuda:0")
    torch.manual_seed(1)
    for name, (make, hidden, nh, kind) in TRAINING_TOWERS.items():
        enc = QuadEncoder(make(), hidden=hidden, neighbor_hidden=nh, neighbor_encoder=kind).to(dev)
        assert enc.kind == ("none" if name == "no_neighbours" else kind)
        with torch.no_grad():
            for m in enc.modules():
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.4, 0.4)
        D = enc.S + enc.W * enc.V + enc.O
        obs = torch.randn(1500 + 7, D, device=dev)
        g = torch.randn(obs.shape[0], enc.out_size, device=dev)
        res = []
        for fused in (True, False):
            TanhMLP.fused = fused
            try:
                enc.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    y = enc(obs)
                (y.float() * g).sum().backward()
                res.append((y.detach().float().clone(), {n: p.grad.clone() for n, p in enc.named_parameters()}))
            finally:
                TanhMLP.fused = True
        tol = 4e-2 if autocast else 3e-5
        d_out = float((res[0][0] - res[1][0]).abs().max())
        worst = max(float((res[0][1][n] - res[1][1][n]).abs().max()) / max(1.0, float(res[1][1][n].abs().max())) for n in res[0][1])
        print(f"\n[{name}] autocast={autocast}: max |d out| {d_out:.1e}, max scaled |d grad| {worst:.1e}")
        assert d_out <= tol, name
        for n in res[0][1]:
            ref = res[1][1][n]
            assert float((res[0][1][n] - ref).abs().max()) <= tol * max(1.0, float(ref.abs().max())), (name, n)
