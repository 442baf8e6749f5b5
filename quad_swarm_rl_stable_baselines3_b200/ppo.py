"""Device-resident PPO over the CUDA simulator (SURVEY.md 8 f1): rollout storage, GAE and minibatching never leave HBM.

What it replaces: `stable_baselines3.PPO(...).learn()` as driven by `swarm_rl/sb_train.py:54-99` -- SB3's
`collect_rollouts` / `RolloutBuffer` are numpy-based, so every env step costs a D2H of the observations and an H2D of the
actions; at the simulator's throughput that host round trip is the only bottleneck left (SURVEY H1).  Here the policy reads
`QuadSwarmSim.step`'s CUDA tensors directly and the rollout is a set of preallocated CUDA tensors.

The policy mirrors the reference's `ActorCriticPolicyCustomSeparateWeights` (swarm_rl/models/ActorCriticPolicyCustom.py:284-556)
with a `QuadMultiEncoder` per tower (swarm_rl/models/quad_multi_model.py:250-354): self-observation MLP, neighbour encoder
('mlp' or deep-sets 'mean_embed'), optional obstacle MLP, tanh feed-forward to 2*rnn_size; separate actor and critic weights;
state-independent log-std diagonal Gaussian (log_std_init 0, no squashing), xavier-uniform initialisation.  The dense layers
of the torch module are plain PyTorch (cuBLAS) and are what the update differentiates; at rollout time the forward runs on the
hand-written tcgen05 kernel (`fused_policy.py`, csrc/policy_kernels.cu: both towers and heads in one launch, activations in
tensor memory; deep-sets or no neighbour encoder, with or without the obstacle encoder, or the 'mlp' neighbour encoder with at most
40 inputs and no obstacle encoder; parity against this module in tests/test_gpu_policy.py, tests/test_gpu_policy_obstacles.py and
tests/test_gpu_policy_mlp.py; the 'attention' encoder and the other 'mlp' policies stay on the torch path) and GAE on `qp_gae` (one launch).
SB3 itself is not installed; tests/test_ppo_reference.py pins `collect` + `update` against a float64 restatement of SB3 2.x's
`collect_rollouts`, `RolloutBuffer` and `PPO.train`: the rollout buffers (a replay of the simulator reproduces them bitwise, `logp_buf`
is the log-prob of the stored action, GAE), and for every minibatch, at the device's own parameters, the post-clip gradient (advantage
normalisation, Gaussian log-prob / entropy, clipped surrogate, value and entropy terms, global-norm clip) and the Adam step (eps 1e-5).
Measured gradient errors and tolerances are listed there and in DESIGN.md section 11.

Multi-GPU: one process per GPU, each with its own env shard (sharding.py); the only collectives are the gradient all-reduce
per minibatch (one flat NCCL buffer) and the episode-stat all-reduce per rollout.
"""
from __future__ import annotations

import math
import time
from dataclasses import asdict, dataclass
from typing import Dict, Optional

import torch
import torch.nn as nn

from .config import NEIGHBOR_OBS_DIM, OBS_REPR_DIM, QuadSimConfig


class _BiasTanh(torch.autograd.Function):
    """tanh(z + b) with a fused backward (`qp_bias_tanh[_backward]`): the bias gradient is reduced in the same pass that applies 1 - y^2."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, z, b):
        from . import fused_policy
        y = fused_policy.bias_tanh(z, b)
        ctx.save_for_backward(y)
        ctx.bias_dtype = b.dtype
        return y

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, gy):
        from . import fused_policy
        (y,) = ctx.saved_tensors
        gz, gb = fused_policy.bias_tanh_backward(gy, y)
        return gz, gb.to(ctx.bias_dtype)


class _FirstBiasTanh(torch.autograd.Function):
    """tanh(z + b) of a first layer with few inputs, z = x @ w^T computed outside without autograd: the backward returns the weight and bias
    gradients from one pass over (grad_y, y, x) and no grad_z at all (`qp_bias_tanh_backward_first`).  x must not need a gradient."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, z, x, w, b):
        from . import fused_policy
        y = fused_policy.bias_tanh(z, b)
        ctx.save_for_backward(y, x)
        ctx.dtypes = (w.dtype, b.dtype)
        return y

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, gy):
        from . import fused_policy
        y, x = ctx.saved_tensors
        gw, gb = fused_policy.bias_tanh_backward_first(gy, y, x)
        return None, None, gw.to(ctx.dtypes[0]), gb.to(ctx.dtypes[1])


class _BiasTanhMean(torch.autograd.Function):
    """mean over the V rows of each group of tanh(z + b): the deep-sets tail in one pass, backward without the expanded gradient."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, z, b, V):
        from . import fused_policy
        y, m = fused_policy.bias_tanh_mean(z, b, V)
        ctx.save_for_backward(y)
        ctx.V, ctx.bias_dtype = V, b.dtype
        return m

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, gm):
        from . import fused_policy
        (y,) = ctx.saved_tensors
        gz, gb = fused_policy.bias_tanh_mean_backward(gm, y, ctx.V)
        return gz, gb.to(ctx.bias_dtype), None


class TanhMLP(nn.Sequential):
    """nn.Sequential of Linear / Tanh modules (same parameter names).  On CUDA, when gradients are recorded, every (Linear, Tanh) pair runs
    as a bias-free GEMM (cuBLAS) followed by the fused bias + tanh kernel; everywhere else it is the plain Sequential."""
    fused = True

    def forward(self, x):
        if not (self.fused and x.is_cuda and torch.is_grad_enabled() and x.dtype in (torch.float32, torch.bfloat16)):
            return super().forward(x)
        mods = list(self)
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, nn.Linear) and i + 1 < len(mods) and isinstance(mods[i + 1], nn.Tanh) and m.out_features % 2 == 0 and m.bias is not None:
                if i == 0 and m.in_features <= 8 and m.out_features % 8 == 0 and x.dim() == 2 and not x.requires_grad:
                    with torch.no_grad():                                # first layer on raw observations: no input gradient, dW fused into the backward
                        z = torch.nn.functional.linear(x, m.weight)
                    x = _FirstBiasTanh.apply(z.contiguous(), x, m.weight, m.bias)
                else:
                    z = torch.nn.functional.linear(x, m.weight)
                    lead = z.shape[:-1]
                    x = _BiasTanh.apply(z.reshape(-1, z.shape[-1]).contiguous(), m.bias).reshape(*lead, z.shape[-1])
                i += 2
            else:
                x = m(x)
                i += 1
        return x


def _mlp(sizes, act=nn.Tanh):
    layers = []
    for a, b in zip(sizes[:-1], sizes[1:]):
        layers += [nn.Linear(a, b), act()]
    return TanhMLP(*layers)


class QuadEncoder(nn.Module):
    """One tower: QuadMultiEncoder (quad_multi_model.py:250-354)."""

    def __init__(self, cfg: QuadSimConfig, hidden: int = 256, neighbor_hidden: int = 256, neighbor_encoder: str = "mean_embed"):
        super().__init__()
        self.S = OBS_REPR_DIM[cfg.obs_repr]
        self.V = cfg.visible
        self.W = NEIGHBOR_OBS_DIM[cfg.neighbor_obs_type] if self.V > 0 else 0
        self.O = 9 if cfg.use_obstacles else 0
        self.kind = neighbor_encoder if self.V > 0 else "none"
        self.self_encoder = _mlp([self.S, hidden, hidden])
        out = hidden
        if self.kind == "mlp":                       # QuadNeighborhoodEncoderMlp (:104-122)
            self.neighbor = _mlp([self.W * self.V, neighbor_hidden, neighbor_hidden, neighbor_hidden])
            out += neighbor_hidden
        elif self.kind == "mean_embed":              # QuadNeighborhoodEncoderDeepsets (:23-41): phi(nbr_j) -- the neighbour row alone -- averaged
            self.neighbor = _mlp([self.W, neighbor_hidden, neighbor_hidden])
            out += neighbor_hidden
        elif self.kind == "attention":               # QuadNeighborhoodEncoderAttention (:42-102), the fork's default (global_cfg.py:71)
            self.neighbor = _mlp([self.S + self.W, neighbor_hidden, neighbor_hidden])                       # e_i = phi([self, nbr_i])
            self.neighbor_value = _mlp([neighbor_hidden, neighbor_hidden, neighbor_hidden])                 # h_i
            self.attention = TanhMLP(*_mlp([2 * neighbor_hidden, neighbor_hidden, neighbor_hidden]), nn.Linear(neighbor_hidden, 1))   # alpha_i
            out += neighbor_hidden
        elif self.kind != "none":
            raise NotImplementedError(f"neighbor_encoder {neighbor_encoder!r} (available: mlp, mean_embed, attention)")
        if self.O:
            self.obstacle = _mlp([self.O, hidden, hidden])
            out += hidden
        self.feed_forward = TanhMLP(nn.Linear(out, 2 * hidden), nn.Tanh())
        self.out_size = 2 * hidden

    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        s = obs[:, :self.S]
        parts = [self.self_encoder(s)]
        if self.kind == "mlp":
            parts.append(self.neighbor(obs[:, self.S:self.S + self.W * self.V]))
        elif self.kind == "mean_embed":
            nb = obs[:, self.S:self.S + self.W * self.V].reshape(-1, self.W)
            H = self.neighbor[-2].out_features
            if TanhMLP.fused and nb.is_cuda and torch.is_grad_enabled() and H % 8 == 0 and len(self.neighbor) == 4:
                # training on CUDA: layer 1 through the fused bias + tanh, layer 2 + the mean over neighbours in one pass (no [n * V, H] mean / division)
                h1 = self.neighbor[:2](nb)
                z2 = torch.nn.functional.linear(h1, self.neighbor[2].weight)
                parts.append(_BiasTanhMean.apply(z2.contiguous(), self.neighbor[2].bias, self.V))
            else:
                parts.append(self.neighbor(nb).reshape(-1, self.V, H).mean(dim=1))
        elif self.kind == "attention":
            # Quirk replicated (quad_multi_model.py:79-96): the neighbour rows are flattened batch-major ([b0 n0, b0 n1, ...]) but the self
            # observation and the mean embedding are tiled with .repeat(V, 1) ([b0, b1, ..., b0, b1, ...]), so for batch sizes > 1 row
            # b*V + j is paired with the self observation of batch element (b*V + j) mod n.  Exact only for n == 1; kept as the reference has it.
            n, H = s.shape[0], self.neighbor[-2].out_features
            nb = obs[:, self.S:self.S + self.W * self.V].reshape(-1, self.W)
            e = self.neighbor(torch.cat([s.repeat(self.V, 1), nb], dim=1))                     # e_i
            h = self.neighbor_value(e)                                                          # h_i
            em = e.reshape(n, -1, H).mean(dim=1)                                                # e_m
            alpha = torch.softmax(self.attention(torch.cat([e, em.repeat(self.V, 1)], dim=1)).view(n, -1), dim=1).view(-1, 1)
            parts.append((alpha * h).view(n, -1, H).sum(dim=1))
        if self.O:
            parts.append(self.obstacle(obs[:, self.S + self.W * self.V:]))
        return self.feed_forward(torch.cat(parts, dim=1))


class QuadActorCritic(nn.Module):
    """Separate actor / critic towers + diagonal Gaussian head (ActorCriticPolicyCustom.py:284-556)."""

    def __init__(self, cfg: QuadSimConfig, hidden: int = 256, neighbor_hidden: int = 256, neighbor_encoder: str = "mean_embed",
                 log_std_init: float = 0.0):
        super().__init__()
        self.actor = QuadEncoder(cfg, hidden, neighbor_hidden, neighbor_encoder)
        self.critic = QuadEncoder(cfg, hidden, neighbor_hidden, neighbor_encoder)
        self.action_net = nn.Linear(self.actor.out_size, cfg.act_dim)
        self.value_net = nn.Linear(self.critic.out_size, 1)
        self.log_std = nn.Parameter(torch.full((cfg.act_dim,), float(log_std_init)))
        for m in self.modules():                                  # :176-182, 405-411
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight, gain=1.0)
                nn.init.zeros_(m.bias)

    def dist(self, obs):
        # float32 Gaussian under bf16 autocast too (SB3's is float32): with the head's bf16 output as loc, act() would sample a bf16
        # action and take its log-prob with a bf16 (action - mean), which is then not the log-prob of the stored action to fp32 rounding
        mean = self.action_net(self.actor(obs)).float()
        # validate_args=False: the argument check reads a device boolean on the host (a sync per call, and illegal under graph capture)
        return torch.distributions.Normal(mean, self.log_std.exp().expand_as(mean), validate_args=False)

    def value(self, obs):
        return self.value_net(self.critic(obs)).squeeze(-1)

    @torch.no_grad()
    def act(self, obs):
        d = self.dist(obs)
        a = d.sample()
        return a, d.log_prob(a).sum(-1), self.value(obs)

    def evaluate(self, obs, actions):
        d = self.dist(obs)
        return d.log_prob(actions).sum(-1), d.entropy().sum(-1), self.value(obs)


def compute_gae(rewards, values, dones, last_values, gamma: float, lam: float):
    """SB3 `RolloutBuffer.compute_returns_and_advantage`: rewards/values/dones [T, n]; dones[t] marks the transition
    produced by step t (the env auto-reset after it), last_values [n] = V(s_T).  Returns (advantages, returns), [T, n]."""
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    last = torch.zeros_like(last_values)
    for t in reversed(range(T)):
        nonterminal = 1.0 - dones[t].to(rewards.dtype)
        next_v = last_values if t == T - 1 else values[t + 1]
        delta = rewards[t] + gamma * next_v * nonterminal - values[t]
        last = delta + gamma * lam * nonterminal * last
        adv[t] = last
    return adv, adv + values


@dataclass
class PPOConfig:
    n_steps: int = 128          # env.step calls per rollout (sb_train.py:58 uses 512 with 13 envs)
    batch_size: int = 32768     # minibatch rows
    n_epochs: int = 4           # sb_train.py:60 uses 10
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    learning_rate: float = 1e-4     # global_cfg.py:29
    normalize_advantage: bool = True
    hidden: int = 256
    neighbor_hidden: int = 256
    neighbor_encoder: str = "mean_embed"
    autocast_bf16: bool = False     # bf16 autocast for the dense layers (tensor cores); the simulator stays fp32
    fused_rollout: bool = True      # rollout-time forward on the tcgen05 kernel (fused_policy.py) when the architecture is the one it is built for



class DevicePPO:
    def __init__(self, sim, cfg: QuadSimConfig, ppo: Optional[PPOConfig] = None, seed: int = 0):
        self.sim, self.cfg, self.p = sim, cfg, ppo or PPOConfig()
        self.device = torch.device(sim.device)
        torch.manual_seed(seed)                                   # same initial weights on every rank
        self.policy = QuadActorCritic(cfg, self.p.hidden, self.p.neighbor_hidden, self.p.neighbor_encoder).to(self.device)
        self.opt = torch.optim.Adam(self.policy.parameters(), lr=self.p.learning_rate, eps=1e-5)
        # identical weights everywhere, but every rank draws its own exploration noise and minibatch permutations
        rank = torch.distributed.get_rank() if torch.distributed.is_available() and torch.distributed.is_initialized() else 0
        torch.manual_seed(seed + 1 + rank)
        n, T, D, A = cfg.num_envs * cfg.num_agents, self.p.n_steps, cfg.obs_dim, cfg.act_dim
        dev = self.device
        self.obs_buf = torch.empty((T, n, D), device=dev)
        self.act_buf = torch.empty((T, n, A), device=dev)
        self.logp_buf = torch.empty((T, n), device=dev)
        self.val_buf = torch.empty((T, n), device=dev)
        self.rew_buf = torch.empty((T, n), device=dev)
        self.done_buf = torch.empty((T, n), dtype=torch.bool, device=dev)
        self.world = torch.distributed.get_world_size() if torch.distributed.is_available() and torch.distributed.is_initialized() else 1
        self._flat = None
        self.obs = sim.reset().clone()
        self.total_agent_steps = 0
        self._rollout_pending = False                             # collect() filled the buffers, update() has not consumed them
        self.fused = None
        if self.p.fused_rollout and self.device.type == "cuda":
            from . import fused_policy
            if fused_policy.supported(self.policy):
                self.fused = fused_policy.FusedPolicy(self.policy, self.device)

    def _sync(self):
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

    def _autocast(self):
        return torch.autocast(self.device.type, dtype=torch.bfloat16, enabled=self.p.autocast_bf16)

    # ---- rollout: policy inference and env stepping, all on the device ---------------------------------------------
    @torch.no_grad()
    def collect(self) -> Dict[str, float]:
        p = self.p
        t0 = time.perf_counter()
        for t in range(p.n_steps):
            if self.fused is not None:
                a, logp, v = self.fused.act(self.obs)                    # one tcgen05 kernel: both towers, heads included
            else:
                with self._autocast():
                    a, logp, v = self.policy.act(self.obs)
            self.obs_buf[t].copy_(self.obs)
            self.act_buf[t].copy_(a); self.logp_buf[t].copy_(logp.float()); self.val_buf[t].copy_(v.float())
            obs, rew, done = self.sim.step(a.float().contiguous())       # the env clips the action itself (RawControl.step)
            self.rew_buf[t].copy_(rew); self.done_buf[t].copy_(done)
            self.obs.copy_(obs)                                          # sim.obs aliases a buffer that the next step overwrites
        if self.fused is not None:
            from . import fused_policy
            last_v = self.fused.forward(self.obs)[1]
            self.adv, self.ret = fused_policy.gae(self.rew_buf, self.val_buf, self.done_buf, last_v, p.gamma, p.gae_lambda)   # one launch
        else:
            with self._autocast():
                last_v = self.policy.value(self.obs).float()
            self.adv, self.ret = compute_gae(self.rew_buf, self.val_buf, self.done_buf, last_v, p.gamma, p.gae_lambda)
        self._sync()
        self._rollout_pending = True
        n = self.obs.shape[0]
        self.total_agent_steps += n * p.n_steps * self.world
        return {"rollout_s": time.perf_counter() - t0, "mean_reward": float(self.rew_buf.mean()),
                "done_frac": float(self.done_buf.float().mean())}

    def _flatten_grads(self):
        """Every parameter's .grad becomes a view into one flat buffer (once): the gradient all-reduce is then ONE NCCL call on that buffer
        with no gather / scatter copies around it, and zero_grad(set_to_none=False) is one memset-like pass."""
        params = [q for q in self.policy.parameters() if q.requires_grad]
        self._flat = torch.zeros(sum(q.numel() for q in params), device=self.device, dtype=params[0].dtype)
        off = 0
        for q in params:
            q.grad = self._flat[off:off + q.numel()].view_as(q)
            off += q.numel()

    def _allreduce_grads(self):
        if self.world == 1:
            return
        torch.distributed.all_reduce(self._flat)                  # NCCL over NVLink: the gradient all-reduce
        self._flat.div_(self.world)

    # ---- PPO update: minibatches gathered on the device ------------------------------------------------------------
    def _minibatch_loss(self, obs_mb, act_mb, logp_old_mb, adv_mb, ret_mb, acc):
        """Clipped-surrogate PPO loss of one minibatch (SB3 PPO.train); adds the five diagnostics to `acc` on the device."""
        p = self.p
        if p.normalize_advantage and adv_mb.numel() > 1:
            adv_mb = (adv_mb - adv_mb.mean()) / (adv_mb.std() + 1e-8)
        with self._autocast():
            logp, ent, v = self.policy.evaluate(obs_mb, act_mb)
        logp, ent, v = logp.float(), ent.float(), v.float()
        ratio = (logp - logp_old_mb).exp()
        pg = -torch.min(adv_mb * ratio, adv_mb * ratio.clamp(1 - p.clip_range, 1 + p.clip_range)).mean()
        vf = torch.nn.functional.mse_loss(v, ret_mb)
        loss = pg + p.vf_coef * vf - p.ent_coef * ent.mean()
        with torch.no_grad():
            acc += torch.stack([pg.detach(), vf.detach(), ent.mean(), (logp_old_mb - logp).mean(), ((ratio - 1).abs() > p.clip_range).float().mean()])
        return loss

    def update(self) -> Dict[str, float]:
        """PPO.train of SB3: n_epochs passes over the rollout in shuffled minibatches.  Measured on the device (round 2): capturing the
        minibatch step in CUDA graphs buys 4 % (0.365 -> 0.349 s per 4.2 M samples) -- the step is bound by its ~5.5 ms of GPU work per
        65536 rows (tanh / cast / reduction kernels around small-K GEMMs), not by launches -- so the plain eager step ships."""
        p = self.p
        t0 = time.perf_counter()
        T, n = self.rew_buf.shape
        total = T * n
        obs = self.obs_buf.view(total, -1); act = self.act_buf.view(total, -1)
        logp_old = self.logp_buf.view(total); adv = self.adv.reshape(total); ret = self.ret.reshape(total)
        acc = torch.zeros(5, device=self.device)                    # pg, vf, ent, kl, clip_frac: summed on the device, read once
        nb = 0
        for _ in range(p.n_epochs):
            perm = torch.randperm(total, device=self.device)
            for s in range(0, total, p.batch_size):
                idx = perm[s:s + p.batch_size]
                loss = self._minibatch_loss(obs[idx], act[idx], logp_old[idx], adv[idx], ret[idx], acc)
                if self._flat is None:
                    self._flatten_grads()
                self._flat.zero_()                                     # = opt.zero_grad(set_to_none=False) on the flat views
                loss.backward()
                self._allreduce_grads()
                # nn.utils.clip_grad_norm_ on the flat buffer: total 2-norm, scale by min(1, max_norm / (norm + 1e-6))
                self._flat.mul_((p.max_grad_norm / (self._flat.norm() + 1e-6)).clamp(max=1.0))
                self.opt.step()
                nb += 1
        if self.fused is not None:
            self.fused.sync()                                          # re-pack the updated weights for the next rollout
        self._sync()
        self._rollout_pending = False
        out = dict(zip(("pg", "vf", "ent", "kl", "clip_frac"), (acc / max(nb, 1)).tolist()))
        out["update_s"] = time.perf_counter() - t0
        out["minibatches"] = nb
        return out

    def learn(self, iterations: int, log=None):
        hist = []
        for it in range(iterations):
            r = self.collect()
            u = self.update()
            es = self.sim.episode_stats(reset=True, reduce=self.world > 1)      # the episode-stat all-reduce
            row = dict(iteration=it, agent_steps=self.total_agent_steps, episodes=es["episodes"], **r, **u)
            hist.append(row)
            if log:
                log(row)
        return hist

    # ---- checkpoints (SB3 model.save / CheckpointCallback) ---------------------------------------------------------
    CHECKPOINT_VERSION = 1

    def save(self, path) -> None:
        """Write a checkpoint between iterations: configurations, policy and Adam state, step count, the last observation, the torch
        RNG states (exploration noise, minibatch permutations) and the exact simulator snapshot.  Only tensors and plain containers,
        so `torch.load(path, weights_only=True)` reads it.  Under torchrun every rank saves its own file (its env shard).  The rollout
        buffers are not saved: saving between collect() and update() raises RuntimeError."""
        if self._rollout_pending:
            raise RuntimeError("DevicePPO.save: collect() filled a rollout that update() has not used yet; save between iterations")
        self._sync()
        ckpt = {
            "version": self.CHECKPOINT_VERSION,
            "ppo_config": asdict(self.p),
            "sim_config": asdict(self.cfg),
            "policy": self.policy.state_dict(),
            "optimizer": self.opt.state_dict(),
            "total_agent_steps": self.total_agent_steps,
            "obs": self.obs.cpu(),
            "rng_cpu": torch.get_rng_state(),
            "rng_cuda": torch.cuda.get_rng_state(self.device) if self.device.type == "cuda" else None,
            "sim": self.sim.snapshot(),
        }
        torch.save(ckpt, path)

    def load(self, path) -> None:
        """Resume from `save(path)` on a freshly built DevicePPO whose simulator has the same configuration (the simulator rejects
        another one; the policy architecture must match exactly).  The live PPOConfig keeps the optimisation hyperparameters: the
        learning rate is set back to `self.p.learning_rate` after Adam's state is loaded.  The next collect() continues the saved
        run bitwise."""
        ckpt = torch.load(path, map_location="cpu", weights_only=True)
        if ckpt.get("version") != self.CHECKPOINT_VERSION:
            raise ValueError(f"DevicePPO.load: checkpoint format {ckpt.get('version')!r}, this code reads {self.CHECKPOINT_VERSION}")
        if tuple(ckpt["obs"].shape) != tuple(self.obs.shape):
            raise ValueError(f"DevicePPO.load: checkpoint observations {tuple(ckpt['obs'].shape)}, this run's {tuple(self.obs.shape)}")
        self.sim.restore(ckpt["sim"])
        self.policy.load_state_dict(ckpt["policy"], strict=True)
        self.opt.load_state_dict(ckpt["optimizer"])
        for g in self.opt.param_groups:
            g["lr"] = self.p.learning_rate
        self.total_agent_steps = int(ckpt["total_agent_steps"])
        self.obs.copy_(ckpt["obs"])
        torch.set_rng_state(ckpt["rng_cpu"])
        if self.device.type == "cuda":
            torch.cuda.set_rng_state(ckpt["rng_cuda"], self.device)
        self._rollout_pending = False
        if self.fused is not None:
            self.fused.sync()
        self._sync()

    def load_shards(self, paths) -> None:
        """Resume on another number of GPUs: load this rank's envs from the rank files `save` wrote in a run of any world size, into a
        freshly built DevicePPO whose simulator config is the saved one but for `num_envs` / `env_id_offset` (e.g. `shard_config` of
        the same total for the new world size).  Every rank may pass the full list of old files: the files are memory-mapped and only
        the headers, the replicated policy / Adam state and this rank's slices are read.  Nothing this object keeps refers to the
        mapped files afterwards, so a later `save` may overwrite them.
        Checks that every file has the same checkpoint version and step count, bitwise-identical policy and optimizer tensors (the
        gradient all-reduce keeps them so; ValueError naming the first tensor that differs otherwise) and the same simulator config
        up to `num_envs` / `env_id_offset`; the simulator then rejects gaps, overlaps and shards of different steps
        (`QuadSwarmSim.restore_shards`).
        The simulator continues bitwise where the old shards stood; the policy and Adam state are the saved ones, with the learning
        rate set back to the live PPOConfig as in `load`.  The torch RNG states stay those this instance was built with: the exploration
        noise and minibatch order after a resharded resume are not those of any continued run.  A resume on the same number of GPUs
        should use `load`, which is bitwise."""
        paths = list(paths)
        if not paths:
            raise ValueError("DevicePPO.load_shards: no checkpoint files")
        cks = [torch.load(p, map_location="cpu", weights_only=True, mmap=True) for p in paths]
        for p, ck in zip(paths, cks):
            if ck.get("version") != self.CHECKPOINT_VERSION:
                raise ValueError(f"DevicePPO.load_shards: {p}: checkpoint format {ck.get('version')!r}, this code reads {self.CHECKPOINT_VERSION}")
            if ck["total_agent_steps"] != cks[0]["total_agent_steps"]:
                raise ValueError(f"DevicePPO.load_shards: {p}: total_agent_steps {ck['total_agent_steps']}, {paths[0]}: "
                                 f"{cks[0]['total_agent_steps']} (files of different iterations)")
            want = asdict(self.cfg)
            for k, v in ck["sim_config"].items():
                if k not in ("num_envs", "env_id_offset") and want.get(k) != v:
                    raise ValueError(f"DevicePPO.load_shards: {p}: sim_config.{k} is {v!r}, this run's {want.get(k)!r}")
            rows = ck["sim_config"]["num_envs"] * self.cfg.num_agents
            if tuple(ck["obs"].shape) != (rows, self.obs.shape[1]):
                raise ValueError(f"DevicePPO.load_shards: {p}: observations {tuple(ck['obs'].shape)}, its "
                                 f"{ck['sim_config']['num_envs']} envs need {(rows, self.obs.shape[1])}")
            for what in ("policy", "optimizer"):
                name = _first_difference(cks[0][what], ck[what], what)
                if name is not None:
                    raise ValueError(f"DevicePPO.load_shards: {p}: {name} differs from {paths[0]}'s (the policy and Adam state of "
                                     f"the ranks of one run are identical)")
        self.sim.restore_shards([ck["sim"] for ck in cks])
        # this rank's rows of the saved observations (DevicePPO.obs; the simulator's own copy came with restore_shards)
        lo, hi, K = self.cfg.env_id_offset, self.cfg.env_id_offset + self.cfg.num_envs, self.cfg.num_agents
        for ck in cks:
            b0 = ck["sim_config"]["env_id_offset"]
            a, b = max(lo, b0), min(hi, b0 + ck["sim_config"]["num_envs"])
            if a < b:
                self.obs[(a - lo) * K:(b - lo) * K].copy_(ck["obs"][(a - b0) * K:(b - b0) * K])
        self.policy.load_state_dict(cks[0]["policy"], strict=True)            # copies into the parameters
        # Adam keeps the CPU `step` tensors it is given: hand it copies, or they would stay views of the memory-mapped file, which
        # a later save to that path truncates under them
        self.opt.load_state_dict(_owned(cks[0]["optimizer"]))
        for g in self.opt.param_groups:
            g["lr"] = self.p.learning_rate
        self.total_agent_steps = int(cks[0]["total_agent_steps"])
        self._rollout_pending = False
        if self.fused is not None:
            self.fused.sync()
        self._sync()


def _owned(x):
    """A copy of a state dict whose tensors own their memory (none is a view of a memory-mapped checkpoint)."""
    if isinstance(x, dict):
        return {k: _owned(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return type(x)(_owned(v) for v in x)
    return x.clone() if torch.is_tensor(x) else x


def _first_difference(a, b, name: str):
    """The dotted name of the first tensor or value in which two state dicts differ (tensors bitwise), or None."""
    if isinstance(a, dict) and isinstance(b, dict):
        if list(a) != list(b):
            return f"{name} (keys)"
        for k in a:
            d = _first_difference(a[k], b[k], f"{name}.{k}")
            if d is not None:
                return d
        return None
    if isinstance(a, (list, tuple)) and isinstance(b, (list, tuple)):
        if len(a) != len(b):
            return f"{name} (length)"
        for i, (x, y) in enumerate(zip(a, b)):
            d = _first_difference(x, y, f"{name}.{i}")
            if d is not None:
                return d
        return None
    if torch.is_tensor(a) and torch.is_tensor(b):
        same = (a.dtype == b.dtype and a.shape == b.shape
                and torch.equal(a.contiguous().reshape(-1).view(torch.uint8), b.contiguous().reshape(-1).view(torch.uint8)))
        return None if same else name
    return None if (type(a) is type(b) and a == b) else name
