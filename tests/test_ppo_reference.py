"""DevicePPO's rollout (`collect`) and update (`update`) against a float64 restatement of SB3 2.x's `collect_rollouts`,
`RolloutBuffer` and `PPO.train`.

SB3 is not installed, so the reference is written out here and calls none of `DevicePPO._minibatch_loss`, `ppo.compute_gae` or
`QuadActorCritic.dist / evaluate / act`.  It runs the module's towers (`actor`, `critic`, `action_net`, `value_net`, themselves pinned
against the reference's QuadMultiEncoder in tests/test_ppo_cpu.py) on a float64 copy of the parameters, and restates around them:
  * the minibatch loss: advantages normalised with the unbiased std + 1e-8 when the minibatch has more than one row; the diagonal
    Gaussian's log-prob and entropy; ratio = exp(logp - logp_old); the clipped surrogate; vf_coef * MSE; - ent_coef * mean entropy;
  * the global-norm gradient clip, scale min(1, max_norm / (||g|| + 1e-6));
  * Adam as torch computes it, with SB3's settings: betas (0.9, 0.999), eps 1e-5, no weight decay;
  * GAE / returns (SB3's recursion, returns = advantages + values before any normalisation);
  * the minibatch indices: one randperm(total) per epoch from the generator state before update(), sliced into batch_size rows,
    the last, partial slice kept.

Recording: `ppo.opt.step` is wrapped on the instance, and keeps for every minibatch k the parameters before the step (theta_k), the
post-clip gradient (`ppo._flat`) and the parameters after.  Every minibatch is compared at the device's own theta_k, so differences do
not accumulate over the Adam steps (the bias-gradient kernels reduce with atomics and are not bitwise repeatable).  Per minibatch:
  * the post-clip gradient, as a whole and per parameter tensor, against the reference's;
  * theta_{k+1} against the restated Adam step applied to the device's own gradient (this pins lr, betas and eps);
and per update the five diagnostics `update()` returns and the number of minibatches.

Clip-boundary rows: a row whose float64 ratio lies within MARGIN of 1 +- clip_range can take the other branch of the min in fp32 or
bf16.  Such rows are counted, and their own surrogate-gradient contribution (one more float64 backward) widens that minibatch's tolerance.

Rollout: the simulator state before collect() is replayed with the stored actions and must reproduce obs / reward / done bitwise; the
stored actions are float32 and unclipped; logp_buf is the log-prob of the stored action under the rollout's own mean; adv / ret are the
float64 GAE of the stored buffers.  With the fused rollout forward, its mean and value stay within tests/test_gpu_policy.py's
TOL_FP32_MAX of the float64 module, and the largest |log ratio| at epoch 0, minibatch 0 (theta is still the rollout's) -- the shift the
bf16 rollout adds to PPO's ratio -- is bounded by measurement.

Every case asserts the conditions that make it able to fail: episodes end inside the rollout; total % batch_size != 0 (one case
has a last minibatch of exactly one row); ent_coef != 0 and a learning rate at which later minibatches clip; log_std random in
[-1.5, 0.5] (log_std_init 0 would hide a missing - log_std term).

The CPU cases run DevicePPO on the oracle-backed TensorOracleSim of tests/test_ppo_cpu.py; the gpu cases on QuadSwarmSim.
"""
import contextlib
import copy
import math
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig  # noqa: E402
from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig, TanhMLP  # noqa: E402
from test_gpu_policy import TOL_FP32_MAX  # noqa: E402
from test_ppo_cpu import TensorOracleSim  # noqa: E402

gpu = pytest.mark.gpu
LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)
BETAS, ADAM_EPS = (0.9, 0.999), 1e-5                 # SB3's PPO: th.optim.Adam(..., eps=1e-5)
MARGIN = {False: 1e-4, True: 3e-2}                   # clip-boundary margin on the float64 ratio: fp32 / bf16 autocast update
FP32_ULP = 2.0 ** -23


# ---- the float64 reference --------------------------------------------------------------------------------------------------
def gauss_logp(a, mean, log_std):
    """log N(a; mean, exp(log_std)) summed over the action dimensions."""
    z = (a - mean) / log_std.exp()
    return (-0.5 * z * z - log_std - LOG_SQRT_2PI).sum(-1)


def gauss_entropy(log_std):
    return (0.5 + LOG_SQRT_2PI + log_std).sum(-1)


def gae64(rew, val, done, last_v, gamma, lam):
    """SB3 RolloutBuffer.compute_returns_and_advantage in float64: done[t] ends the episode of step t's transition."""
    rew, val, last_v = rew.double(), val.double(), last_v.double()
    nonterminal = 1.0 - done.double()
    adv = torch.zeros_like(rew)
    last = torch.zeros_like(last_v)
    for t in reversed(range(rew.shape[0])):
        next_v = last_v if t == rew.shape[0] - 1 else val[t + 1]
        delta = rew[t] + gamma * next_v * nonterminal[t] - val[t]
        last = delta + gamma * lam * nonterminal[t] * last
        adv[t] = last
    return adv, adv + val


def clip_scale(gnorm, max_norm):
    """torch.nn.utils.clip_grad_norm_: scale by min(1, max_norm / (||g|| + 1e-6))."""
    return min(1.0, max_norm / (gnorm + 1e-6))


class Adam64:
    """torch.optim.Adam's arithmetic in float64 (no weight decay, no amsgrad): bias-corrected step size, eps added after dividing
    sqrt(v) by sqrt(1 - beta2^t)."""

    def __init__(self, numel, lr, betas=BETAS, eps=ADAM_EPS):
        self.lr, self.betas, self.eps = lr, betas, eps
        self.m = torch.zeros(numel, dtype=torch.float64)
        self.v = torch.zeros(numel, dtype=torch.float64)
        self.t = 0

    def step(self, theta, g):
        b1, b2 = self.betas
        self.t += 1
        self.m = b1 * self.m + (1 - b1) * g
        self.v = b2 * self.v + (1 - b2) * g * g
        denom = (self.v.sqrt() / math.sqrt(1 - b2 ** self.t)) + self.eps
        return theta - (self.lr / (1 - b1 ** self.t)) * self.m / denom


@contextlib.contextmanager
def plain_torch():
    """The towers as plain nn.Sequential (the fused bias + tanh kernels take float32 / bf16 only)."""
    fused = TanhMLP.fused
    TanhMLP.fused = False
    try:
        yield
    finally:
        TanhMLP.fused = fused


class Reference:
    """A float64 copy of the policy; `minibatch` evaluates SB3's PPO.train loss at given parameters."""

    def __init__(self, ppo):
        self.p = ppo.p
        self.names = [n for n, _ in ppo.policy.named_parameters()]
        self.sizes = [q.numel() for q in ppo.policy.parameters()]
        self.pol = copy.deepcopy(ppo.policy).double()
        for q in self.pol.parameters():
            q.grad = None
        self.params = list(self.pol.parameters())

    def load(self, theta):
        torch.nn.utils.vector_to_parameters(theta.to(self.params[0].device, torch.float64), self.params)

    def forward(self, obs):
        with plain_torch():
            mean = self.pol.action_net(self.pol.actor(obs))
            value = self.pol.value_net(self.pol.critic(obs)).squeeze(-1)
        return mean, value

    def split(self, flat):
        return dict(zip(self.names, flat.split(self.sizes)))

    def minibatch(self, theta, obs, act, logp_old, adv, ret, margin):
        """(post-clip gradient, clip scale, diagnostics [pg, vf, ent, kl, clip_frac], number of clip-boundary rows, bound on what they can
        move the post-clip gradient by, log ratio logp - logp_old of every row)."""
        p = self.p
        self.load(theta)
        obs, act, logp_old, adv, ret = (x.double() for x in (obs, act, logp_old, adv, ret))
        if p.normalize_advantage and adv.numel() > 1:
            adv = (adv - adv.mean()) / (adv.std(unbiased=True) + 1e-8)
        mean, value = self.forward(obs)
        log_std = self.pol.log_std
        logp = gauss_logp(act, mean, log_std)
        ent = gauss_entropy(log_std).expand(logp.shape[0])
        ratio = (logp - logp_old).exp()
        surr = torch.min(adv * ratio, adv * ratio.clamp(1 - p.clip_range, 1 + p.clip_range))
        pg = -surr.mean()
        vf = ((value - ret) ** 2).mean()
        loss = pg + p.vf_coef * vf - p.ent_coef * ent.mean()
        g = torch.cat([x.reshape(-1) for x in torch.autograd.grad(loss, self.params, retain_graph=True)])
        scale = clip_scale(float(g.norm()), p.max_grad_norm)
        with torch.no_grad():
            near = ((ratio - (1 - p.clip_range)).abs() < margin) | ((ratio - (1 + p.clip_range)).abs() < margin)
        widen = 0.0
        for i in near.nonzero().reshape(-1).tolist():
            # a boundary row adds -adv * grad(ratio) / rows on the unclipped branch and nothing on the other; any subset of them may
            # flip, so the bound is the sum of the rows' own norms
            gb = torch.autograd.grad(-adv[i] * ratio[i] / ratio.shape[0], self.params, retain_graph=True, allow_unused=True)
            widen += scale * math.sqrt(sum(float(x.pow(2).sum()) for x in gb if x is not None))
        with torch.no_grad():
            diag = torch.stack([pg, vf, ent.mean(), (logp_old - logp).mean(), ((ratio - 1).abs() > p.clip_range).double().mean()])
        return (g * scale).detach(), scale, diag.detach(), int(near.sum()), widen, (logp - logp_old).detach()


def permutations(ppo, rng_state, total):
    """The update's minibatch indices: one randperm(total) per epoch from the generator state captured before update()."""
    cuda = ppo.device.type == "cuda"
    after = torch.cuda.get_rng_state(ppo.device) if cuda else torch.get_rng_state()
    if cuda:
        torch.cuda.set_rng_state(rng_state, ppo.device)
    else:
        torch.set_rng_state(rng_state)
    perms = [torch.randperm(total, device=ppo.device) for _ in range(ppo.p.n_epochs)]
    if cuda:
        torch.cuda.set_rng_state(after, ppo.device)
    else:
        torch.set_rng_state(after)
    return [perm[s:s + ppo.p.batch_size] for perm in perms for s in range(0, total, ppo.p.batch_size)]


def rng_state(ppo):
    return torch.cuda.get_rng_state(ppo.device) if ppo.device.type == "cuda" else torch.get_rng_state()


class Recorder:
    """Wraps ppo.opt.step on the instance: (theta before, post-clip gradient, theta after) of every minibatch, on the CPU in float64."""

    def __init__(self, ppo):
        self.steps = []
        params = list(ppo.policy.parameters())
        inner = ppo.opt.step

        def step(*args, **kw):
            before = torch.nn.utils.parameters_to_vector(params).detach().double().cpu()
            grad = ppo._flat.detach().double().cpu()
            out = inner(*args, **kw)
            after = torch.nn.utils.parameters_to_vector(params).detach().double().cpu()
            self.steps.append((before, grad, after))
            return out

        ppo.opt.step = step


# ---- cases ------------------------------------------------------------------------------------------------------------------
# Upstream episodes of 0.12 s are 12 control steps and fork episodes of 1 s are 12.5 calls, so every case's episodes end inside its
# 16-step rollout.  PPO settings shared by all cases unless a case overrides them:
PPO_BASE = dict(n_steps=16, n_epochs=3, ent_coef=0.01, learning_rate=3e-3)


def cfg2(n, **kw):
    return QuadSimConfig(num_envs=n, num_agents=8, ep_time=0.12, seed=1, **kw)


def cfg3(n):
    return QuadSimConfig(num_envs=n, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                         obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2, ep_time=0.12, seed=2)


def fork(n):
    return QuadSimConfig.fork_default(num_envs=n, ep_time=1.0, seed=3)


def k1(n):
    return QuadSimConfig(num_envs=n, num_agents=1, neighbor_obs_type="none", neighbor_visible_num=0, ep_time=0.12, seed=4)


# name: (sim config, PPOConfig overrides, tolerances).  Tolerances, at 3-5x the largest value measured (CPU cases on the oracle; gpu cases on
# an NVIDIA B200 at its 1000 W power limit):
#   grad: ||g_dev - g_ref|| / ||g_ref|| of every minibatch's post-clip gradient (measured fp32 5.2e-6 CPU, 1.2e-6 B200; bf16 autocast 1.5e-2);
#   tensor: the same per parameter tensor (fp32 1.6e-5; bf16 7.5e-2);
#   adam: |dtheta_dev - dtheta_ref| beyond one fp32 ulp of theta, in units of the learning rate (3.1e-7);
#   diag: |d_dev - d_ref| / (1 + |d_ref|) of pg / vf / ent / kl, clip_frac beyond its boundary rows (fp32 8.3e-8; bf16 4.3e-4);
#   logratio: largest |log ratio| of logp_buf against the float64 module at epoch 0, minibatch 0 (fp32 torch rollout 2.8e-6; fused bf16
#   rollout 3.5e-2; torch rollout under bf16 autocast 4.1e-2).  None for the attention encoder: it pairs each row with other rows of the
#   same batch (quad_multi_model.py:79-96, replicated), so a minibatch's outputs differ from the rollout's in float64 too (1.2 measured).
FP32_TOL = dict(grad=2e-5, tensor=6e-5, adam=1.5e-6, diag=3e-7, logratio=1e-5)
FUSED_TOL = dict(FP32_TOL, logratio=0.15)
BF16_TOL = dict(grad=5e-2, tensor=0.25, adam=1.5e-6, diag=2e-3, logratio=0.15)
CPU_TOL = FP32_TOL
CPU_CASES = {
    "cfg2_h64": (lambda: cfg2(8), dict(hidden=64, neighbor_hidden=64, batch_size=100), CPU_TOL),          # 1024 rows: 10 x 100 + 24
    "cfg3_h32_last_row_alone": (lambda: cfg3(4), dict(hidden=32, neighbor_hidden=32, batch_size=73), CPU_TOL),   # 512 rows: 7 x 73 + 1
    "fork_attention_h32": (lambda: fork(6), dict(hidden=32, neighbor_hidden=32, neighbor_encoder="attention", batch_size=90),
                           dict(CPU_TOL, logratio=None)),                                               # 384 rows: 4 x 90 + 24
}
GPU_CASES = {
    "cfg2_fused_fp32": (lambda: cfg2(16), dict(batch_size=700), FUSED_TOL),                                 # 2048 rows: 2 x 700 + 648
    "cfg2_fused_bf16_cfg5_ppo": (lambda: cfg2(16), dict(batch_size=65536, n_epochs=1, autocast_bf16=True),  # the benchmark's settings
                                 dict(BF16_TOL, logratio=FUSED_TOL["logratio"])),
    "cfg2_fused_bf16_minibatches": (lambda: cfg2(16), dict(batch_size=700, autocast_bf16=True), dict(BF16_TOL, logratio=FUSED_TOL["logratio"])),
    "cfg3_fused_obstacles": (lambda: cfg3(20), dict(batch_size=853), FUSED_TOL),                            # 2560 rows: 3 x 853 + 1
    "cfg2_fused_mlp": (lambda: cfg2(16), dict(batch_size=700, neighbor_encoder="mlp"), FUSED_TOL),
    "fork_fused": (lambda: fork(32), dict(batch_size=700), FUSED_TOL),                                      # 2048 rows
    "k1_fused": (lambda: k1(128), dict(batch_size=700), FUSED_TOL),                                         # 2048 rows
    "cfg2_torch_h64_fp32": (lambda: cfg2(16), dict(hidden=64, neighbor_hidden=64, batch_size=700), FP32_TOL),
    "cfg2_torch_h64_bf16": (lambda: cfg2(16), dict(hidden=64, neighbor_hidden=64, batch_size=700, autocast_bf16=True), BF16_TOL),
    "fork_torch_attention_h64": (lambda: fork(32), dict(hidden=64, neighbor_hidden=64, neighbor_encoder="attention", batch_size=700),
                                 dict(FP32_TOL, logratio=None)),
}


def make_ppo(sim, cfg, kw, seed=0):
    pc = PPOConfig(**{**PPO_BASE, **kw})
    ppo = DevicePPO(sim, cfg, pc, seed=seed)
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():                    # random log_std in [-1.5, 0.5]: log_std_init 0 would hide a missing - log_std term
        ppo.policy.log_std.copy_(torch.rand(cfg.act_dim, generator=g) * 2.0 - 1.5)
    return ppo


def case_conditions(ppo):
    p = ppo.p
    total = ppo.rew_buf.numel()
    assert bool(ppo.done_buf.any()), "no episode ended inside the rollout"
    assert total % p.batch_size != 0, "the case has no partial last minibatch"
    assert p.ent_coef != 0.0
    ls = ppo.policy.log_std.detach()
    assert float(ls.min()) >= -1.5 and float(ls.max()) <= 0.5 and float(ls.max() - ls.min()) > 0.1


def rollout_forward(ppo, obs):
    """(mean, value) as the rollout computed them: on the fused kernel, or on the torch module under the same autocast."""
    if ppo.fused is not None:
        return ppo.fused.forward(obs)
    with torch.no_grad(), ppo._autocast():
        return ppo.policy.action_net(ppo.policy.actor(obs)).float(), ppo.policy.value(obs).float()


def last_values(ppo):
    if ppo.fused is not None:
        return ppo.fused.forward(ppo.obs)[1]
    with torch.no_grad(), ppo._autocast():
        return ppo.policy.value(ppo.obs).float()


# ---- rollout ----------------------------------------------------------------------------------------------------------------
def check_rollout(ppo, replay_sim, replay_obs0, name):
    """collect() once, replay it on `replay_sim` (which stands where ppo.sim stood), then update() and collect() again."""
    p = ppo.p
    ppo.collect()
    T = p.n_steps
    case_conditions(ppo)

    # the buffers: obs_buf[t] is the observation act_buf[t] was taken on; rew / done of the transition it caused
    assert torch.equal(ppo.obs_buf[0], replay_obs0.to(ppo.obs_buf.device)), "obs_buf[0] is not the observation collect() started from"
    for t in range(T):
        o, r, d = replay_sim.step(ppo.act_buf[t].clone())
        nxt = ppo.obs_buf[t + 1] if t + 1 < T else ppo.obs
        assert torch.equal(o.to(nxt.device), nxt), f"obs_buf[{t + 1}] is not what the simulator returned for act_buf[{t}]"
        assert torch.equal(r.to(nxt.device), ppo.rew_buf[t]), f"rew_buf[{t}]"
        assert torch.equal(d.to(nxt.device).bool(), ppo.done_buf[t]), f"done_buf[{t}]"

    # actions: float32, unclipped (the env clips them itself), as SB3 stores them
    assert ppo.act_buf.dtype == torch.float32
    assert float(ppo.act_buf.abs().max()) > 1.0, "the stored actions look clipped"

    # logp_buf: the log-prob of the stored action under the rollout's own mean, to fp32 rounding; val_buf: the rollout's value
    log_std = ppo.policy.log_std.detach().double()
    worst = 0.0
    for t in range(T):
        mean, value = rollout_forward(ppo, ppo.obs_buf[t])
        ref = gauss_logp(ppo.act_buf[t].double(), mean.double(), log_std)
        err = (ppo.logp_buf[t].double() - ref).abs() / (1.0 + ref.abs())
        worst = max(worst, float(err.max()))
        assert torch.equal(value, ppo.val_buf[t]), f"val_buf[{t}] is not the rollout's value of obs_buf[{t}]"
    print(f"[{name}] logp_buf vs the log-prob of act_buf under the rollout's mean: max rel {worst:.2e}")    # measured <= 2.1e-7
    assert worst <= 1e-6, f"logp_buf is not the log-prob of the stored action (max rel err {worst:.2e})"
    if p.autocast_bf16 and ppo.fused is None:        # sampled in float32, not rounded to bf16 with the head's output
        assert not torch.equal(ppo.act_buf, ppo.act_buf.bfloat16().float()), "the stored actions are bf16 values"

    # the fused kernel's mean / value against the float64 module
    if ppo.fused is not None:
        ref = Reference(ppo)
        obs = ppo.obs_buf.reshape(-1, ppo.obs_buf.shape[-1])
        with torch.no_grad():
            m64, v64 = ref.forward(obs.double())
            mk, vk = ppo.fused.forward(obs)
        dm, dv = float((mk.double() - m64).abs().max()), float((vk.double() - v64).abs().max())
        print(f"[{name}] fused rollout forward vs float64 module: mean {dm:.2e}, value {dv:.2e}")
        assert dm <= TOL_FP32_MAX and dv <= TOL_FP32_MAX

    # adv / ret: float64 GAE of the stored buffers, with V(s_T) recomputed
    a64, r64 = gae64(ppo.rew_buf, ppo.val_buf, ppo.done_buf, last_values(ppo), p.gamma, p.gae_lambda)
    scale = 1.0 + float(a64.abs().max())
    ea, er = float((ppo.adv.double() - a64).abs().max()) / scale, float((ppo.ret.double() - r64).abs().max()) / (1.0 + float(r64.abs().max()))
    print(f"[{name}] GAE vs float64: adv {ea:.2e}, ret {er:.2e} (relative to the largest)")    # measured <= 2.5e-7
    assert ea <= 1e-6 and er <= 1e-6

    # the next rollout starts where this one ended
    end = ppo.obs.clone()
    ppo.update()
    ppo.collect()
    assert torch.equal(ppo.obs_buf[0], end), "obs_buf[0] of the next rollout is not the observation the last one ended on"


# ---- update -----------------------------------------------------------------------------------------------------------------
def check_update(ppo, tol, name):
    p = ppo.p
    ppo.collect()
    case_conditions(ppo)
    T, n = ppo.rew_buf.shape
    total = T * n
    ref = Reference(ppo)
    rec = Recorder(ppo)
    state = rng_state(ppo).clone()
    out = ppo.update()
    idx = permutations(ppo, state, total)
    nb = p.n_epochs * math.ceil(total / p.batch_size)
    assert out["minibatches"] == nb == len(idx) == len(rec.steps)
    assert len(idx[-1]) == total % p.batch_size

    dev = ppo.device
    obs = ppo.obs_buf.reshape(total, -1)
    act = ppo.act_buf.reshape(total, -1)
    logp_old, adv, ret = ppo.logp_buf.reshape(total), ppo.adv.reshape(total), ppo.ret.reshape(total)
    adam = Adam64(rec.steps[0][0].numel(), p.learning_rate)
    margin = MARGIN[p.autocast_bf16]
    diags, stats = [], dict(grad=0.0, tensor=0.0, adam=0.0, boundary=0, clip_slack=0.0, logratio=0.0)
    clip_late = []
    for k, ((before, g_dev, after), rows) in enumerate(zip(rec.steps, idx)):
        rows = rows.to(dev)
        g_ref, scale, diag, n_near, widen, log_ratio = ref.minibatch(before, obs[rows], act[rows], logp_old[rows], adv[rows], ret[rows], margin)
        g_ref = g_ref.cpu()
        diags.append(diag.cpu())
        stats["boundary"] += n_near
        stats["clip_slack"] += n_near / len(rows) / nb          # the most the boundary rows can move the averaged clip fraction
        if k == 0:
            stats["logratio"] = float(log_ratio.abs().max())
        if k >= nb // 2:
            clip_late.append(float(diag[4]))
        # the post-clip gradient, whole and per tensor
        gn = float(g_ref.norm())
        err = float((g_dev - g_ref).norm())
        stats["grad"] = max(stats["grad"], err / gn)
        assert err <= tol["grad"] * gn + widen, f"minibatch {k} ({len(rows)} rows): gradient rel err {err / gn:.2e}, {n_near} boundary rows"
        for pname, gd, gr in zip(ref.names, ref.split(g_dev).values(), ref.split(g_ref).values()):
            e, r = float((gd - gr).norm()), float(gr.norm())
            if r > 1e-3 * gn:
                stats["tensor"] = max(stats["tensor"], e / r)
            assert e <= tol["tensor"] * max(r, 1e-3 * gn) + widen, f"minibatch {k}: gradient of {pname}, rel err {e / max(r, 1e-30):.2e}"
        # Adam applied to the device's own gradient
        want = adam.step(before, g_dev)
        slack = (after - want).abs() - FP32_ULP * after.abs()
        stats["adam"] = max(stats["adam"], float(slack.max()) / p.learning_rate)
        assert float(slack.max()) <= tol["adam"] * p.learning_rate, f"minibatch {k}: Adam step off by {float(slack.max()):.2e}"

    d_ref = torch.stack(diags).mean(0)
    d_dev = torch.tensor([out[k] for k in ("pg", "vf", "ent", "kl", "clip_frac")], dtype=torch.float64)
    d_err = (d_dev - d_ref).abs() / (1.0 + d_ref.abs())
    d_err[4] = max(0.0, float((d_dev[4] - d_ref[4]).abs()) - stats["clip_slack"])
    print(f"[{name}] {nb} minibatches: grad rel {stats['grad']:.2e}, per tensor {stats['tensor']:.2e}, Adam {stats['adam']:.2e} lr, "
          f"epoch-0 |log ratio| {stats['logratio']:.2e}, boundary rows {stats['boundary']}, diagnostics {d_err.max():.2e} "
          f"(clip_frac late {max(clip_late):.3f})")
    for i, key in enumerate(("pg", "vf", "ent", "kl", "clip_frac")):
        assert float(d_err[i]) <= tol["diag"], f"diagnostic {key}: device {float(d_dev[i]):.6g}, reference {float(d_ref[i]):.6g}"
    if tol["logratio"] is not None:
        assert stats["logratio"] <= tol["logratio"], f"epoch-0 |log ratio| {stats['logratio']:.2e}"
    if nb > 1:
        assert max(clip_late) > 0.0, "no later minibatch clipped: the learning rate no longer exercises the clip"
    return stats


# ---- the reference against torch / SB3 conventions (CPU) --------------------------------------------------------------------
def test_reference_pieces_match_torch():
    """The restated pieces against torch's own: Normal log-prob / entropy, clip_grad_norm_, and Adam (eps 1e-5) over 20 steps."""
    g = torch.Generator().manual_seed(0)
    mean, a = torch.randn(50, 4, generator=g, dtype=torch.float64), torch.randn(50, 4, generator=g, dtype=torch.float64) * 2
    log_std = torch.rand(4, generator=g, dtype=torch.float64) * 2 - 1.5
    d = torch.distributions.Normal(mean, log_std.exp().expand_as(mean))
    torch.testing.assert_close(gauss_logp(a, mean, log_std), d.log_prob(a).sum(-1), rtol=1e-14, atol=1e-14)
    torch.testing.assert_close(gauss_entropy(log_std).expand(50), d.entropy().sum(-1), rtol=1e-14, atol=1e-14)

    w = torch.nn.Parameter(torch.randn(300, generator=g, dtype=torch.float64))
    w.grad = torch.randn(300, generator=g, dtype=torch.float64)
    want = w.grad * clip_scale(float(w.grad.norm()), 0.5)
    torch.nn.utils.clip_grad_norm_([w], 0.5)
    torch.testing.assert_close(w.grad, want, rtol=1e-15, atol=0)

    opt = torch.optim.Adam([w], lr=3e-3, eps=ADAM_EPS)
    mine = Adam64(300, 3e-3)
    theta = w.detach().clone()
    for _ in range(20):
        w.grad = torch.randn(300, generator=g, dtype=torch.float64) * torch.logspace(-7, 0, 300, dtype=torch.float64)
        theta = mine.step(theta, w.grad)
        opt.step()
        torch.testing.assert_close(w.detach(), theta, rtol=1e-14, atol=1e-16)


@pytest.mark.parametrize("name", list(CPU_CASES))
def test_update_matches_sb3_reference_cpu(name):
    make, kw, tol = CPU_CASES[name]
    cfg = make()
    check_update(make_ppo(TensorOracleSim(cfg), cfg, kw), tol, name)


@pytest.mark.parametrize("name", list(CPU_CASES))
def test_rollout_matches_replay_cpu(name):
    make, kw, _ = CPU_CASES[name]
    cfg = make()
    ppo = make_ppo(TensorOracleSim(cfg), cfg, kw)
    replay = TensorOracleSim(cfg)                               # the same configuration, freshly reset: where ppo.sim stands
    check_rollout(ppo, replay, replay.reset(), name)


def test_cases_keep_their_edges():
    """One case ends each epoch on a minibatch of one row (the numel() > 1 guard); every case has a partial last minibatch."""
    totals = {}
    for table in (CPU_CASES, GPU_CASES):
        for name, (make, kw, _) in table.items():
            cfg = make()
            p = PPOConfig(**{**PPO_BASE, **kw})
            totals[name] = (p.n_steps * cfg.num_envs * cfg.num_agents, p.batch_size)
    assert all(t % b != 0 for t, b in totals.values())
    assert totals["cfg3_h32_last_row_alone"][0] % totals["cfg3_h32_last_row_alone"][1] == 1
    assert totals["cfg3_fused_obstacles"][0] % totals["cfg3_fused_obstacles"][1] == 1


# ---- GPU --------------------------------------------------------------------------------------------------------------------
def _gpu_case(name):
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import supported
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    torch.backends.cuda.matmul.allow_tf32 = False
    make, kw, tol = GPU_CASES[name]
    cfg = make()
    sim = QuadSwarmSim(cfg, device="cuda:0")
    ppo = make_ppo(sim, cfg, kw)
    assert (ppo.fused is not None) == ("fused" in name) == supported(ppo.policy)
    return cfg, sim, ppo, tol


@gpu
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_update_matches_sb3_reference_gpu(name):
    cfg, sim, ppo, tol = _gpu_case(name)
    check_update(ppo, tol, name)


@gpu
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_rollout_matches_replay_gpu(name):
    from quad_swarm_rl_stable_baselines3_b200.sim import QuadSwarmSim
    cfg, sim, ppo, _ = _gpu_case(name)
    snap = sim.snapshot()
    replay = QuadSwarmSim(cfg, device="cuda:0")
    obs0 = replay.restore(snap).clone()
    check_rollout(ppo, replay, obs0, name)
