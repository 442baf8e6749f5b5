"""Fused two-tower policy forward on the tcgen05 tensor cores (csrc/policy_kernels.cu, include/quadpolicy.h): the rollout-time
replacement of `QuadActorCritic.act`'s dense layers (reference: swarm_rl/models/ActorCriticPolicyCustom.py:430-480,
swarm_rl/models/quad_multi_model.py:333-354).  One kernel launch per batch of observations; activations never leave the SM.

The torch module (`ppo.QuadActorCritic`) stays the owner of the parameters and is what the PPO update differentiates; this class
re-packs its weights into the kernel's bf16 tile images (`sync()`, once per rollout) and evaluates mean / value for the rollout.
There is no fallback: on a box without the CUDA library the constructor raises."""
from __future__ import annotations

import ctypes as C

import torch

from . import _capi


QP_API_VERSION = 2


class QpConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("api_version", "self_dim", "nbr_dim", "num_nbr", "hidden", "act_dim", "obst_dim")]


class QpTowerWeightsC(C.Structure):
    FIELDS = ("self_w1", "self_b1", "self_w2", "self_b2", "nbr_w1", "nbr_b1", "nbr_w2", "nbr_b2", "ff_w", "ff_b", "head_w", "head_b",
              "obst_w1", "obst_b1", "obst_w2", "obst_b2")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


def supported(policy) -> bool:
    """The architecture the kernel is built for: deep-sets ('mean_embed') or no neighbour encoder, optionally the obstacle encoder
    (9 SDF inputs), hidden 256."""
    enc = policy.actor
    return (enc.kind in ("mean_embed", "none") and enc.O in (0, 9) and enc.self_encoder[0].out_features == 256
            and enc.S <= 24 and enc.W <= 8 and policy.action_net.out_features <= 8 and (enc.kind == "none" or enc.neighbor[0].out_features == 256)
            and (enc.O == 0 or enc.obstacle[0].out_features == 256))
    # 'attention' (the fork's default, quad_multi_model.py:42-102) and 'mlp' stay on the torch path


def gae(rewards: torch.Tensor, values: torch.Tensor, dones: torch.Tensor, last_values: torch.Tensor, gamma: float, lam: float):
    """`ppo.compute_gae` in one CUDA launch (`qp_gae`): rewards / values [T, n] float32, dones [T, n] bool or uint8, last_values [n];
    ValueError on any other dtype or shape."""
    if rewards.device.type != "cuda":
        raise RuntimeError("fused_policy.gae runs on CUDA tensors only (no CPU path)")
    if rewards.dim() != 2:
        raise ValueError("gae: rewards must be [T, n]")
    T, n = rewards.shape
    # the kernel reads the [T, n] arrays as float32 and one byte per done flag: another dtype would be reinterpreted, not converted
    for name, t, dtypes in (("rewards", rewards, (torch.float32,)), ("values", values, (torch.float32,)), ("dones", dones, (torch.bool, torch.uint8))):
        if t.dtype not in dtypes or tuple(t.shape) != (T, n) or t.device != rewards.device:
            raise ValueError(f"gae: {name} must be {' / '.join(str(d) for d in dtypes)} [{T}, {n}] on {rewards.device}, "
                             f"got {t.dtype} {list(t.shape)} on {t.device}")
    if tuple(last_values.shape) != (n,) or last_values.device != rewards.device:
        raise ValueError(f"gae: last_values must be [{n}] on {rewards.device}, got {list(last_values.shape)} on {last_values.device}")
    rewards, values, last_values = rewards.contiguous(), values.contiguous(), last_values.contiguous().float()
    d8 = dones.contiguous().view(torch.uint8)
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    lib = _capi.lib()
    with torch.cuda.device(rewards.device):
        rc = lib.qp_gae(rewards.data_ptr(), values.data_ptr(), d8.data_ptr(), last_values.data_ptr(), T, n, gamma, lam, adv.data_ptr(), ret.data_ptr(),
                        C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qp_gae failed ({rc}): {lib.qp_last_error(None).decode()}")
    return adv, ret


def _bt_check(t: torch.Tensor):
    if t.device.type != "cuda" or t.dtype not in (torch.float32, torch.bfloat16) or t.dim() != 2 or not t.is_contiguous():
        raise ValueError("bias_tanh works on contiguous 2-D float32 / bfloat16 CUDA tensors")


def bias_tanh(z: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """y = tanh(z + bias) in one launch (`qp_bias_tanh`); z [n, h] float32 / bfloat16, bias [h]."""
    _bt_check(z)
    b = bias.detach().to(device=z.device, dtype=torch.float32).contiguous()
    y = torch.empty_like(z)
    lib = _capi.lib()
    with torch.cuda.device(z.device):
        rc = lib.qp_bias_tanh(z.data_ptr(), b.data_ptr(), z.shape[0], z.shape[1], int(z.dtype == torch.bfloat16), y.data_ptr(),
                              C.c_void_p(torch.cuda.current_stream(z.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qp_bias_tanh failed ({rc}): {lib.qp_last_error(None).decode()}")
    return y


def bias_tanh_backward(grad_y: torch.Tensor, y: torch.Tensor):
    """(grad_z, grad_bias) of `bias_tanh` in one pass (`qp_bias_tanh_backward`); grad_bias is float32 [h]."""
    _bt_check(y)
    if grad_y.dtype != y.dtype or not grad_y.is_contiguous():
        grad_y = grad_y.to(y.dtype).contiguous()
    gz = torch.empty_like(y)
    gb = torch.empty(y.shape[1], dtype=torch.float32, device=y.device)
    lib = _capi.lib()
    with torch.cuda.device(y.device):
        rc = lib.qp_bias_tanh_backward(grad_y.data_ptr(), y.data_ptr(), y.shape[0], y.shape[1], int(y.dtype == torch.bfloat16), gz.data_ptr(),
                                       gb.data_ptr(), C.c_void_p(torch.cuda.current_stream(y.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qp_bias_tanh_backward failed ({rc}): {lib.qp_last_error(None).decode()}")
    return gz, gb


_first_ws = {}


def bias_tanh_backward_first(grad_y: torch.Tensor, y: torch.Tensor, x: torch.Tensor):
    """(grad_weight [h, in], grad_bias [h]) of a first tanh layer with in <= 8 inputs (`qp_bias_tanh_backward_first`); x float32 [n, in]."""
    _bt_check(y)
    if grad_y.dtype != y.dtype or not grad_y.is_contiguous():
        grad_y = grad_y.to(y.dtype).contiguous()
    x = x.detach().to(torch.float32).contiguous()
    lib = _capi.lib()
    key = (y.device, y.shape[1], x.shape[1])
    if key not in _first_ws:
        _first_ws[key] = torch.empty(int(lib.qp_bias_tanh_backward_first_workspace(y.shape[1], x.shape[1])) // 4, dtype=torch.float32, device=y.device)
    gb = torch.empty(y.shape[1], dtype=torch.float32, device=y.device)
    gw = torch.empty((y.shape[1], x.shape[1]), dtype=torch.float32, device=y.device)
    with torch.cuda.device(y.device):
        rc = lib.qp_bias_tanh_backward_first(grad_y.data_ptr(), y.data_ptr(), x.data_ptr(), y.shape[0], y.shape[1], x.shape[1],
                                             int(y.dtype == torch.bfloat16), _first_ws[key].data_ptr(), gb.data_ptr(), gw.data_ptr(),
                                             C.c_void_p(torch.cuda.current_stream(y.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qp_bias_tanh_backward_first failed ({rc}): {lib.qp_last_error(None).decode()}")
    return gw, gb


def _groups(rows: int, V: int) -> int:
    """Groups of V consecutive rows; a remainder would be left unwritten in the outputs."""
    if V < 1 or rows % V != 0:
        raise ValueError(f"bias_tanh_mean: {rows} rows are not whole groups of V = {V}")
    return rows // V


def bias_tanh_mean(z: torch.Tensor, bias: torch.Tensor, V: int):
    """(y, mean): y = tanh(z + bias) on [n * V, h], mean [n, h] over each group of V rows (`qp_bias_tanh_mean`)."""
    _bt_check(z)
    n = _groups(z.shape[0], V)
    b = bias.detach().to(device=z.device, dtype=torch.float32).contiguous()
    y, m = torch.empty_like(z), torch.empty((n, z.shape[1]), dtype=z.dtype, device=z.device)
    lib = _capi.lib()
    with torch.cuda.device(z.device):
        rc = lib.qp_bias_tanh_mean(z.data_ptr(), b.data_ptr(), n, V, z.shape[1], int(z.dtype == torch.bfloat16), y.data_ptr(), m.data_ptr(),
                                   C.c_void_p(torch.cuda.current_stream(z.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qp_bias_tanh_mean failed ({rc}): {lib.qp_last_error(None).decode()}")
    return y, m


def bias_tanh_mean_backward(grad_mean: torch.Tensor, y: torch.Tensor, V: int):
    _bt_check(y)
    n = _groups(y.shape[0], V)
    if tuple(grad_mean.shape) != (n, y.shape[1]):
        raise ValueError(f"bias_tanh_mean_backward: grad_mean must be [{n}, {y.shape[1]}], got {list(grad_mean.shape)}")
    if grad_mean.dtype != y.dtype or not grad_mean.is_contiguous():
        grad_mean = grad_mean.to(y.dtype).contiguous()
    gz = torch.empty_like(y)
    gb = torch.empty(y.shape[1], dtype=torch.float32, device=y.device)
    lib = _capi.lib()
    with torch.cuda.device(y.device):
        rc = lib.qp_bias_tanh_mean_backward(grad_mean.data_ptr(), y.data_ptr(), n, V, y.shape[1], int(y.dtype == torch.bfloat16),
                                            gz.data_ptr(), gb.data_ptr(), C.c_void_p(torch.cuda.current_stream(y.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qp_bias_tanh_mean_backward failed ({rc}): {lib.qp_last_error(None).decode()}")
    return gz, gb


class FusedPolicy:
    def __init__(self, policy, device):
        if not supported(policy):
            raise ValueError("the fused policy kernel is built for hidden 256, deep-sets / no neighbour encoder, optional obstacle encoder, S <= 24, W <= 8")
        self.policy = policy
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("FusedPolicy runs on CUDA devices only (no CPU path)")
        enc = policy.actor
        self.S, self.W, self.V, self.O = enc.S, enc.W, (enc.V if enc.kind == "mean_embed" else 0), enc.O
        self.A = policy.action_net.out_features
        self._lib = _capi.lib()
        cfg = QpConfigC(QP_API_VERSION, self.S, self.W, self.V, 256, self.A, self.O)
        if self._lib.qp_config_size() != C.sizeof(QpConfigC):
            raise RuntimeError("qp_config layout mismatch")
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            rc = self._lib.qp_create(C.byref(cfg), self.device.index or 0, C.byref(h))
        if rc != 0:
            raise RuntimeError(f"qp_create failed ({rc}): {self._lib.qp_last_error(None).decode()}")
        self._h = h
        self._keep = []
        self.sync()

    def close(self):
        if getattr(self, "_h", None):
            self._lib.qp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self._lib.qp_launch_count(self._h))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @torch.no_grad()
    def sync(self):
        """Re-pack the torch module's current weights (call after every optimiser phase)."""
        pol = self.policy
        self._keep = []
        for tower, (enc, head) in enumerate(((pol.actor, pol.action_net), (pol.critic, pol.value_net))):
            t = {"self_w1": enc.self_encoder[0].weight, "self_b1": enc.self_encoder[0].bias,
                 "self_w2": enc.self_encoder[2].weight, "self_b2": enc.self_encoder[2].bias,
                 "ff_w": enc.feed_forward[0].weight, "ff_b": enc.feed_forward[0].bias, "head_w": head.weight, "head_b": head.bias}
            if self.V > 0:
                t.update({"nbr_w1": enc.neighbor[0].weight, "nbr_b1": enc.neighbor[0].bias,
                          "nbr_w2": enc.neighbor[2].weight, "nbr_b2": enc.neighbor[2].bias})
            if self.O > 0:
                t.update({"obst_w1": enc.obstacle[0].weight, "obst_b1": enc.obstacle[0].bias,
                          "obst_w2": enc.obstacle[2].weight, "obst_b2": enc.obstacle[2].bias})
            w = QpTowerWeightsC()
            for name in QpTowerWeightsC.FIELDS:
                v = t.get(name)
                if v is None:
                    setattr(w, name, None)
                    continue
                v = v.detach().to(device=self.device, dtype=torch.float32).contiguous()
                if name == "ff_w" and self.V == 0:       # no neighbour encoder: its block of the feed-forward input, [self | neighbour | obstacle], is zeros
                    v = torch.cat([v[:, :256], torch.zeros_like(v[:, :256]), v[:, 256:]], dim=1).contiguous()
                self._keep.append(v)
                setattr(w, name, v.data_ptr())
            with torch.cuda.device(self.device):
                rc = self._lib.qp_set_weights(self._h, tower, C.byref(w), self._stream())
            if rc != 0:
                raise RuntimeError(f"qp_set_weights failed ({rc}): {self._lib.qp_last_error(self._h).decode()}")

    @torch.no_grad()
    def forward(self, obs: torch.Tensor):
        """obs [n, D] float32 CUDA -> (action mean [n, A], value [n])."""
        if obs.device != self.device or obs.dtype != torch.float32 or obs.dim() != 2:
            raise ValueError("obs must be a 2-D float32 tensor on the policy's device")
        if not obs.is_contiguous():
            obs = obs.contiguous()
        n = obs.shape[0]
        mean = torch.empty((n, self.A), dtype=torch.float32, device=self.device)
        value = torch.empty((n,), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            rc = self._lib.qp_forward(self._h, obs.data_ptr(), n, obs.shape[1], mean.data_ptr(), value.data_ptr(), self._stream())
        if rc != 0:
            raise RuntimeError(f"qp_forward failed ({rc}): {self._lib.qp_last_error(self._h).decode()}")
        return mean, value

    @torch.no_grad()
    def act(self, obs: torch.Tensor):
        """`QuadActorCritic.act` with the dense layers on the fused kernel: (action, log-prob, value)."""
        mean, value = self.forward(obs)
        log_std = self.policy.log_std.detach().to(mean.dtype)
        eps = torch.randn_like(mean)
        action = mean + eps * log_std.exp()
        logp = (-0.5 * eps * eps - log_std - 0.9189385332046727).sum(-1)
        return action, logp, value
