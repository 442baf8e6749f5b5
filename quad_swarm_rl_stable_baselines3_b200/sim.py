"""Device-resident batched simulator: the thin torch layer over the C-ABI.

`QuadSwarmSim` owns one `qs_env` handle (N environments x K drones on one GPU).  Observations, rewards and dones
are returned as CUDA tensors that alias buffers owned by this object (valid until the next step/reset); nothing in
`step` touches the host.  PyTorch is plumbing here (memory, streams); all simulation arithmetic is in
csrc/quadsim_kernels.cuh.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _capi
from .config import PARAM_KEYS, QS_ER_COUNT, QS_SC_COUNT, QsConfigC, QsStateViewC, QsStatsC, QuadSimConfig

_STATE_SHAPES = {"pos": (3, torch.float32), "vel": (3, torch.float32), "rot": (9, torch.float32),
                 "omega": (3, torch.float32), "rot_damp": (4, torch.float32), "cmds_damp": (4, torch.float32),
                 "ou": (4, torch.float32), "goal": (3, torch.float32), "flags": (1, torch.int32),
                 "col_mask": (1, torch.int32)}
_FORK_SHAPES = {"pid": (24, torch.float32), "heading": (3, torch.float32)}     # fork mode only: (angle, ang_vel, heading snapshot)
_ENV_FIELDS = {"tick": torch.int32, "svd_ctr": torch.int32, "step_ctr": torch.int32}


# the qs_config fields the rows and width of a handle's observation follow from (fill_const, csrc/quadsim.cu)
_OBS_LAYOUT_FIELDS = ("num_agents", "env_mode", "obs_repr", "neighbor_obs_type", "neighbor_visible_num", "use_obstacles")


def _blob_config(blob: torch.Tensor) -> QsConfigC:
    """The qs_config of a snapshot blob: it sits at offset 16 (include/quadsim.h)."""
    return QsConfigC.from_buffer_copy(blob[16:16 + C.sizeof(QsConfigC)].numpy().tobytes())


class QuadSwarmSim:
    def __init__(self, cfg: QuadSimConfig, device: Optional[torch.device | int | str] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("QuadSwarmSim needs a CUDA device: the simulator has no CPU path")
        self.cfg = cfg
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("QuadSwarmSim runs on CUDA devices only")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self._lib = _capi.lib()
        self._c = cfg.to_c()
        h = C.c_void_p()
        with torch.cuda.device(dev):
            rc = self._lib.qs_create(C.byref(self._c), dev.index, C.byref(h))
        _capi.check(None, rc, "qs_create")
        self._h = h
        self.N, self.K = cfg.num_envs, cfg.num_agents
        self.D, self.A = self._lib.qs_obs_dim(h), self._lib.qs_act_dim(h)
        assert self.D == cfg.obs_dim, (self.D, cfg.obs_dim)
        n = self.N * self.K
        self.obs = torch.zeros((n, self.D), dtype=torch.float32, device=dev)
        self.rew = torch.zeros((n,), dtype=torch.float32, device=dev)
        self._done_u8 = torch.zeros((n,), dtype=torch.uint8, device=dev)
        self.terminal_obs = torch.zeros((n, self.D), dtype=torch.float32, device=dev)
        self.reset_success = torch.zeros((self.N,), dtype=torch.uint8, device=dev)   # reset_info["success"] of envs that just finished
        self.want_terminal_obs = True
        self.rew_info = None                      # per-step reward terms (enable_reward_info)
        self.rew_coeff_overrides: Dict[str, float] = {}
        self.is_fork = cfg.env_mode == "fork"
        # formation scenarios keep a per-env scenario row on the device (static_same_goal needs none)
        self.has_scenario_state = (not self.is_fork) and (not cfg.use_obstacles) and cfg.quads_mode != "static_same_goal"

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.qs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def done(self) -> torch.Tensor:
        return self._done_u8.view(torch.bool)

    @property
    def launch_count(self) -> int:
        return int(self._lib.qs_launch_count(self._h))

    # ------------------------------------------------------------------------------------------
    def reset(self, env_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Reset every env (or those with env_mask[e] true).  Returns obs [N*K, D] (aliases self.obs)."""
        mp = None
        if env_mask is not None:
            env_mask = env_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if env_mask.numel() != self.N:
                raise ValueError("env_mask must have one entry per env")
            mp = C.c_void_p(env_mask.data_ptr())
        with torch.cuda.device(self.device):
            rc = self._lib.qs_reset(self._h, mp, C.c_void_p(self.obs.data_ptr()), self._stream())
        _capi.check(self._h, rc, "qs_reset")
        return self.obs

    def step(self, actions: torch.Tensor):
        """One step for all envs (upstream mode: one control step; fork mode: `fork.substeps` control steps, like the
        reference's step()).  actions: CUDA float32 [N*K, A].  Returns (obs, rew, done) CUDA tensors; `self.terminal_obs`
        and `self.reset_success` hold the finished envs' last observation / reset_info["success"]."""
        if actions.device != self.device or actions.dtype != torch.float32:
            raise ValueError("actions must be a float32 tensor on the simulator's device (use step_host for numpy)")
        if actions.numel() != self.N * self.K * self.A:
            raise ValueError(f"actions must have shape [{self.N * self.K}, {self.A}]")
        if not actions.is_contiguous():
            actions = actions.contiguous()
        tp = C.c_void_p(self.terminal_obs.data_ptr()) if self.want_terminal_obs else None
        with torch.cuda.device(self.device):
            rc = self._lib.qs_step(self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(self.obs.data_ptr()),
                                   C.c_void_p(self.rew.data_ptr()), C.c_void_p(self._done_u8.data_ptr()), tp,
                                   C.c_void_p(self.reset_success.data_ptr()), self._stream())
        _capi.check(self._h, rc, "qs_step")
        return self.obs, self.rew, self.done

    # host-buffer path (what an SB3 numpy rollout loop calls) ------------------------------------
    def reset_host(self) -> np.ndarray:
        out = np.empty((self.N * self.K, self.D), dtype=np.float32)
        with torch.cuda.device(self.device):
            rc = self._lib.qs_reset_host(self._h, out.ctypes.data_as(C.c_void_p), self._stream())
        _capi.check(self._h, rc, "qs_reset_host")
        return out

    def step_host(self, actions: np.ndarray, out=None, terminal_obs: Optional[np.ndarray] = None,
                  reset_success: Optional[np.ndarray] = None):
        """Host-buffer step.  `out` = (obs, rew, done_u8) numpy arrays to fill (pinned ones are DMA'd directly);
        `terminal_obs` [N*K, D] float32 / `reset_success` [N] uint8 are filled for envs that finished."""
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.N * self.K, self.A)
        if out is None:
            out = (np.empty((self.N * self.K, self.D), dtype=np.float32), np.empty(self.N * self.K, dtype=np.float32),
                   np.empty(self.N * self.K, dtype=np.uint8))
        obs, rew, done = out
        tp = None if terminal_obs is None else terminal_obs.ctypes.data_as(C.c_void_p)
        sp = None if reset_success is None else reset_success.ctypes.data_as(C.c_void_p)
        with torch.cuda.device(self.device):
            rc = self._lib.qs_step_host(self._h, a.ctypes.data_as(C.c_void_p), obs.ctypes.data_as(C.c_void_p),
                                        rew.ctypes.data_as(C.c_void_p), done.ctypes.data_as(C.c_void_p), tp, sp,
                                        self._stream())
        _capi.check(self._h, rc, "qs_step_host")
        return obs, rew, done.view(np.bool_)

    # state access ----------------------------------------------------------------------------------
    def _view(self, tensors: Dict[str, torch.Tensor]) -> QsStateViewC:
        v = QsStateViewC()
        for name in QsStateViewC.FIELDS:
            t = tensors.get(name)
            setattr(v, name, None if t is None else t.data_ptr())
        return v

    def get_state(self, fields=None) -> Dict[str, torch.Tensor]:
        n = self.N * self.K
        names = list(fields) if fields is not None else (list(_STATE_SHAPES) + list(_ENV_FIELDS) + ["obst_xy"] +
                                                         (list(_FORK_SHAPES) + ["evader"] if self.is_fork else []) +
                                                         (["scenario"] if self.has_scenario_state else []))
        shapes = dict(_STATE_SHAPES, **_FORK_SHAPES)
        out = {}
        for name in names:
            if name in shapes:
                w, dt = shapes[name]
                out[name] = torch.zeros((n, w) if w > 1 else (n,), dtype=dt, device=self.device)
            elif name in _ENV_FIELDS:
                out[name] = torch.zeros((self.N,), dtype=_ENV_FIELDS[name], device=self.device)
            elif name == "obst_xy":
                out[name] = torch.zeros((self.N, 64, 2), dtype=torch.float32, device=self.device)
            elif name == "evader":
                out[name] = torch.zeros((self.N, 2), dtype=torch.float32, device=self.device)
            elif name == "scenario":        # QS_SC_* rows (include/quadsim.h): the reference scenario object's state
                out[name] = torch.zeros((self.N, QS_SC_COUNT), dtype=torch.float32, device=self.device)
            else:
                raise KeyError(name)
        v = self._view(out)
        with torch.cuda.device(self.device):
            rc = self._lib.qs_get_state(self._h, C.byref(v), self._stream())
        _capi.check(self._h, rc, "qs_get_state")
        torch.cuda.current_stream(self.device).synchronize()
        return out

    def get_state_host(self, fields=None) -> Dict[str, np.ndarray]:
        """`get_state` as numpy arrays (the `envs[i].dynamics.*` views of the QuadrotorEnvMulti facade read through this)."""
        return {k: v.cpu().numpy() for k, v in self.get_state(fields).items()}

    # per-step reward breakdown: infos[i]["rewards"] / infos[i]["goal_dist"] -------------------------------------------------
    def enable_reward_info(self, on: bool = True) -> Optional[torch.Tensor]:
        """Switch the per-step reward-term output on (QS_RI_* columns, include/quadsim.h).  Returns the CUDA tensor
        [N*K, 8] the next steps fill (owned by this object), or None when switched off."""
        if on:
            if getattr(self, "rew_info", None) is None:
                self.rew_info = torch.zeros((self.N * self.K, 8), dtype=torch.float32, device=self.device)
            ptr = C.c_void_p(self.rew_info.data_ptr())
        else:
            self.rew_info, ptr = None, None
        _capi.check(self._h, self._lib.qs_set_reward_info(self._h, ptr), "qs_set_reward_info")
        return self.rew_info

    def reward_info_host(self) -> np.ndarray:
        if getattr(self, "rew_info", None) is None:
            raise RuntimeError("reward info is off: call enable_reward_info() first")
        return self.rew_info.cpu().numpy()

    def set_state(self, **fields):
        n = self.N * self.K
        keep = {}
        shapes = dict(_STATE_SHAPES, **_FORK_SHAPES)
        for name, val in fields.items():
            if val is None:
                continue
            if name in shapes:
                w, dt = shapes[name]
                t = torch.as_tensor(np.asarray(val) if not torch.is_tensor(val) else val)
                if name == "col_mask":
                    t = t.to(torch.int64).to(torch.int32) if t.dtype != torch.int32 else t
                keep[name] = t.to(device=self.device, dtype=dt).reshape((n, w) if w > 1 else (n,)).contiguous()
            elif name in _ENV_FIELDS:
                t = torch.as_tensor(np.asarray(val) if not torch.is_tensor(val) else val)
                keep[name] = t.to(device=self.device, dtype=torch.int32).reshape(self.N).contiguous()
            elif name == "obst_xy":
                t = torch.as_tensor(np.asarray(val) if not torch.is_tensor(val) else val).to(self.device, torch.float32)
                full = torch.zeros((self.N, 64, 2), dtype=torch.float32, device=self.device)
                t = t.reshape(self.N, -1, 2)
                full[:, :t.shape[1]] = t
                keep[name] = full
            elif name == "evader":
                t = torch.as_tensor(np.asarray(val) if not torch.is_tensor(val) else val)
                keep[name] = t.to(device=self.device, dtype=torch.float32).reshape(self.N, 2).contiguous()
            elif name == "scenario":
                t = torch.as_tensor(np.asarray(val) if not torch.is_tensor(val) else val)
                keep[name] = t.to(device=self.device, dtype=torch.float32).reshape(self.N, QS_SC_COUNT).contiguous()
            else:
                raise KeyError(name)
        v = self._view(keep)
        with torch.cuda.device(self.device):
            rc = self._lib.qs_set_state(self._h, C.byref(v), self._stream())
        _capi.check(self._h, rc, "qs_set_state")
        torch.cuda.current_stream(self.device).synchronize()

    def episode_records(self) -> Dict[str, torch.Tensor]:
        """Record of the last finished episode per env (QS_ER_* rows, include/quadsim.h) as CUDA tensors:
        {"env": int32 [N, QS_ER_COUNT], "agent": float32 [N*K, 4]}.  No host synchronisation."""
        env = torch.empty((self.N, QS_ER_COUNT), dtype=torch.int32, device=self.device)
        agent = torch.empty((self.N * self.K, 4), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            rc = self._lib.qs_episode_records(self._h, env.data_ptr(), agent.data_ptr(), self._stream())
        _capi.check(self._h, rc, "qs_episode_records")
        return {"env": env, "agent": agent}

    def episode_records_host(self, env_out: Optional[np.ndarray] = None, agent_out: Optional[np.ndarray] = None):
        """Same, into host arrays (allocated if not given); returns (env_rec [N, QS_ER_COUNT] int32, agent_rec [N*K, 4] float32)."""
        env = np.empty((self.N, QS_ER_COUNT), dtype=np.int32) if env_out is None else env_out
        agent = np.empty((self.N * self.K, 4), dtype=np.float32) if agent_out is None else agent_out
        with torch.cuda.device(self.device):
            rc = self._lib.qs_episode_records_host(self._h, env.ctypes.data, agent.ctypes.data, self._stream())
        _capi.check(self._h, rc, "qs_episode_records_host")
        return env, agent

    # snapshots: exact save / resume ------------------------------------------------------------------
    def snapshot(self) -> Dict[str, torch.Tensor]:
        """The whole simulator state (`qs_snapshot`, include/quadsim.h) plus the last observation, on the host:
        {"blob": uint8 pinned CPU tensor, "obs": float32 CPU tensor [N*K, D]}.  `restore` on any handle created with the same
        configuration continues bitwise where this one stands."""
        n = int(self._lib.qs_snapshot_size(self._h))
        blob = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        with torch.cuda.device(self.device):
            rc = self._lib.qs_snapshot(self._h, C.c_void_p(blob.data_ptr()), n, self._stream())
        _capi.check(self._h, rc, "qs_snapshot")
        return {"blob": blob, "obs": self.obs.cpu()}

    def restore(self, snap: Dict[str, torch.Tensor]) -> torch.Tensor:
        """Load a `snapshot()` into this handle (`qs_restore` rejects one of another configuration and leaves the handle as it was).
        The snapshot's reward coefficients / capture radius replace this handle's.  Returns the restored observation (self.obs)."""
        blob = torch.as_tensor(snap["blob"]).detach().to("cpu", torch.uint8).contiguous().reshape(-1)
        obs = torch.as_tensor(snap["obs"])
        if obs.numel() != self.obs.numel():
            raise ValueError(f"snapshot obs has {obs.numel()} values, this simulator's observation {self.obs.numel()}")
        with torch.cuda.device(self.device):
            rc = self._lib.qs_restore(self._h, C.c_void_p(blob.data_ptr()), blob.numel(), self._stream())
        _capi.check(self._h, rc, "qs_restore")
        self.obs.copy_(obs.reshape(self.obs.shape))
        self._take_rew_coeffs(_blob_config(blob))
        return self.obs

    def restore_shards(self, snaps) -> torch.Tensor:
        """Load this handle's envs from the `snapshot()`s of the shards of a run saved on any number of GPUs (`qs_restore_shards`,
        include/quadsim.h): every blob whose env range meets this handle's contributes its slice, the others are ignored, so every
        new rank may pass the full list.  The ranges must not overlap and must cover this handle's; everything else must match as for
        `restore`.  On a rejection nothing changes.  Returns the restored observation (self.obs)."""
        snaps = list(snaps)
        blobs = [torch.as_tensor(s["blob"]).detach().to("cpu", torch.uint8).contiguous().reshape(-1) for s in snaps]
        obs = [torch.as_tensor(s["obs"]) for s in snaps]
        lo, K = self.cfg.env_id_offset, self.K
        ranges = []
        # Each snapshot's observation must fit its blob's env range, checked before the call so that a misfit changes nothing.  The
        # check needs the blob's observation width, which is this handle's when the qs_config fields it follows from are; a blob that
        # differs there, or has no readable header, is left to qs_restore_shards, which rejects it and names the field.  Every blob
        # the call accepts has therefore been checked.
        for i, (b, o) in enumerate(zip(blobs, obs)):
            if b.numel() < 16 + C.sizeof(QsConfigC) or bytes(b[:4].numpy()) != b"QSSN":
                ranges.append(None)
                continue
            c = _blob_config(b)
            ranges.append((c.env_id_offset, c.env_id_offset + c.num_envs))
            if any(getattr(c, f) != getattr(self._c, f) for f in _OBS_LAYOUT_FIELDS):
                continue
            if o.numel() != c.num_envs * K * self.D:
                raise ValueError(f"restore_shards: snapshot {i} has {o.numel()} observation values, its {c.num_envs} envs "
                                 f"x {K} x {self.D} need {c.num_envs * K * self.D}")
        n = len(blobs)
        ptrs = (C.c_void_p * n)(*[b.data_ptr() for b in blobs])
        sizes = (C.c_size_t * n)(*[b.numel() for b in blobs])
        with torch.cuda.device(self.device):
            rc = self._lib.qs_restore_shards(self._h, ptrs, sizes, n, self._stream())
        _capi.check(self._h, rc, "qs_restore_shards")
        hi = lo + self.N
        for (b0, b1), o in zip(ranges, obs):
            a, b = max(lo, b0), min(hi, b1)
            if a < b:
                self.obs[(a - lo) * K:(b - lo) * K].copy_(o.reshape(-1, self.D)[(a - b0) * K:(b - b0) * K])
        self._take_rew_coeffs(_blob_config(blobs[0]))
        return self.obs

    def _take_rew_coeffs(self, c: QsConfigC):
        """The reward coefficients a restored snapshot brought in, as far as they differ from this handle's configuration."""
        self.rew_coeff_overrides = {k: getattr(c, "rew_" + k) for k in PARAM_KEYS if k != "capture_radius"
                                    and getattr(c, "rew_" + k) != getattr(self._c, "rew_" + k)}

    # parameters / stats ------------------------------------------------------------------------------
    def set_rew_coeff(self, **coeffs):
        """rew_coeff updates (reference: reward-shaping wrapper writing env.rew_coeff, reward_shaping.py:52-60)."""
        for k, v in coeffs.items():
            if k not in PARAM_KEYS:
                raise KeyError(k)
            _capi.check(self._h, self._lib.qs_set_param(self._h, PARAM_KEYS[k], float(v)), "qs_set_param")
            self.rew_coeff_overrides[k] = float(v)

    def set_capture_radius(self, value: float):
        """QuadrotorEnvMulti.set_capture_radius (quadrotor_multi_rewards.py:210-211), all envs of this handle."""
        _capi.check(self._h, self._lib.qs_set_param(self._h, PARAM_KEYS["capture_radius"], float(value)), "qs_set_param")

    def episode_stats(self, reset: bool = False, reduce: bool = False) -> Dict[str, float]:
        """Sums of the per-episode `episode_extra_stats` over the episodes finished since the last reset=True call.
        reduce=True additionally sums over all ranks (one small NCCL all-reduce; the only collective of the simulator)."""
        s = QsStatsC()
        with torch.cuda.device(self.device):
            rc = self._lib.qs_episode_stats(self._h, C.byref(s), int(reset), self._stream())
        _capi.check(self._h, rc, "qs_episode_stats")
        out = s.as_dict()
        if reduce:
            from .sharding import all_reduce_stats
            out = all_reduce_stats(out, device=self.device)
        return out
