"""CPU-side checks of the resharded resume (include/quadsim.h: qs_restore_shards): the NULL-handle contract, the ctypes signature
against the header's prototype, the export list, and the state-dict comparison DevicePPO.load_shards uses to refuse rank files whose
replicated policy or optimizer state differ."""
import ctypes as C
import os
import re

import pytest
import torch

from quad_swarm_rl_stable_baselines3_b200 import _capi
from quad_swarm_rl_stable_baselines3_b200.ppo import _first_difference

QS_ERR_NULL = -4
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "quadsim.h")


@pytest.fixture(scope="module")
def lib():
    _capi.build()
    return _capi.lib()


def test_restore_shards_rejects_null_handle(lib):
    buf = (C.c_uint8 * 64)()
    blobs = (C.c_void_p * 1)(C.cast(buf, C.c_void_p).value)
    sizes = (C.c_size_t * 1)(64)
    assert lib.qs_restore_shards(None, blobs, sizes, 1, None) == QS_ERR_NULL
    assert lib.qs_restore_shards(None, None, None, 0, None) == QS_ERR_NULL
    assert lib.qs_restore_shards(None, None, None, 3, None) == QS_ERR_NULL


def test_restore_shards_signature_follows_the_header(lib):
    with open(HEADER) as f:
        text = f.read()
    m = re.search(r"int\s+qs_restore_shards\s*\(([^)]*)\)\s*;", text)
    assert m, "qs_restore_shards is not declared in include/quadsim.h"
    params = [re.sub(r"\s+", " ", p.strip()) for p in m.group(1).split(",")]
    assert params == ["qs_env *env", "const void *const *blobs", "const size_t *bytes", "int count", "void *stream"], params
    vp = C.c_void_p
    at = lib.qs_restore_shards.argtypes
    assert at[0] is vp and at[4] is vp and at[3] is C.c_int
    assert at[1] == C.POINTER(vp) and at[2] == C.POINTER(C.c_size_t)     # arrays of 64-bit pointers and sizes
    assert lib.qs_restore_shards.restype is C.c_int
    assert "qs_restore_shards" in _capi.EXPORTS


def test_every_export_is_declared_in_the_header():
    with open(HEADER) as f:
        text = f.read()
    for name in _capi.EXPORTS:
        assert re.search(r"\b" + name + r"\s*\(", text), name


def test_first_difference_names_the_tensor():
    a = {"policy": {"w": torch.ones(3), "b": torch.zeros(2)},
         "opt": {"state": {0: {"step": torch.tensor(4.0), "exp_avg": torch.ones(3)}}, "param_groups": [{"lr": 1e-4, "params": [0]}]}}
    b = {"policy": {"w": torch.ones(3), "b": torch.zeros(2)},
         "opt": {"state": {0: {"step": torch.tensor(4.0), "exp_avg": torch.ones(3)}}, "param_groups": [{"lr": 1e-4, "params": [0]}]}}
    assert _first_difference(a, b, "ckpt") is None
    b["opt"]["state"][0]["exp_avg"][1] = torch.nextafter(torch.tensor(1.0), torch.tensor(2.0))   # one ulp
    assert _first_difference(a, b, "ckpt") == "ckpt.opt.state.0.exp_avg"
    b["policy"]["b"] = -b["policy"]["b"]                                 # -0.0: equal as numbers, not as bits
    assert _first_difference(a, b, "ckpt") == "ckpt.policy.b"
    c = {"policy": {"w": torch.ones(3, dtype=torch.float64), "b": torch.zeros(2)}, "opt": a["opt"]}
    assert _first_difference(a, c, "ckpt") == "ckpt.policy.w"
    d = dict(a, opt={"state": a["opt"]["state"], "param_groups": [{"lr": 2e-4, "params": [0]}]})
    assert _first_difference(a, d, "ckpt") == "ckpt.opt.param_groups.0.lr"
    nan = {"x": torch.tensor([float("nan")])}
    assert _first_difference(nan, {"x": nan["x"].clone()}, "s") is None   # the same bits, NaN included


# ---------------------------------------------------------------------------------------------------------------------------------
# DevicePPO.load_shards on the CPU: the training-side state a resharded resume takes from memory-mapped rank files
# ---------------------------------------------------------------------------------------------------------------------------------
class StubSim:
    """CPU stand-in with the part of QuadSwarmSim's interface DevicePPO uses; `restore_shards` records what it was given."""

    def __init__(self, cfg):
        self.cfg, self.device = cfg, torch.device("cpu")
        self.obs = torch.randn(cfg.num_envs * cfg.num_agents, cfg.obs_dim, generator=torch.Generator().manual_seed(cfg.env_id_offset))
        self.restored = None

    def reset(self):
        return self.obs

    def step(self, a):
        n = self.obs.shape[0]
        return self.obs, torch.ones(n), torch.zeros(n, dtype=torch.bool)

    def episode_stats(self, reset=False, reduce=False):
        return {"episodes": 0}

    def snapshot(self):
        return {"blob": torch.arange(64, dtype=torch.uint8), "obs": self.obs.clone()}

    def restore_shards(self, snaps):
        self.restored = [s["blob"].clone() for s in snaps]
        return self.obs


def _ppo(num_envs=4, env_id_offset=0):
    from quad_swarm_rl_stable_baselines3_b200.config import QuadSimConfig
    from quad_swarm_rl_stable_baselines3_b200.ppo import DevicePPO, PPOConfig
    cfg = QuadSimConfig(num_envs=num_envs, num_agents=8, env_id_offset=env_id_offset, seed=3)
    return DevicePPO(StubSim(cfg), cfg, PPOConfig(n_steps=4, batch_size=64, n_epochs=1, hidden=32, neighbor_hidden=16))


def test_load_shards_state_survives_overwriting_the_file_it_came_from(tmp_path):
    """The optimizer state load_shards installs owns its memory: saving over the memory-mapped rank file it was read from (what
    rank 0 does when it checkpoints under the old name) must neither fault nor lose the state."""
    a = _ppo(num_envs=4)
    a.learn(1)
    path = tmp_path / "ckpt_rank0.pt"
    a.save(path)
    saved = torch.load(path, weights_only=True)
    halves = [_ppo(num_envs=2, env_id_offset=r * 2) for r in range(2)]
    for h in halves:
        h.load_shards([path])
    halves[0].save(path)                                  # truncates and rewrites the file halves[1]'s state was read from
    again = torch.load(path, weights_only=True)
    for h in halves:
        assert _first_difference(saved["optimizer"], h.opt.state_dict(), "optimizer") is None
        assert _first_difference(saved["policy"], h.policy.state_dict(), "policy") is None
    assert _first_difference(saved["optimizer"], again["optimizer"], "optimizer") is None
    # this rank's rows of the saved observation
    assert torch.equal(halves[1].obs, saved["obs"][16:32]) and halves[1].total_agent_steps == saved["total_agent_steps"]
    halves[1].learn(1)                                    # and the restored optimizer steps


def test_load_shards_checks_the_saved_observation_before_restoring(tmp_path):
    a = _ppo(num_envs=4)
    a.learn(1)
    path = tmp_path / "ckpt.pt"
    a.save(path)
    ck = torch.load(path, weights_only=True)
    ck["obs"] = ck["obs"][:-8]                            # one env short of the file's sim_config.num_envs
    torch.save(ck, path)
    b = _ppo(num_envs=4)
    with pytest.raises(ValueError, match=r"observations \(24, 54\)"):
        b.load_shards([path])
    assert b.sim.restored is None, "the simulator was restored before the refusal"
