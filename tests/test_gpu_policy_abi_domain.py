"""qp_forward (csrc/policy_kernels.cu, include/quadpolicy.h) over the dimensions the C-ABI accepts but no QuadSimConfig produces:
A up to 8 (the head's outputs 4..7 are read through L1: the only tests of that branch), S 1..24 (the edges of the 8-wide K chunks of the
24 self slots), W 1 and 8 (the whole neighbour chunk live), V 1 (stream 1 never runs a neighbour pass) and 5, O 1..24 (O = 24: every
self slot of stream 1's x tile holds an obstacle column), with and without neighbours.

Handles are made directly (qp_create / qp_set_weights on QpConfigC / QpTowerWeightsC) from weights built here: xavier-uniform, biases
uniform +-0.3.  The reference is float64 with the kernel's bf16 rounding points -- the observations, every tensor-core weight, each
activation fed to the next layer and the neighbour mean after its fp32 sum * (1 / V) -- and everything else, heads included, in float64 on
the fp32 weights; the tolerance is that of the other policy parity files.  Each observation block is drawn at its own scale and offset,
so a column-offset error cannot pass.
"""
import ctypes as C
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu
TOL_EMU_MAX = 3e-3                    # tests/test_gpu_policy.py, tests/test_gpu_policy_obstacles.py
H, FF = 256, 512
WAVE = 148 * 128                      # one 128-row tile per SM of a B200


def bf16(x):
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def xavier(out_dim, in_dim, g):
    a = (6.0 / (in_dim + out_dim)) ** 0.5
    return (torch.rand(out_dim, in_dim, generator=g) * 2 - 1) * a


def make_tower(S, W, V, O, n_out, g):
    t = {"self_w1": xavier(H, S, g), "self_w2": xavier(H, H, g), "head_w": xavier(n_out, FF, g)}
    if V > 0:
        t["nbr_w1"], t["nbr_w2"] = xavier(H, W, g), xavier(H, H, g)
    if O > 0:
        t["obst_w1"], t["obst_w2"] = xavier(H, O, g), xavier(H, H, g)
    ff = xavier(FF, 3 * H if O > 0 else 2 * H, g)
    if V == 0:
        ff[:, H:2 * H] = 0.0                                      # the header: without neighbours the neighbour block is zeros
    t["ff_w"] = ff
    for w, b, n in (("self_w1", "self_b1", H), ("self_w2", "self_b2", H), ("nbr_w1", "nbr_b1", H), ("nbr_w2", "nbr_b2", H),
                    ("obst_w1", "obst_b1", H), ("obst_w2", "obst_b2", H), ("ff_w", "ff_b", FF), ("head_w", "head_b", n_out)):
        if w in t:
            t[b] = (torch.rand(n, generator=g) * 2 - 1) * 0.3
    return {k: v.float().cuda().contiguous() for k, v in t.items()}


def make_obs(n, S, W, V, O, stride, g):
    """Self block N(0, 0.8), neighbour block 0.4 + N(0, 1.5), obstacle block uniform [0.5, 3] (positive, like the SDF distances);
    padding columns behind them are large, so reading one would show."""
    obs = torch.full((n, stride), 50.0)
    obs[:, :S] = 0.8 * torch.randn(n, S, generator=g)
    obs[:, S:S + V * W] = 0.4 + 1.5 * torch.randn(n, V * W, generator=g)
    obs[:, S + V * W:S + V * W + O] = 0.5 + 2.5 * torch.rand(n, O, generator=g)
    return obs.cuda()


def reference(t, obs, S, W, V, O):
    x = obs.double()
    w = {k: v.double() for k, v in t.items()}

    def mlp2(p, inp, round_out):
        h1 = bf16(torch.tanh(bf16(inp) @ bf16(w[p + "_w1"]).t() + w[p + "_b1"]))
        h2 = torch.tanh(h1 @ bf16(w[p + "_w2"]).t() + w[p + "_b2"])
        return bf16(h2) if round_out else h2

    parts = [mlp2("self", x[:, :S], True)]
    if V > 0:
        s = sum(mlp2("nbr", x[:, S + j * W:S + (j + 1) * W], False) for j in range(V))
        parts.append(bf16(s * (1.0 / V)))                          # fp32 running sum times 1 / V, then one rounding
    else:
        parts.append(torch.zeros_like(parts[0]))
    if O > 0:
        parts.append(mlp2("obst", x[:, S + V * W:S + V * W + O], True))
    y = torch.tanh(torch.cat(parts, 1) @ bf16(w["ff_w"]).t() + w["ff_b"])
    return y @ w["head_w"].t() + w["head_b"]                       # heads: fp32 weights, no rounding


CASES = {
    # name: (S, W, V, O, A, n, stride padding)
    "S1-W1-V1-A3": (1, 1, 1, 0, 3, 77, 0),
    "S8-W8-V5-A5": (8, 8, 5, 0, 5, 77, 2),
    "S9-W1-V5-O1-A8": (9, 1, 5, 1, 8, 77, 0),
    "S24-W8-V1-O24-A8": (24, 8, 1, 24, 8, 77, 3),
    "S17-V0-O8-A3": (17, 6, 0, 8, 3, 77, 0),
    "S24-V0-O24-A5": (24, 6, 0, 24, 5, 77, 1),
    "S8-V0-O1-A8": (8, 0, 0, 1, 8, 77, 0),
    "S17-W8-V5-O8-A8": (17, 8, 5, 8, 8, 77, 0),
    "S1-W8-V5-A8-multiwave": (1, 8, 5, 0, 8, WAVE + 300 + 41, 0),
    "S24-W1-V1-O24-A5-multiwave": (24, 1, 1, 24, 5, 2 * WAVE + 77, 0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_forward_matches_emulated_reference(name):
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import QP_API_VERSION, QpConfigC, QpTowerWeightsC
    S, W, V, O, A, n, pad = CASES[name]
    stride = S + V * W + O + pad
    lib = _capi.lib()
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    towers = [make_tower(S, W, V, O, A, g), make_tower(S, W, V, O, 1, g)]
    obs = make_obs(n, S, W, V, O, stride, g)
    # NaN-filled outputs with 128 rows to spare: every live row must be written, nothing behind row n
    mean = torch.full((n + 128, A), float("nan"), device="cuda")
    value = torch.full((n + 128,), float("nan"), device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = C.c_void_p()
    assert lib.qp_create(C.byref(QpConfigC(QP_API_VERSION, S, W, V, H, A, O)), 0, C.byref(h)) == 0, lib.qp_last_error(None)
    try:
        for i, t in enumerate(towers):
            w = QpTowerWeightsC()
            for f in QpTowerWeightsC.FIELDS:
                setattr(w, f, t[f].data_ptr() if f in t else None)
            assert lib.qp_set_weights(h, i, C.byref(w), s) == 0, lib.qp_last_error(h)
        assert lib.qp_forward(h, obs.data_ptr(), n, stride, mean.data_ptr(), value.data_ptr(), s) == 0, lib.qp_last_error(h)
        torch.cuda.synchronize()
    finally:
        lib.qp_destroy(h)
    assert bool(mean[n:].isnan().all()) and bool(value[n:].isnan().all())
    r_mean, r_value = reference(towers[0], obs, S, W, V, O), reference(towers[1], obs, S, W, V, O)[:, 0]
    d_mean, d_value = (mean[:n].double() - r_mean).abs(), (value[:n].double() - r_value).abs()
    assert bool(d_mean.isfinite().all()) and bool(d_value.isfinite().all())
    per_out = d_mean.max(0).values
    print(f"\n[{name}] n={n} stride={stride}: max |d mean| per output {[f'{float(e):.1e}' for e in per_out]}, "
          f"max |d value| {float(d_value.max()):.1e}; |mean| up to {float(r_mean.abs().max()):.2f}")
    assert float(per_out.max()) <= TOL_EMU_MAX and float(d_value.max()) <= TOL_EMU_MAX
