"""qp_forward (csrc/policy_kernels.cu, include/quadpolicy.h) over the dimensions the C-ABI accepts but no QuadSimConfig produces:
A up to 8 (the head's outputs 4..7 are read through L1: the only tests of that branch), S 1..24 (the edges of the 8-wide K chunks of the
24 self slots), W 1 and 8 (the whole neighbour chunk live), V 1 (stream 1 never runs a neighbour pass) and 5, O 1..24 (O = 24: every
self slot of stream 1's x tile holds an obstacle column), with and without neighbours.

The MLP neighbour encoder (qp_create_encoder(QP_NBR_MLP)) reads its W * V inputs as one vector: inputs 0..31 fill stream 1's x tile,
inputs 32..39 the neighbour slots (24..31) of stream 0's, beside the self columns.  Its cases reach W * V = 1 .. 40 at the chunk edges
(8, 24, 31, 32, 33, 39, 40), with W 1 and 8, S 1..24 (S = 24 beside a full neighbour chunk of stream 0 at W * V = 32 and 40) and A 1..8.
`test_table_reaches_every_mlp_edge` fails when a case that reaches one of these edges is removed.

Handles are made directly (qp_create_encoder / qp_set_weights on QpConfigC / QpTowerWeightsC) from weights built here: xavier-uniform,
biases uniform +-0.3.  The reference is float64 with the kernel's bf16 rounding points -- the observations, every tensor-core weight, each
activation fed to the next layer, the MLP encoder's output and the neighbour mean after its fp32 sum * (1 / V) -- and everything else,
heads included, in float64 on the fp32 weights.  Each observation block is drawn at its own scale and offset (the MLP inputs 32..39 at
another one again), so a column-offset error cannot pass; `test_mlp_cases_see_every_input_slot` shows that dropping one edge column moves
each MLP case's reference by ten times its tolerance.  Every forward reads observations with NaN rows behind row n and writes outputs
with NaN rows behind row n: no live row may read them, and nothing behind row n may be written.

The tests without the gpu marker check the reference and the table and run anywhere.
"""
import ctypes as C
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from test_gpu_policy_mlp import TOL_EMU_MAX as TOL_EMU_MAX_MLP  # noqa: E402

gpu = pytest.mark.gpu
TOL_EMU_MAX = 3e-3                    # tests/test_gpu_policy.py, tests/test_gpu_policy_obstacles.py
H, FF = 256, 512
WAVE = 148 * 128                      # one 128-row tile per SM of a B200
SPARE = 128                           # NaN rows behind row n, in the observations and the outputs
MLP_MAX_INPUTS = 40


def bf16(x):
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def xavier(out_dim, in_dim, g):
    a = (6.0 / (in_dim + out_dim)) ** 0.5
    return (torch.rand(out_dim, in_dim, generator=g) * 2 - 1) * a


def make_tower(S, W, V, O, n_out, g, mlp=False):
    """One tower's weights (fp32, on the CPU).  mlp: nbr_w1 is [256, W * V] and the encoder has a third layer."""
    t = {"self_w1": xavier(H, S, g), "self_w2": xavier(H, H, g), "head_w": xavier(n_out, FF, g)}
    if V > 0:
        t["nbr_w1"], t["nbr_w2"] = xavier(H, W * V if mlp else W, g), xavier(H, H, g)
    if mlp:
        t["nbr_w3"] = xavier(H, H, g)
    if O > 0:
        t["obst_w1"], t["obst_w2"] = xavier(H, O, g), xavier(H, H, g)
    ff = xavier(FF, 3 * H if O > 0 else 2 * H, g)
    if V == 0:
        ff[:, H:2 * H] = 0.0                                      # the header: without neighbours the neighbour block is zeros
    t["ff_w"] = ff
    for w, b, n in (("self_w1", "self_b1", H), ("self_w2", "self_b2", H), ("nbr_w1", "nbr_b1", H), ("nbr_w2", "nbr_b2", H),
                    ("obst_w1", "obst_b1", H), ("obst_w2", "obst_b2", H), ("ff_w", "ff_b", FF), ("head_w", "head_b", n_out),
                    ("nbr_w3", "nbr_b3", H)):
        if w in t:
            t[b] = (torch.rand(n, generator=g) * 2 - 1) * 0.3
    return {k: v.float().contiguous() for k, v in t.items()}


def make_obs(n, S, W, V, O, stride, g, mlp=False):
    """[n + SPARE, stride] fp32 on the CPU.  Self block N(0, 0.8), neighbour block 0.4 + N(0, 1.5) (MLP inputs 32..39: uniform [1, 3]),
    obstacle block uniform [0.5, 3] (positive, like the SDF distances); padding columns behind them are 50, so reading one would show;
    rows n.. are NaN."""
    obs = torch.full((n + SPARE, stride), 50.0)
    obs[:n, :S] = 0.8 * torch.randn(n, S, generator=g)
    obs[:n, S:S + V * W] = 0.4 + 1.5 * torch.randn(n, V * W, generator=g)
    obs[:n, S + V * W:S + V * W + O] = 0.5 + 2.5 * torch.rand(n, O, generator=g)
    if mlp and V * W > 32:
        obs[:n, S + 32:S + V * W] = 1.0 + 2.0 * torch.rand(n, V * W - 32, generator=g)
    obs[n:] = float("nan")
    return obs


def reference(t, obs, S, W, V, O, mlp=False, rounded=True):
    """One tower on obs [n, >= S + V * W + O] in float64; rounded: with the kernel's bf16 rounding points."""
    r = bf16 if rounded else (lambda v: v)
    x = obs.double()
    w = {k: v.double() for k, v in t.items()}

    def layer(p, inp):
        return torch.tanh(inp @ r(w[p[0]]).t() + w[p[1]])

    def mlp2(p, inp, round_out):
        h1 = r(layer((p + "_w1", p + "_b1"), r(inp)))
        h2 = layer((p + "_w2", p + "_b2"), h1)
        return r(h2) if round_out else h2

    parts = [mlp2("self", x[:, :S], True)]
    if mlp:
        h = r(x[:, S:S + V * W])
        for i in (1, 2, 3):
            h = r(layer((f"nbr_w{i}", f"nbr_b{i}"), h))
        parts.append(h)
    elif V > 0:
        s = sum(mlp2("nbr", x[:, S + j * W:S + (j + 1) * W], False) for j in range(V))
        parts.append(r(s * (1.0 / V)))                             # fp32 running sum times 1 / V, then one rounding
    else:
        parts.append(torch.zeros_like(parts[0]))
    if O > 0:
        parts.append(mlp2("obst", x[:, S + V * W:S + V * W + O], True))
    y = torch.tanh(torch.cat(parts, 1) @ r(w["ff_w"]).t() + w["ff_b"])
    return y @ w["head_w"].t() + w["head_b"]                       # heads: fp32 weights, no rounding


CASES = {
    # name: (neighbour encoder, S, W, V, O, A, n, stride padding)
    "S1-W1-V1-A3": ("mean_embed", 1, 1, 1, 0, 3, 77, 0),
    "S8-W8-V5-A5": ("mean_embed", 8, 8, 5, 0, 5, 77, 2),
    "S9-W1-V5-O1-A8": ("mean_embed", 9, 1, 5, 1, 8, 77, 0),
    "S24-W8-V1-O24-A8": ("mean_embed", 24, 8, 1, 24, 8, 77, 3),
    "S17-V0-O8-A3": ("mean_embed", 17, 6, 0, 8, 3, 77, 0),
    "S24-V0-O24-A5": ("mean_embed", 24, 6, 0, 24, 5, 77, 1),
    "S8-V0-O1-A8": ("mean_embed", 8, 0, 0, 1, 8, 77, 0),
    "S17-W8-V5-O8-A8": ("mean_embed", 17, 8, 5, 8, 8, 77, 0),
    "S1-W8-V5-A8-multiwave": ("mean_embed", 1, 8, 5, 0, 8, WAVE + 300 + 41, 0),
    "S24-W1-V1-O24-A5-multiwave": ("mean_embed", 24, 1, 1, 24, 5, 2 * WAVE + 77, 0),
    # MLP neighbour encoder, named by W * V
    "mlp-WV1-S1-W1-V1-A1": ("mlp", 1, 1, 1, 0, 1, 77, 0),
    "mlp-WV8-S8-W8-V1-A5": ("mlp", 8, 8, 1, 0, 5, 77, 0),
    "mlp-WV24-S9-W3-V8-A8": ("mlp", 9, 3, 8, 0, 8, 77, 0),
    "mlp-WV31-S23-W1-V31-A3": ("mlp", 23, 1, 31, 0, 3, 77, 0),
    "mlp-WV32-S24-W8-V4-A8": ("mlp", 24, 8, 4, 0, 8, 77, 0),
    "mlp-WV33-S1-W3-V11-A5": ("mlp", 1, 3, 11, 0, 5, 77, 0),
    "mlp-WV39-S17-W1-V39-A2": ("mlp", 17, 1, 39, 0, 2, 77, 0),
    "mlp-WV40-S24-W8-V5-A8-padded": ("mlp", 24, 8, 5, 0, 8, 77, 3),
    "mlp-WV40-S24-W5-V8-A8-multiwave": ("mlp", 24, 5, 8, 0, 8, 2 * WAVE + 77, 0),
    "mlp-WV40-S7-W1-V40-A4-multiwave": ("mlp", 7, 1, 40, 0, 4, 3 * WAVE + 41, 0),
    "mlp-cfg2-n1": ("mlp", 18, 6, 6, 0, 4, 1, 0),
    "mlp-cfg2-n128": ("mlp", 18, 6, 6, 0, 4, 128, 0),
    "mlp-cfg2-n129": ("mlp", 18, 6, 6, 0, 4, 129, 0),
}
MLP_CASES = [name for name, c in CASES.items() if c[0] == "mlp"]


def case_inputs(name, n=None):
    """(towers [actor, critic], obs [n + SPARE, stride], stride) of a case, on the CPU; n: fewer rows than the case has."""
    kind, S, W, V, O, A, n_case, pad = CASES[name]
    mlp = kind == "mlp"
    stride = S + V * W + O + pad
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    towers = [make_tower(S, W, V, O, A, g, mlp), make_tower(S, W, V, O, 1, g, mlp)]
    return towers, make_obs(n or n_case, S, W, V, O, stride, g, mlp), stride


@gpu
@pytest.mark.parametrize("name", list(CASES))
def test_forward_matches_emulated_reference(name):
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    from quad_swarm_rl_stable_baselines3_b200.fused_policy import QP_API_VERSION, QP_NBR, QpConfigC, QpTowerWeightsC
    kind, S, W, V, O, A, n, pad = CASES[name]
    mlp = kind == "mlp"
    lib = _capi.lib()
    towers, obs, stride = case_inputs(name)
    towers = [{k: v.cuda() for k, v in t.items()} for t in towers]
    obs = obs.cuda()
    # NaN-filled outputs with SPARE rows to spare: every live row must be written, nothing behind row n
    mean = torch.full((n + SPARE, A), float("nan"), device="cuda")
    value = torch.full((n + SPARE,), float("nan"), device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = C.c_void_p()
    cfg = QpConfigC(QP_API_VERSION, S, W, V, H, A, O)
    assert lib.qp_create_encoder(C.byref(cfg), QP_NBR[kind], 0, C.byref(h)) == 0, lib.qp_last_error(None)
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
    r_mean = reference(towers[0], obs[:n], S, W, V, O, mlp)
    r_value = reference(towers[1], obs[:n], S, W, V, O, mlp)[:, 0]
    d_mean, d_value = (mean[:n].double() - r_mean).abs(), (value[:n].double() - r_value).abs()
    assert bool(d_mean.isfinite().all()) and bool(d_value.isfinite().all())
    per_out = d_mean.max(0).values
    print(f"\n[{name}] n={n} stride={stride}: max |d mean| per output {[f'{float(e):.1e}' for e in per_out]}, "
          f"max |d value| {float(d_value.max()):.1e}; |mean| up to {float(r_mean.abs().max()):.2f}")
    tol = TOL_EMU_MAX_MLP if mlp else TOL_EMU_MAX
    assert float(per_out.max()) <= tol and float(d_value.max()) <= tol


# ---- checks of the reference and of the table: no GPU -------------------------------------------------------------------------
def load_module(towers, cfg, kind):
    """QuadActorCritic in float64 with the weights of the tower dicts [actor, critic] (a strict load: every parameter comes from them)."""
    from quad_swarm_rl_stable_baselines3_b200.ppo import QuadActorCritic
    pol = QuadActorCritic(cfg, neighbor_encoder=kind).double()
    layers = {"self_encoder.0": "self_w1", "self_encoder.2": "self_w2", "feed_forward.0": "ff_w", "neighbor.0": "nbr_w1",
              "neighbor.2": "nbr_w2", "neighbor.4": "nbr_w3", "obstacle.0": "obst_w1", "obstacle.2": "obst_w2"}
    sd = {}
    for enc, head, t in (("actor", "action_net", towers[0]), ("critic", "value_net", towers[1])):
        for mod, key in layers.items():
            if key in t:
                sd[f"{enc}.{mod}.weight"], sd[f"{enc}.{mod}.bias"] = t[key], t[key.replace("_w", "_b")]
        sd[f"{head}.weight"], sd[f"{head}.bias"] = t["head_w"], t["head_b"]
    sd["log_std"] = pol.log_std.detach()
    pol.load_state_dict({k: v.double() for k, v in sd.items()})
    return pol


@pytest.mark.parametrize("which", ["mean_embed", "mean_embed_obstacles", "mlp"])
def test_unrounded_reference_is_the_module(which):
    """`reference` without its rounding points is QuadActorCritic's forward, in float64 on the same weights."""
    from quad_swarm_rl_stable_baselines3_b200.config import NEIGHBOR_OBS_DIM, OBS_REPR_DIM, QuadSimConfig
    if which == "mean_embed_obstacles":
        cfg = QuadSimConfig(num_envs=2, num_agents=8, quads_mode="mix", use_obstacles=True, use_downwash=True,
                            obs_repr="xyz_vxyz_R_omega_floor", neighbor_visible_num=2)                 # cfg3: S 19, W 6, V 2, O 9
    else:
        cfg = QuadSimConfig(num_envs=2, num_agents=8)                                              # cfg2: S 18, W 6, V 6
    kind = "mlp" if which == "mlp" else "mean_embed"
    mlp = kind == "mlp"
    S, W, V, O, A = OBS_REPR_DIM[cfg.obs_repr], NEIGHBOR_OBS_DIM[cfg.neighbor_obs_type], cfg.visible, 9 * cfg.use_obstacles, cfg.act_dim
    g = torch.Generator().manual_seed(11)
    towers = [make_tower(S, W, V, O, A, g, mlp), make_tower(S, W, V, O, 1, g, mlp)]
    pol = load_module(towers, cfg, kind)
    n = 300
    obs = make_obs(n, S, W, V, O, cfg.obs_dim, g, mlp)[:n].double()
    with torch.no_grad():
        m_mean, m_value = pol.action_net(pol.actor(obs)), pol.value(obs)
    r_mean = reference(towers[0], obs, S, W, V, O, mlp, rounded=False)
    r_value = reference(towers[1], obs, S, W, V, O, mlp, rounded=False)[:, 0]
    assert float((m_mean - r_mean).abs().max()) <= 1e-12 and float((m_value - r_value).abs().max()) <= 1e-12
    # the rounding points are where the tolerance goes: without them the reference would sit well outside it
    e_mean = reference(towers[0], obs, S, W, V, O, mlp)
    assert float((e_mean - r_mean).abs().max()) > (TOL_EMU_MAX_MLP if mlp else TOL_EMU_MAX)


@pytest.mark.parametrize("name", MLP_CASES)
def test_mlp_cases_see_every_input_slot(name):
    """Zeroing one edge column -- the last self column, the last of inputs 0..31, input 32, the last input -- moves the rounded reference
    by more than ten times the tolerance: a kernel that drops, duplicates or shifts that slot cannot pass the case."""
    _, S, W, V, O, A, _, _ = CASES[name]
    WV = W * V
    n = 128
    towers, obs, _ = case_inputs(name, n)
    x = obs[:n].double()
    base = [reference(t, x, S, W, V, O, True) for t in towers]
    cols = {S - 1, S + min(WV, 32) - 1, S + WV - 1} | ({S + 32} if WV > 32 else set())
    for c in sorted(cols):
        xz = x.clone()
        xz[:, c] = 0.0
        moved = max(float((reference(t, xz, S, W, V, O, True) - b).abs().max()) for t, b in zip(towers, base))
        assert moved > 10 * TOL_EMU_MAX_MLP, (name, c, moved)


def test_table_reaches_every_mlp_edge():
    """The MLP cases reach every edge of the variant's input layout, head and row loop (see the module docstring)."""
    mlp = [CASES[k][1:] for k in MLP_CASES]                       # (S, W, V, O, A, n, pad)
    wv = {W * V for S, W, V, O, A, n, pad in mlp}
    assert {1, 8, 24, 31, 32, 33, 39, 40} <= wv, wv
    assert max(W * V for S, W, V, O, A, n, pad in mlp) == MLP_MAX_INPUTS
    assert any(W == 1 and V == MLP_MAX_INPUTS for S, W, V, O, A, n, pad in mlp)           # one neighbour column per row, V at the limit
    assert any(W == 8 for S, W, V, O, A, n, pad in mlp)
    assert {1, 8, 9, 23, 24} <= {S for S, W, V, O, A, n, pad in mlp}
    assert {(24, 32), (24, 40)} <= {(S, W * V) for S, W, V, O, A, n, pad in mlp}           # stream 0's x tile full: self and neighbour slots
    assert {1, 5, 8} <= {A for S, W, V, O, A, n, pad in mlp}
    assert {1, 128, 129} <= {n for S, W, V, O, A, n, pad in mlp}
    assert any(n > 2 * WAVE and n % 128 for S, W, V, O, A, n, pad in mlp)                 # more than two waves, ragged last tile
    assert any(pad > 0 for S, W, V, O, A, n, pad in mlp)
    assert {1, 128, 129} <= {n for S, W, V, O, A, n, pad in mlp if (S, W, V, A) == (18, 6, 6, 4)}   # cfg2's shape
    assert all(O == 0 and 1 <= S <= 24 and 1 <= W <= 8 and W * V <= MLP_MAX_INPUTS and 1 <= A <= 8 for S, W, V, O, A, n, pad in mlp)
