"""The PPO update's elementwise kernels and GAE (include/quadpolicy.h: qp_bias_tanh[_mean][_backward], qp_bias_tanh_backward_first,
qp_gae) called through the C-ABI, against plain float64 restatements of each operation.

Two kinds of case:
  * exact arithmetic: inputs for which every fp32 product and every partial column sum is exact (y in {0, +-1/4, +-1/2, +-3/4}, so 1 - y^2
    is a multiple of 1/16; integer gradients and inputs).  The kernels must then match float64 bit for bit, whatever their summation
    order: a lost, duplicated or misattributed row, column, block partial or atomic fails.  All these values are exact in bf16 too.
  * random values, with a tolerance derived next to each assert.

Shapes are chosen to reach each kernel's paths (see `lanes` and `bwd_stride`): the 16-byte (v8) kernels and their two-rows-in-flight
loop, the pair fallback (h % 8 != 0 or pointers not 16-byte aligned), every first-layer template instantiation.  Every case id names
the kernel path it is for; each case prints its largest error.

The reference functions are checked against torch.autograd in float64 by the tests without the gpu marker, which run anywhere.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

gpu = pytest.mark.gpu
U = 2.0 ** -24                       # fp32 unit roundoff
BWD_GRID_CAP = 592                   # the backward launches use at most 592 blocks (4 per SM of a B200)
B200_SMS = 148
EXACT_VALUES_Y = (0.0, 0.25, -0.25, 0.5, -0.5, 0.75, -0.75)


# ---- float64 references: plain restatements of the operations ------------------------------------------------------------------
def ref_bias_tanh(z, b):
    return torch.tanh(z.double() + b.double())


def ref_bias_tanh_backward(gy, y):
    gz = gy.double() * (1.0 - y.double() ** 2)
    return gz, gz.sum(0)


def ref_backward_first(gy, y, x):
    gz = gy.double() * (1.0 - y.double() ** 2)
    return gz.t() @ x.double(), gz.sum(0)                       # grad_weight [h, in] (nn.Linear layout), grad_bias [h]


def ref_mean(y, V):
    return y.double().reshape(-1, V, y.shape[1]).sum(1) / V


def ref_mean_backward(gm, y, V):
    yy = y.double().reshape(-1, V, y.shape[1])
    gz = (gm.double()[:, None, :] / V) * (1.0 - yy ** 2)
    gz = gz.reshape(-1, y.shape[1])
    return gz, gz.sum(0)


def ref_gae(rew, val, done, last_val, gamma, lam):
    """SB3's recursion, backwards in time: delta_t = r_t + gamma V_{t+1} (1 - d_t) - V_t, A_t = delta_t + gamma lam (1 - d_t) A_{t+1}."""
    rew, val, last_val = rew.double(), val.double(), last_val.double()
    nt = 1.0 - done.double()
    adv = torch.empty_like(rew)
    nxt, last = last_val, torch.zeros_like(last_val)
    for t in range(rew.shape[0] - 1, -1, -1):
        delta = rew[t] + gamma * nxt * nt[t] - val[t]
        last = delta + gamma * lam * nt[t] * last
        adv[t] = last
        nxt = val[t]
    return adv, adv + val


def bf16_ulp(x):
    """Spacing of bf16 numbers (8 significand bits) at |x|, x float64."""
    _, e = torch.frexp(x.abs())
    return torch.ldexp(torch.ones_like(x), e - 8)


def bf16_rn(x):
    """x float64 rounded to the nearest bf16, ties to even, in one step (no detour through fp32)."""
    q = bf16_ulp(x)
    return torch.round(x / q) * q


# ---- kernel geometry (csrc/policy_kernels.cu) ---------------------------------------------------------------------------------
def lanes(h):
    """v8 kernels: a thread owns 8 adjacent columns; G column groups x RL row lanes per block."""
    G = h // 8
    return G, (1 if G >= 256 else 256 // G)


def bwd_stride(h, n, sms=B200_SMS):
    """Rows between two trips of one lane of a v8 backward kernel (grid * RL).  Its main loop handles rows r and r + stride per trip
    while r + stride < n, so it runs only when n > stride; n >= 4 * stride makes every lane take it twice."""
    _, RL = lanes(h)
    return min(-(-n // RL), 8 * sms, BWD_GRID_CAP) * RL


def loop_n(h, trips=4):
    """trips * 592 * RL rows plus a remainder that is not a multiple of RL: with the grid at its 592-block cap, every lane runs the
    two-row loop trips // 2 times and some lanes the one-row tail after it."""
    _, RL = lanes(h)
    return trips * BWD_GRID_CAP * RL + 37 * RL + 5


# ---- case tables ----------------------------------------------------------------------------------------------------------------
def _bt_cases():
    out = []
    for h in (8, 24, 48, 256, 1000, 2048):
        for n in (1, 7, 1003, loop_n(h)):
            out.append(("v8", h, n, 0))
    for h in (2, 6, 250, 2046):
        for n in (1, 7, 1003, 3 * 8 * B200_SMS + 17):
            out.append(("pair", h, n, 0))
    for n in (7, 1003, 3 * 8 * B200_SMS + 17):
        out.append(("pair", 256, n, 2))          # pair-aligned but not 16-byte aligned: the v8 kernels are skipped
    return out


def _bt_id(c):
    path, h, n, off = c
    tag = "loop2+tail" if path == "v8" and n == loop_n(h) else "tail" if path == "v8" else "rows"
    return f"{path}-{tag}-h{h}-n{n}" + (f"-off{off}" if off else "")


BT_CASES = _bt_cases()
FIRST_CASES = [(h, k, n) for h in (8, 48, 256, 2048) for k in range(1, 9) for n in (37, loop_n(h, trips=2))]
MEAN_CASES = ([(V, h, g) for V in (1, 2, 3) for h in (8, 48, 256, 2048) for g in (1, 5, loop_n(h, trips=2))]
              + [(V, h, g) for V in (7, 31) for h in (8, 48, 256, 2048) for g in (1, 5)]
              + [(V, 48, loop_n(48, trips=2)) for V in (7, 31)])
GAE_SHAPES = [(1, 1), (2, 255), (128, 256), (1024, 257), (128, 65537), (1024, 1)]
DONE_PATTERNS = ("none", "all", "last", "first", "random")
DTYPES = ("fp32", "bf16")
TD = {"fp32": torch.float32, "bf16": torch.bfloat16}


# ---- input generators ------------------------------------------------------------------------------------------------------------
def exact_y(shape, g):
    vals = torch.tensor(EXACT_VALUES_Y, dtype=torch.float64)
    return vals[torch.randint(0, len(EXACT_VALUES_Y), shape, generator=g)]


def exact_int(shape, g, lo=-2, hi=2):
    return torch.randint(lo, hi + 1, shape, generator=g).double()


def assert_exact_bound(abs_sums, quantum):
    """Every term is a multiple of `quantum` and every partial sum of a column is bounded by the column's sum of |terms|: if that is
    below 2^24 quanta, fp32 holds every partial sum exactly, in any order."""
    bound = float(abs_sums.max()) / quantum
    assert bound < 2 ** 24, f"exact-arithmetic case too large: {bound:.3g} quanta >= 2^24"


def done_pattern(kind, T, n, g):
    d = torch.zeros((T, n), dtype=torch.bool)
    if kind == "all":
        d[:] = True
    elif kind == "last":
        d[T - 1] = True
    elif kind == "first":
        d[0] = True
    elif kind == "random":
        d = torch.rand((T, n), generator=g) < 0.1
    return d


# ---- CPU self-checks of the references ------------------------------------------------------------------------------------------
def test_reference_bias_tanh_matches_autograd():
    g = torch.Generator().manual_seed(0)
    z = torch.randn(37, 24, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(24, generator=g, dtype=torch.float64, requires_grad=True)
    y = torch.tanh(z + b)
    gy = torch.randn(37, 24, generator=g, dtype=torch.float64)
    y.backward(gy)
    assert torch.allclose(ref_bias_tanh(z.detach(), b.detach()), y.detach(), rtol=0, atol=1e-15)
    gz, gb = ref_bias_tanh_backward(gy, y.detach())
    assert torch.allclose(gz, z.grad, rtol=1e-13, atol=1e-15) and torch.allclose(gb, b.grad, rtol=1e-13, atol=1e-14)


def test_reference_backward_first_matches_autograd():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(53, 6, generator=g, dtype=torch.float64)
    lin = torch.nn.Linear(6, 16).double()
    y = torch.tanh(lin(x))
    gy = torch.randn(53, 16, generator=g, dtype=torch.float64)
    y.backward(gy)
    gw, gb = ref_backward_first(gy, y.detach(), x)
    assert gw.shape == lin.weight.shape
    assert torch.allclose(gw, lin.weight.grad, rtol=1e-13, atol=1e-14) and torch.allclose(gb, lin.bias.grad, rtol=1e-13, atol=1e-14)


@pytest.mark.parametrize("V", [1, 3, 7])
def test_reference_mean_matches_autograd(V):
    g = torch.Generator().manual_seed(V)
    z = torch.randn(5 * V, 16, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(16, generator=g, dtype=torch.float64, requires_grad=True)
    y = torch.tanh(z + b)
    m = y.view(5, V, 16).mean(1)
    gm = torch.randn(5, 16, generator=g, dtype=torch.float64)
    m.backward(gm)
    assert torch.allclose(ref_mean(y.detach(), V), m.detach(), rtol=0, atol=1e-15)
    gz, gb = ref_mean_backward(gm, y.detach(), V)
    assert torch.allclose(gz, z.grad, rtol=1e-13, atol=1e-15) and torch.allclose(gb, b.grad, rtol=1e-13, atol=1e-14)


@pytest.mark.parametrize("pattern", DONE_PATTERNS)
def test_reference_gae_matches_explicit_sum(pattern):
    """The recursion against its closed form A_t = sum_k (gamma lam)^(k - t) [no episode end in t .. k-1] delta_k, one element at a time."""
    g = torch.Generator().manual_seed(5)
    T, n, gamma, lam = 9, 4, 0.99, 0.95
    rew, val = torch.randn(T, n, generator=g, dtype=torch.float64), torch.randn(T, n, generator=g, dtype=torch.float64)
    last = torch.randn(n, generator=g, dtype=torch.float64)
    done = done_pattern(pattern, T, n, g)
    adv, ret = ref_gae(rew, val, done, last, gamma, lam)
    for i in range(n):
        for t in range(T):
            a, w = 0.0, 1.0
            for k in range(t, T):
                nv = float(last[i]) if k == T - 1 else float(val[k + 1, i])
                nt = 0.0 if done[k, i] else 1.0
                a += w * (float(rew[k, i]) + gamma * nv * nt - float(val[k, i]))
                w *= gamma * lam * nt
            assert abs(a - float(adv[t, i])) <= 1e-12
            assert abs(a + float(val[t, i]) - float(ret[t, i])) <= 1e-12


def test_bf16_rounding_helper():
    # ties go to the even neighbour: 1 + 2^-8 lies between 1 and 1 + 2^-7, 1 + 3 * 2^-8 between 1 + 2^-7 and 1 + 2^-6
    ties = torch.tensor([1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -(0.5 + 2 ** -9)], dtype=torch.float64)
    assert bf16_rn(ties).tolist() == [1.0, 1.0 + 2 ** -6, -0.5]
    x = torch.randn(10000, generator=torch.Generator().manual_seed(0), dtype=torch.float32)   # fp32 -> bf16 is one rounding in torch
    assert torch.equal(bf16_rn(x.double()), x.to(torch.bfloat16).double())
    assert float(bf16_ulp(torch.tensor([0.75], dtype=torch.float64))) == 2 ** -8


def test_cases_reach_the_two_row_loops():
    """On a B200 (148 SMs) the large cases run the backward kernels' two-row loop: twice per lane for the v8 table, once for the
    first-layer and mean tables; the exact-arithmetic bound of 2^24 quanta leaves room for them."""
    for path, h, n, _ in BT_CASES:
        if path == "v8" and n > 1003:
            s = bwd_stride(h, n)
            assert s == BWD_GRID_CAP * lanes(h)[1] and n >= 4 * s and n % s != 0, (h, n)
            assert 2 * n * 16 < 2 ** 24 or h == 8      # |grad_z| <= 2; h = 8 (606 k rows) is checked on its drawn values
    for h, _, n in FIRST_CASES:
        if n > 37:
            assert n > 2 * bwd_stride(h, n)
    for V, h, groups in MEAN_CASES:
        if groups > 5:
            assert groups > 2 * bwd_stride(h, groups)


# ---- GPU helpers -----------------------------------------------------------------------------------------------------------------
def _lib():
    from quad_swarm_rl_stable_baselines3_b200 import _capi
    return _capi.lib()


def _stream(s=None):
    return C.c_void_p((s if s is not None else torch.cuda.current_stream()).cuda_stream)


def _err():
    return _lib().qp_last_error(None).decode()


def _view(n, h, dtype, off=0, fill=float("nan")):
    """[n, h] contiguous CUDA tensor starting `off` elements into its allocation (the allocation itself is 512-byte aligned)."""
    buf = torch.full((n * h + off + 8,), fill, dtype=dtype, device="cuda")
    return buf[off:off + n * h].view(n, h)


def _close_bf16(got, ref64, ulps, what, atol=0.0):
    """|got - RN(ref)| <= ulps bf16 ulps (at the larger magnitude of the two) + atol (an fp32 error before the final rounding)."""
    r = bf16_rn(ref64)
    d = (got.double() - r).abs()
    lim = ulps * bf16_ulp(torch.maximum(got.double().abs(), r.abs())) + atol
    bad = d > lim
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} elements beyond {ulps} bf16 ulp, max |d| {float(d.max()):.3g}"
    return float(d.max())


# ---- qp_bias_tanh / qp_bias_tanh_backward ------------------------------------------------------------------------------------------
def _call_fwd(z, b, y, s=None):
    return _lib().qp_bias_tanh(z.data_ptr(), b.data_ptr(), z.shape[0], z.shape[1], int(z.dtype == torch.bfloat16), y.data_ptr(), _stream(s))


def _call_bwd(gy, y, gz, gb, s=None):
    return _lib().qp_bias_tanh_backward(gy.data_ptr(), y.data_ptr(), y.shape[0], y.shape[1], int(y.dtype == torch.bfloat16), gz.data_ptr(),
                                        gb.data_ptr(), _stream(s))


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("case", BT_CASES, ids=_bt_id)
def test_bias_tanh_forward(case, dt):
    path, h, n, off = case
    g = torch.Generator().manual_seed(h * 7919 + n)
    z = _view(n, h, TD[dt], off)
    z.copy_((2.0 * torch.randn(n, h, generator=g)).to("cuda"))
    b = (torch.rand(h, generator=g) * 2 - 1).cuda()
    y = _view(n, h, TD[dt], off)
    assert _call_fwd(z, b, y) == 0, _err()
    torch.cuda.synchronize()
    ref = ref_bias_tanh(z, b)
    if dt == "fp32":
        # one rounding of z + b (|z + b| < 16: <= 2^-20, times tanh' <= 1) plus tanhf's 2 ulp of a result below 1 (2^-23): < 1.3e-6
        err = float((y.double() - ref).abs().max())
        assert err <= 1.3e-6
    else:
        # bf16 z is exact in fp32; the fp32 error above (~1e-6) can move the final rounding across a bf16 tie: 1 ulp of RN(ref)
        err = _close_bf16(y, ref, 1, "y")
    print(f"\n[bias_tanh {_bt_id(case)} {dt}] max |y - ref| {err:.2e}")


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("case", BT_CASES, ids=_bt_id)
def test_bias_tanh_backward_exact(case, dt):
    path, h, n, off = case
    g = torch.Generator().manual_seed(h * 104729 + n)
    yv, gv = exact_y((n, h), g), exact_int((n, h), g)
    y, gy = _view(n, h, TD[dt], off), _view(n, h, TD[dt], off)
    y.copy_(yv.to("cuda")); gy.copy_(gv.to("cuda"))
    gz = _view(n, h, TD[dt], off, fill=1e30)
    gb = torch.full((h,), 1e30, device="cuda")                  # garbage: the call zeroes grad_bias itself
    ref_gz, ref_gb = ref_bias_tanh_backward(gy.cuda(), y.cuda())
    assert_exact_bound((gv * (1 - yv ** 2)).abs().sum(0), 1 / 16)
    assert _call_bwd(gy, y, gz, gb) == 0, _err()
    torch.cuda.synchronize()
    assert torch.equal(gz.double(), ref_gz), f"grad_z: max |d| {float((gz.double() - ref_gz).abs().max())}"
    assert torch.equal(gb.double(), ref_gb), f"grad_bias: max |d| {float((gb.double() - ref_gb).abs().max())}"
    print(f"\n[bias_tanh_backward {_bt_id(case)} {dt}] exact" + (f", lane stride {bwd_stride(h, n)}" if path == "v8" else ""))


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("h", [8, 48, 1000, 2048])
def test_bias_tanh_backward_random(h, dt):
    n = loop_n(h)
    g = torch.Generator().manual_seed(h)
    y = torch.tanh(torch.randn(n, h, generator=g) * 1.5).to("cuda", TD[dt])
    gy = torch.randn(n, h, generator=g).to("cuda", TD[dt])
    gz, gb = torch.empty_like(y), torch.empty(h, device="cuda")
    assert _call_bwd(gy, y, gz, gb) == 0, _err()
    torch.cuda.synchronize()
    ref_gz, ref_gb = ref_bias_tanh_backward(gy, y)              # products of the values as stored (bf16 exact in fp32)
    if dt == "fp32":
        # o = g (1 - t t): t t rounds (u t^2), 1 - t t at most once more (u), the product once (u |o|): |d| <= 3 u |g|
        e_gz = float((gz.double() - ref_gz).abs().max())
        assert bool(((gz.double() - ref_gz).abs() <= 3 * U * gy.double().abs() + 1e-30).all())
    else:
        e_gz = _close_bf16(gz, ref_gz, 1, "grad_z")             # fp32 o (3 u) rounded once to bf16
    # grad_bias sums the fp32 products (never the bf16-rounded grad_z): each product is off by <= 3 u |g| (above), and the longest chain
    # of additions is 2 per lane trip + RL shared-memory partials + one atomic per block: |d| <= chain u sum |o| + 3 u sum |g|
    _, RL = lanes(h)
    s = bwd_stride(h, n)
    chain = 2 * -(-n // s) + RL + s // RL
    lim = chain * U * ref_gz.abs().sum(0) + 3 * U * gy.double().abs().sum(0)
    e_gb = (gb.double() - ref_gb).abs()
    assert bool((e_gb <= lim).all()), float((e_gb / lim).max())
    print(f"\n[bias_tanh_backward v8-loop2+tail-h{h}-n{n} {dt} random] max |d grad_z| {e_gz:.2e}, max |d grad_bias| {float(e_gb.max()):.2e}")


# ---- qp_bias_tanh_backward_first ----------------------------------------------------------------------------------------------------
def _call_first(gy, y, x, ws, gb, gw, s=None):
    return _lib().qp_bias_tanh_backward_first(gy.data_ptr(), y.data_ptr(), x.data_ptr(), y.shape[0], y.shape[1], x.shape[1],
                                              int(y.dtype == torch.bfloat16), ws.data_ptr(), gb.data_ptr(), gw.data_ptr(), _stream(s))


def _workspace(h, k):
    nbytes = int(_lib().qp_bias_tanh_backward_first_workspace(h, k))
    assert nbytes == BWD_GRID_CAP * (k + 1) * h * 4                 # one fp32 partial per block (<= 592), input and column
    buf = torch.full((nbytes // 4 + 64,), float("nan"), device="cuda")  # NaN garbage, and 64 canaries behind the workspace
    return buf[:nbytes // 4], buf[nbytes // 4:]


def _first_id(c):
    h, k, n = c
    return f"w_kernel-IN{k}-h{h}-n{n}-" + ("loop+tail" if n > 37 else "tail")


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("case", FIRST_CASES, ids=_first_id)
def test_bias_tanh_backward_first_exact(case, dt):
    h, k, n = case
    g = torch.Generator().manual_seed(h * 31 + k * 7 + n)
    yv, gv, xv = exact_y((n, h), g), exact_int((n, h), g), exact_int((n, k), g)
    y, gy, x = yv.to("cuda", TD[dt]), gv.to("cuda", TD[dt]), xv.float().cuda()
    ws, canary = _workspace(h, k)
    gb, gw = torch.full((h,), 1e30, device="cuda"), torch.full((h, k), 1e30, device="cuda")
    gz = gv * (1 - yv ** 2)
    assert_exact_bound(torch.cat([gz.abs().sum(0), (gz.abs().t() @ xv.abs()).reshape(-1)]), 1 / 16)
    ref_gw, ref_gb = ref_backward_first(gy, y, x)
    for _ in range(2):                                              # a second call into the same buffers gives the same result
        assert _call_first(gy, y, x, ws, gb, gw) == 0, _err()
        torch.cuda.synchronize()
        assert torch.equal(gb.double(), ref_gb), f"grad_bias: max |d| {float((gb.double() - ref_gb).abs().max())}"
        assert torch.equal(gw.double(), ref_gw), f"grad_weight: max |d| {float((gw.double() - ref_gw).abs().max())}"
    assert bool(canary.isnan().all())
    print(f"\n[bias_tanh_backward_first {_first_id(case)} {dt}] exact")


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("k", [1, 6, 8])
def test_bias_tanh_backward_first_random(k, dt):
    h = 256
    n = loop_n(h, trips=2)
    g = torch.Generator().manual_seed(k)
    y = torch.tanh(torch.randn(n, h, generator=g)).to("cuda", TD[dt])
    gy = torch.randn(n, h, generator=g).to("cuda", TD[dt])
    x = torch.randn(n, k, generator=g).cuda()
    ws, _ = _workspace(h, k)
    gb, gw = torch.empty(h, device="cuda"), torch.empty(h, k, device="cuda")
    assert _call_first(gy, y, x, ws, gb, gw) == 0, _err()
    torch.cuda.synchronize()
    ref_gw, ref_gb = ref_backward_first(gy, y, x)                   # unrounded products of the stored inputs, as the kernel sums them
    # per term: o = g (1 - t t) off by <= 3 u |g| (test_bias_tanh_backward_random), o x by 3 u |g x|; additions: 2 per lane trip (the fma
    # rounds once per term, +1), RL partials, one per block in the reduce kernel: |d| <= chain u sum |terms| + 3 u sum |g| (|x|)
    _, RL = lanes(h)
    s = bwd_stride(h, n)
    chain = 2 * -(-n // s) + RL + s // RL + 1
    gz, ga, xa = gy.double() * (1 - y.double() ** 2), gy.double().abs(), x.double().abs()
    lim_b = chain * U * gz.abs().sum(0) + 3 * U * ga.sum(0)
    lim_w = chain * U * (gz.abs().t() @ xa) + 3 * U * (ga.t() @ xa)
    e_b, e_w = (gb.double() - ref_gb).abs(), (gw.double() - ref_gw).abs()
    assert bool((e_b <= lim_b).all()) and bool((e_w <= lim_w).all()), (float((e_b / lim_b).max()), float((e_w / lim_w).max()))
    print(f"\n[bias_tanh_backward_first w_kernel-IN{k}-h{h}-n{n} {dt} random] max |d gb| {float(e_b.max()):.2e} |d gw| {float(e_w.max()):.2e}")


# ---- qp_bias_tanh_mean / qp_bias_tanh_mean_backward --------------------------------------------------------------------------------
def _call_mean(z, b, V, y, m, s=None):
    return _lib().qp_bias_tanh_mean(z.data_ptr(), b.data_ptr(), z.shape[0] // V, V, z.shape[1], int(z.dtype == torch.bfloat16), y.data_ptr(),
                                    m.data_ptr(), _stream(s))


def _call_mean_bwd(gm, y, V, gz, gb, s=None):
    return _lib().qp_bias_tanh_mean_backward(gm.data_ptr(), y.data_ptr(), gm.shape[0], V, y.shape[1], int(y.dtype == torch.bfloat16),
                                             gz.data_ptr(), gb.data_ptr(), _stream(s))


def _mean_id(c):
    V, h, groups = c
    return f"mean-V{V}-h{h}-g{groups}-" + ("loop" if groups > 5 else "tail")


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("case", MEAN_CASES, ids=_mean_id)
def test_bias_tanh_mean(case, dt):
    V, h, groups = case
    rows = groups * V
    g = torch.Generator().manual_seed(V * 1009 + h + groups)
    z = (1.5 * torch.randn(rows, h, generator=g)).to("cuda", TD[dt])
    b = (torch.rand(h, generator=g) * 2 - 1).cuda()
    y = torch.full_like(z, float("nan"))
    m = torch.full((groups, h), float("nan"), dtype=TD[dt], device="cuda")
    assert _call_mean(z, b, V, y, m) == 0, _err()
    torch.cuda.synchronize()
    ref_y = ref_bias_tanh(z, b)
    ref_m = ref_mean(y, V)                                          # the kernel averages y as stored (bf16-rounded under autocast)
    if dt == "fp32":
        e_y = float((y.double() - ref_y).abs().max())
        assert e_y <= 1.3e-6                                         # as test_bias_tanh_forward
        # the j-th fp32 partial sum is below j (|y| < 1): the V - 1 additions err by < u V^2 / 2, u V / 2 after the division; the rounded
        # 1 / V and the product add u |mean| each: |d| <= (V / 2 + 2) u
        e_m = float((m.double() - ref_m).abs().max())
        assert e_m <= (V / 2 + 2) * U
    else:
        e_y = _close_bf16(y, ref_y, 1, "y")
        # the fp32 mean (error above, absolute: it matters for a mean near 0) is rounded once to bf16; with 1 / V inexact (V = 3, 7, 31)
        # allow 2 ulp
        e_m = _close_bf16(m, ref_m, 1 if V & (V - 1) == 0 else 2, "mean", atol=(V / 2 + 2) * U)
    print(f"\n[bias_tanh_mean {_mean_id(case)} {dt}] max |d y| {e_y:.2e}, max |d mean| {e_m:.2e}")


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("case", MEAN_CASES, ids=_mean_id)
def test_bias_tanh_mean_backward(case, dt):
    """Exact arithmetic for V = 1, 2 (grad_z a multiple of 1/32); random values with a tolerance for V = 3, 7, 31 (1 / V inexact)."""
    V, h, groups = case
    rows = groups * V
    g = torch.Generator().manual_seed(V * 7 + h * 13 + groups)
    exact = V in (1, 2)
    if exact:
        yv, gmv = exact_y((rows, h), g), exact_int((groups, h), g)
        assert_exact_bound((gmv.repeat_interleave(V, 0) / V * (1 - yv ** 2)).abs().sum(0), 1 / 32)
    else:
        yv, gmv = torch.tanh(torch.randn(rows, h, generator=g)), torch.randn(groups, h, generator=g)
    y, gm = yv.to("cuda", TD[dt]), gmv.to("cuda", TD[dt])
    gz = torch.full_like(y, 1e30)
    gb = torch.full((h,), 1e30, device="cuda")
    ref_gz, ref_gb = ref_mean_backward(gm, y, V)
    assert _call_mean_bwd(gm, y, V, gz, gb) == 0, _err()
    torch.cuda.synchronize()
    if exact:
        assert torch.equal(gz.double(), ref_gz), float((gz.double() - ref_gz).abs().max())
        assert torch.equal(gb.double(), ref_gb), float((gb.double() - ref_gb).abs().max())
        print(f"\n[bias_tanh_mean_backward {_mean_id(case)} {dt}] exact")
        return
    # o = fl(gm fl(1/V)) (1 - t t): 1 / V, the product with gm, t t, 1 - t t and the last product round once each: |d| <= 5 u |gm| / V
    if dt == "fp32":
        lim = 5 * U * gm.double().abs().repeat_interleave(V, 0) / V
        e_gz = float((gz.double() - ref_gz).abs().max())
        assert bool(((gz.double() - ref_gz).abs() <= lim + 1e-30).all())
    else:
        e_gz = _close_bf16(gz, ref_gz, 2, "grad_z")
    # grad_bias: the 5 u |gm| / V per term (above), V additions per group within a lane, RL partials, one atomic per block
    _, RL = lanes(h)
    s = bwd_stride(h, groups)
    chain = V * -(-groups // s) + RL + s // RL
    e_gb = (gb.double() - ref_gb).abs()
    lim_b = chain * U * ref_gz.abs().sum(0) + 5 * U * gm.double().abs().sum(0)
    assert bool((e_gb <= lim_b).all()), float((e_gb / lim_b).max())
    print(f"\n[bias_tanh_mean_backward {_mean_id(case)} {dt} random] max |d grad_z| {e_gz:.2e}, max |d grad_bias| {float(e_gb.max()):.2e}")


# ---- qp_gae -----------------------------------------------------------------------------------------------------------------------
def _call_gae(rew, val, d8, last, gamma, lam, adv, ret, s=None):
    T, n = rew.shape
    return _lib().qp_gae(rew.data_ptr(), val.data_ptr(), d8.data_ptr(), last.data_ptr(), T, n, gamma, lam, adv.data_ptr(), ret.data_ptr(),
                         _stream(s))


def _gae_inputs(T, n, pattern, g, exact):
    if exact:
        rew, val, last = exact_int((T, n), g, -4, 4), exact_int((T, n), g, -4, 4), exact_int((n,), g, -4, 4)
    else:
        rew, val, last = torch.randn(T, n, generator=g), torch.randn(T, n, generator=g), torch.randn(n, generator=g)
    d = done_pattern(pattern, T, n, g)
    return rew.float().cuda(), val.float().cuda(), d.to(torch.uint8).cuda(), last.float().cuda()


@gpu
@pytest.mark.parametrize("pattern", DONE_PATTERNS)
@pytest.mark.parametrize("shape", GAE_SHAPES, ids=lambda s: f"T{s[0]}-n{s[1]}")
def test_gae_exact(shape, pattern):
    """gamma = lam = 1, integer rewards and values in [-4, 4]: |delta| <= 12, |A| <= 12 T < 2^14, every fp32 step exact."""
    T, n = shape
    g = torch.Generator().manual_seed(T * 3 + n)
    rew, val, d8, last = _gae_inputs(T, n, pattern, g, exact=True)
    adv, ret = torch.full_like(rew, float("nan")), torch.full_like(rew, float("nan"))
    assert _call_gae(rew, val, d8, last, 1.0, 1.0, adv, ret) == 0, _err()
    torch.cuda.synchronize()
    ref_adv, ref_ret = ref_gae(rew, val, d8.bool(), last, 1.0, 1.0)
    assert float(ref_adv.abs().max()) < 2 ** 14
    assert torch.equal(adv.double(), ref_adv) and torch.equal(ret.double(), ref_ret), float((adv.double() - ref_adv).abs().max())
    print(f"\n[gae T{T}-n{n} {pattern}] exact")


@gpu
@pytest.mark.parametrize("shape", [(1, 257), (128, 256), (128, 65537)], ids=lambda s: f"T{s[0]}-n{s[1]}")
def test_gae_gamma_zero(shape):
    """gamma = 0: A_t = r_t - V_t (one rounding, exact for integers), whatever lam and the done flags."""
    T, n = shape
    g = torch.Generator().manual_seed(n)
    rew, val, d8, last = _gae_inputs(T, n, "random", g, exact=True)
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    assert _call_gae(rew, val, d8, last, 0.0, 0.95, adv, ret) == 0, _err()
    torch.cuda.synchronize()
    assert torch.equal(adv, rew - val) and torch.equal(ret, rew)


@gpu
@pytest.mark.parametrize("pattern", ["none", "random", "last"])
@pytest.mark.parametrize("shape", [(2, 255), (128, 257), (1024, 256)], ids=lambda s: f"T{s[0]}-n{s[1]}")
def test_gae_random(shape, pattern):
    T, n = shape
    g = torch.Generator().manual_seed(T + n)
    rew, val, d8, last = _gae_inputs(T, n, pattern, g, exact=False)
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    assert _call_gae(rew, val, d8, last, 0.99, 0.95, adv, ret) == 0, _err()
    torch.cuda.synchronize()
    gamma, lam = float(np.float32(0.99)), float(np.float32(0.95))     # what the C-ABI receives
    ref_adv, ref_ret = ref_gae(rew, val, d8.bool(), last, gamma, lam)
    # each step rounds <= 5 times at magnitudes <= M = max |A| + max |r| + 2 max |V|, and the recursion damps an earlier error by c = gamma
    # lam = 0.9405: 5 u M / (1 - c); the rounded coefficient c (u) perturbs the term of lag j by j u: u M c / (1 - c)^2.  Together < 350 u M
    M = float(ref_adv.abs().max()) + float(rew.abs().max()) + 2 * float(val.abs().max())
    e = max(float((adv.double() - ref_adv).abs().max()), float((ret.double() - ref_ret).abs().max()))
    assert e <= 350 * U * M
    print(f"\n[gae T{T}-n{n} {pattern} gamma 0.99 lam 0.95] max |d| {e:.2e} (M {M:.1f})")


# ---- properties: repeated calls, non-default streams ------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_backward_calls_are_repeatable(dt):
    """The backward entry points zero grad_bias themselves: two calls into the same buffers, pre-filled with garbage, agree bit for bit
    and with the reference.  Exact-arithmetic inputs: with random values the fp32 atomics of the blocks may add up in another order."""
    h, n, V = 256, loop_n(256, trips=2), 2
    g = torch.Generator().manual_seed(99)
    y = exact_y((n * V, h), g).to("cuda", TD[dt])
    gy = exact_int((n * V, h), g).to("cuda", TD[dt])
    for name, call, ref, outs in (
            ("bias_tanh_backward", lambda gz, gb: _call_bwd(gy, y, gz, gb), ref_bias_tanh_backward(gy, y),
             (torch.empty_like(y), torch.empty(h, device="cuda"))),
            ("bias_tanh_mean_backward", lambda gz, gb: _call_mean_bwd(gy[:n], y, V, gz, gb), ref_mean_backward(gy[:n], y, V),
             (torch.empty_like(y), torch.empty(h, device="cuda")))):
        res = []
        for fill in (float("nan"), -3e38):
            for t in outs:
                t.fill_(fill)
            assert call(*outs) == 0, _err()
            torch.cuda.synchronize()
            res.append([t.clone() for t in outs])
        assert all(torch.equal(a, b) for a, b in zip(*res)), name
        assert all(torch.equal(a.double(), r) for a, r in zip(res[0], ref)), name


def _side_stream_case(name, dt):
    """(launch(stream) -> rc, check() -> max error) for one entry point, inputs made on the current stream."""
    g = torch.Generator().manual_seed(3)
    h, n, V = 48, 5000, 3
    z = torch.randn(n, h, generator=g).to("cuda", TD[dt])
    b = torch.rand(h, generator=g).cuda()
    y = torch.tanh(torch.randn(n, h, generator=g)).to("cuda", TD[dt])
    out = torch.full_like(z, float("nan"))
    gb = torch.full((h,), float("nan"), device="cuda")
    if name == "bias_tanh":
        return (lambda s: _call_fwd(z, b, out, s)), (lambda: float((out.double() - ref_bias_tanh(z, b)).abs().max()))
    if name == "bias_tanh_backward":
        return (lambda s: _call_bwd(z, y, out, gb, s)), (lambda: float((gb.double() - ref_bias_tanh_backward(z, y)[1]).abs().max()))
    if name == "bias_tanh_backward_first":
        x = torch.randn(n, 6, generator=g).cuda()
        ws, _ = _workspace(h, 6)
        gw = torch.full((h, 6), float("nan"), device="cuda")
        return (lambda s: _call_first(z, y, x, ws, gb, gw, s)), (lambda: float((gw.double() - ref_backward_first(z, y, x)[0]).abs().max()))
    m = torch.full((n // V, h), float("nan"), dtype=TD[dt], device="cuda")
    if name == "bias_tanh_mean":
        zz, yy = z[:n // V * V], out[:n // V * V]
        return (lambda s: _call_mean(zz, b, V, yy, m, s)), (lambda: float((m.double() - ref_mean(yy, V)).abs().max()))
    if name == "bias_tanh_mean_backward":
        yy, gz = y[:n // V * V], out[:n // V * V]
        gm = z[:n // V]
        return (lambda s: _call_mean_bwd(gm, yy, V, gz, gb, s)), (lambda: float((gb.double() - ref_mean_backward(gm, yy, V)[1]).abs().max()))
    rew, val, d8, last = _gae_inputs(64, 1000, "random", g, exact=False)
    adv, ret = torch.full_like(rew, float("nan")), torch.full_like(rew, float("nan"))
    return (lambda s: _call_gae(rew, val, d8, last, 0.99, 0.95, adv, ret, s)), \
        (lambda: float((adv.double() - ref_gae(rew, val, d8.bool(), last, 0.99, 0.95)[0]).abs().max()))


@gpu
@pytest.mark.parametrize("name", ["bias_tanh", "bias_tanh_backward", "bias_tanh_backward_first", "bias_tanh_mean", "bias_tanh_mean_backward", "gae"])
def test_entry_points_run_on_the_given_stream(name):
    """Launched on a non-default stream and read after synchronising that stream only."""
    dt = "bf16" if name != "gae" else "fp32"
    launch, check = _side_stream_case(name, dt)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        assert launch(s) == 0, _err()
    s.synchronize()
    with torch.cuda.stream(s):
        e = check()
    assert e <= 0.05, e                                             # loose: this checks where the work ran; the tables check how well
    print(f"\n[{name} on a side stream] max |d| {e:.2e}")


# ---- error paths -------------------------------------------------------------------------------------------------------------------
SENTINEL = 7.0


def _rejected(call, rc, words, outs):
    """The call returns `rc`, names `words` in qp_last_error(NULL) and launches nothing: every output keeps its sentinel."""
    for t in outs:
        t.fill_(SENTINEL)
    torch.cuda.synchronize()
    got = call()
    torch.cuda.synchronize()
    msg = _err()
    assert got == rc, (got, msg)
    for w in words:
        assert w in msg, (w, msg)
    for t in outs:
        assert bool((t == SENTINEL).all()), msg


@gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_bias_tanh_rejects_bad_calls(dt):
    lib, s, bf = _lib(), _stream(), int(dt == "bf16")
    n, h = 64, 256
    z, y = torch.zeros(n, h, dtype=TD[dt], device="cuda"), torch.zeros(n, h, dtype=TD[dt], device="cuda")
    b, gb = torch.zeros(h, device="cuda"), torch.zeros(h, device="cuda")
    fwd = lambda zp, nn, hh, yp: (lambda: lib.qp_bias_tanh(zp, b.data_ptr(), nn, hh, bf, yp, s))
    bwd = lambda gp, yp, nn, hh, gzp, gbp: (lambda: lib.qp_bias_tanh_backward(gp, yp, nn, hh, bf, gzp, gbp, s))
    _rejected(fwd(None, n, h, y.data_ptr()), -1, ["null"], [y])
    _rejected(fwd(z.data_ptr(), n, h, None), -1, ["null"], [])
    _rejected(bwd(z.data_ptr(), z.data_ptr(), n, h, y.data_ptr(), None), -1, ["null"], [y])
    for nn, hh in ((0, h), (n, 7), (n, 0), (n, 2050)):
        _rejected(fwd(z.data_ptr(), nn, hh, y.data_ptr()), -2, ["h must be even", "n >= 1"], [y])
        _rejected(bwd(z.data_ptr(), z.data_ptr(), nn, hh, y.data_ptr(), gb.data_ptr()), -2, ["h must be even", "n >= 1"], [y, gb])
    # one element off: not even pair-aligned (the pair kernels would make a misaligned float2 / bf16x2 access)
    zo, yo = _view(n, h, TD[dt], 1), _view(n, h, TD[dt], 1)
    _rejected(fwd(zo.data_ptr(), n, h, y.data_ptr()), -2, ["aligned"], [y])
    _rejected(fwd(z.data_ptr(), n, h, yo.data_ptr()), -2, ["aligned"], [yo])
    _rejected(bwd(zo.data_ptr(), z.data_ptr(), n, h, y.data_ptr(), gb.data_ptr()), -2, ["aligned"], [y, gb])
    _rejected(bwd(z.data_ptr(), zo.data_ptr(), n, h, y.data_ptr(), gb.data_ptr()), -2, ["aligned"], [y, gb])
    _rejected(bwd(z.data_ptr(), z.data_ptr(), n, h, yo.data_ptr(), gb.data_ptr()), -2, ["aligned"], [yo, gb])


@gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_bias_tanh_backward_first_rejects_bad_calls(dt):
    lib, s, bf = _lib(), _stream(), int(dt == "bf16")
    n, h, k = 64, 256, 6
    y = torch.zeros(n + 1, h, dtype=TD[dt], device="cuda")
    x = torch.zeros(n, k, device="cuda")
    ws = torch.zeros(int(lib.qp_bias_tanh_backward_first_workspace(h, 8)) // 4, device="cuda")
    gb, gw = torch.zeros(h, device="cuda"), torch.zeros(h, 8, device="cuda")
    call = lambda gp, yp, nn, hh, kk, wsp: (lambda: lib.qp_bias_tanh_backward_first(gp, yp, x.data_ptr(), nn, hh, kk, bf, wsp, gb.data_ptr(),
                                                                                    gw.data_ptr(), s))
    yp = y.data_ptr()
    _rejected(call(yp, yp, n, h, k, None), -1, ["null"], [gb, gw, ws])
    _rejected(call(None, yp, n, h, k, ws.data_ptr()), -1, ["null"], [gb, gw, ws])
    for nn, hh, kk in ((0, h, k), (n, 12, k), (n, 250, k), (n, 7, k), (n, 0, k), (n, 2050, k), (n, h, 0), (n, h, 9)):
        _rejected(call(yp, yp, nn, hh, kk, ws.data_ptr()), -2, ["multiple of 8", "in_dim"], [gb, gw, ws])
    off = y.view(-1)[8 // y.element_size():].data_ptr()            # 8 bytes in: pair-aligned, not 16-byte aligned
    _rejected(call(off, yp, n, h, k, ws.data_ptr()), -2, ["16-byte"], [gb, gw, ws])
    _rejected(call(yp, off, n, h, k, ws.data_ptr()), -2, ["16-byte"], [gb, gw, ws])


@gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_bias_tanh_mean_rejects_bad_calls(dt):
    lib, s, bf = _lib(), _stream(), int(dt == "bf16")
    n, V, h = 16, 3, 256
    z = torch.zeros(n * V + 1, h, dtype=TD[dt], device="cuda")
    y, m = torch.zeros(n * V, h, dtype=TD[dt], device="cuda"), torch.zeros(n, h, dtype=TD[dt], device="cuda")
    b, gb = torch.zeros(h, device="cuda"), torch.zeros(h, device="cuda")
    fwd = lambda zp, nn, VV, hh: (lambda: lib.qp_bias_tanh_mean(zp, b.data_ptr(), nn, VV, hh, bf, y.data_ptr(), m.data_ptr(), s))
    bwd = lambda gp, nn, VV, hh: (lambda: lib.qp_bias_tanh_mean_backward(gp, z.data_ptr(), nn, VV, hh, bf, y.data_ptr(), gb.data_ptr(), s))
    zp = z.data_ptr()
    _rejected(fwd(None, n, V, h), -1, ["null"], [y, m])
    _rejected(bwd(None, n, V, h), -1, ["null"], [y, gb])
    for nn, VV, hh in ((0, V, h), (n, 0, h), (n, V, 12), (n, V, 7), (n, V, 0), (n, V, 2050)):
        _rejected(fwd(zp, nn, VV, hh), -2, ["n >= 1", "V >= 1", "multiple of 8"], [y, m])
        _rejected(bwd(zp, nn, VV, hh), -2, ["n >= 1", "V >= 1", "multiple of 8"], [y, gb])
    off = z.view(-1)[8 // z.element_size():].data_ptr()
    _rejected(fwd(off, n, V, h), -2, ["16-byte"], [y, m])
    _rejected(bwd(off, n, V, h), -2, ["16-byte"], [y, gb])


@gpu
def test_gae_rejects_bad_calls():
    lib, s = _lib(), _stream()
    T, n = 8, 300
    r = torch.zeros(T, n, device="cuda")
    d8 = torch.zeros(T, n, dtype=torch.uint8, device="cuda")
    adv, ret = torch.zeros(T, n, device="cuda"), torch.zeros(T, n, device="cuda")
    call = lambda rp, TT, nn, retp: (lambda: lib.qp_gae(rp, r.data_ptr(), d8.data_ptr(), r.data_ptr(), TT, nn, 0.99, 0.95, adv.data_ptr(), retp, s))
    _rejected(call(None, T, n, ret.data_ptr()), -1, ["null"], [adv, ret])
    _rejected(call(r.data_ptr(), T, n, None), -1, ["null"], [adv])
    for TT, nn in ((0, n), (-1, n), (T, 0)):
        _rejected(call(r.data_ptr(), TT, nn, ret.data_ptr()), -2, ["T / n"], [adv, ret])


# ---- the fused_policy wrappers -------------------------------------------------------------------------------------------------------
@gpu
def test_wrappers_match_the_references():
    from quad_swarm_rl_stable_baselines3_b200 import fused_policy as fp
    g = torch.Generator().manual_seed(17)
    h, n, V, k = 256, 4100, 3, 6
    z = torch.randn(n * V, h, generator=g).cuda()
    b = torch.rand(h, generator=g).cuda() - 0.5
    assert float((fp.bias_tanh(z, b).double() - ref_bias_tanh(z, b)).abs().max()) <= 1.3e-6
    y, m = fp.bias_tanh_mean(z, b, V)
    assert float((m.double() - ref_mean(y, V)).abs().max()) <= (V / 2 + 2) * U
    yv, gv, xv = exact_y((n * V, h), g), exact_int((n * V, h), g), exact_int((n * V, k), g)
    ye, ge = yv.to("cuda", torch.bfloat16), gv.to("cuda", torch.bfloat16)
    gz, gb = fp.bias_tanh_backward(ge, ye)
    rgz, rgb = ref_bias_tanh_backward(ge, ye)
    assert torch.equal(gz.double(), rgz) and torch.equal(gb.double(), rgb)
    gw, gb = fp.bias_tanh_backward_first(ge, ye, xv.cuda())
    rgw, rgb = ref_backward_first(ge, ye, xv.cuda())
    assert torch.equal(gw.double(), rgw) and torch.equal(gb.double(), rgb)
    gm = exact_int((n * V // 2, h), g).to("cuda", torch.bfloat16)
    gz, gb = fp.bias_tanh_mean_backward(gm, ye, 2)
    rgz, rgb = ref_mean_backward(gm, ye, 2)
    assert torch.equal(gz.double(), rgz) and torch.equal(gb.double(), rgb)
    rew, val, d8, last = _gae_inputs(256, 1000, "random", g, exact=True)
    adv, ret = fp.gae(rew, val, d8.bool(), last, 1.0, 1.0)
    radv, rret = ref_gae(rew, val, d8.bool(), last, 1.0, 1.0)
    assert torch.equal(adv.double(), radv) and torch.equal(ret.double(), rret)


@gpu
def test_mean_wrappers_reject_ragged_rows():
    """rows % V != 0 used to leave the last rows of y / grad_z as uninitialised memory."""
    from quad_swarm_rl_stable_baselines3_b200 import fused_policy as fp
    z = torch.randn(3 * 5 + 2, 64, device="cuda")
    with pytest.raises(ValueError, match="groups"):
        fp.bias_tanh_mean(z, torch.zeros(64, device="cuda"), 3)
    with pytest.raises(ValueError, match="groups"):
        fp.bias_tanh_mean_backward(torch.randn(5, 64, device="cuda"), torch.tanh(z), 3)
    with pytest.raises(ValueError, match="grad_mean"):
        fp.bias_tanh_mean_backward(torch.randn(4, 64, device="cuda"), torch.tanh(z[:15]), 3)


@gpu
def test_gae_wrapper_rejects_wrong_dtypes_and_shapes():
    """float64 rewards used to be read as float32 memory, float dones as four bytes per flag."""
    from quad_swarm_rl_stable_baselines3_b200 import fused_policy as fp
    T, n = 16, 100
    r, v = torch.randn(T, n, device="cuda"), torch.randn(T, n, device="cuda")
    d, last = torch.zeros(T, n, dtype=torch.bool, device="cuda"), torch.randn(n, device="cuda")
    bad = [
        (r.double(), v, d, last, "rewards"),
        (r, v.half(), d, last, "values"),
        (r, v, d.float(), last, "dones"),
        (r, v, d[:, :50], last, "dones"),
        (r, v[:8], d, last, "values"),
        (r, v, d, last[:50], "last_values"),
        (r.reshape(-1), v, d, last, "rewards"),
    ]
    for args in bad:
        with pytest.raises(ValueError, match=args[-1]):
            fp.gae(*args[:-1], 0.99, 0.95)
    fp.gae(r, v, d.to(torch.uint8), last, 0.99, 0.95)                  # uint8 dones are accepted
