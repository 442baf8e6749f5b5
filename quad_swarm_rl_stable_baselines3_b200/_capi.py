"""ctypes binding of libquadsim_b200.so (include/quadsim.h).  No CPU fallback: if the CUDA library is missing or
cannot be loaded, importing the simulator fails loudly."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from .config import QsConfigC, QsStateViewC, QsStatsC

_PKG = os.path.dirname(os.path.abspath(__file__))
# QS_LIB_PATH: load another build of the same sources (tuning sweeps under build/variants/); default is the in-tree library
LIB_PATH = os.environ.get("QS_LIB_PATH") or os.path.join(_PKG, "libquadsim_b200.so")
CSRC = os.path.join(_PKG, "csrc")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              # approximate (2 ulp) fp32 division / square root: the parity budget is 1e-5 relative; threshold tests that
              # must match the oracle "away from ties" use __fsqrt_rn explicitly.  Denormals are NOT flushed.
              "-prec-div=false", "-prec-sqrt=false",
              "-Xcompiler", "-fPIC", "-shared"]

# every symbol include/quadsim.h declares
EXPORTS = ("qs_config_size", "qs_stats_size", "qs_api_version", "qs_last_error", "qs_create", "qs_destroy",
           "qs_num_envs", "qs_num_agents", "qs_obs_dim", "qs_act_dim", "qs_launch_count", "qs_reset", "qs_step",
           "qs_reset_host", "qs_step_host", "qs_get_state", "qs_set_state", "qs_set_param", "qs_episode_stats",
           "qs_episode_records", "qs_episode_records_host", "qs_set_reward_info", "qs_snapshot_size", "qs_snapshot", "qs_restore",
           "qs_restore_shards")
# every symbol include/quadpolicy.h declares (fused policy forward, csrc/policy_kernels.cu)
POLICY_EXPORTS = ("qp_config_size", "qp_last_error", "qp_create", "qp_create_encoder", "qp_destroy", "qp_launch_count", "qp_set_weights", "qp_forward", "qp_gae", "qp_bias_tanh", "qp_bias_tanh_backward", "qp_bias_tanh_mean", "qp_bias_tanh_mean_backward", "qp_bias_tanh_backward_first", "qp_bias_tanh_backward_first_workspace")


KG_VALUES = (1, 2, 4, 8, 16, 32)


def build(force: bool = False, verbose: bool = False, out: str | None = None, defines=()) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU).  One translation unit per
    lane-group width (kernels_kg.cu, -DQS_KG=n) plus the host API (quadsim.cu), compiled in parallel, then linked."""
    from concurrent.futures import ThreadPoolExecutor
    root = os.path.dirname(_PKG)
    deps = [os.path.join(CSRC, f) for f in ("quadsim.cu", "kernels_kg.cu", "quadsim_kernels.cuh", "fork_kernels.cuh", "scenario_kernels.cuh", "launch.h",
                                            "policy_kernels.cu")]
    deps.append(os.path.join(root, "include", "quadsim.h"))
    deps.append(os.path.join(root, "include", "quadpolicy.h"))
    if not force and out is None and os.path.exists(LIB_PATH) and all(
            (not os.path.exists(d)) or os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    target = out or LIB_PATH
    if os.path.exists(target):
        os.remove(target)          # a failed rebuild must not leave a stale library behind
    nvcc = os.environ.get("NVCC", "nvcc")
    objdir = os.path.join(root, "build", "obj" if out is None else "obj_" + os.path.basename(out))
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + [f"-D{d}" for d in defines] + (["-Xptxas", "-v"] if verbose else [])
    jobs = [([nvcc] + flags + ["-c", os.path.join(CSRC, "quadsim.cu"), "-o", os.path.join(objdir, "quadsim.o")]),
            ([nvcc] + flags + ["-c", os.path.join(CSRC, "policy_kernels.cu"), "-o", os.path.join(objdir, "policy.o")])]
    for kg in KG_VALUES:
        jobs.append([nvcc] + flags + [f"-DQS_KG={kg}", "-c", os.path.join(CSRC, "kernels_kg.cu"), "-o", os.path.join(objdir, f"kernels_kg{kg}.o")])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            import sys
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise subprocess.CalledProcessError(r.returncode, cmd)

    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
        list(ex.map(run, jobs))
    objs = [j[-1] for j in jobs]
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", target] + objs)
    return target


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built (run `python -c 'import __graft_entry__ as g; "
            f"g.build()'` at the repo root).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, u8p, fp = C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.POINTER(C.c_float)
    L.qs_config_size.restype = C.c_size_t
    L.qs_stats_size.restype = C.c_size_t
    L.qs_api_version.restype = i32
    L.qs_last_error.restype = C.c_char_p
    L.qs_last_error.argtypes = [vp]
    L.qs_create.argtypes = [C.POINTER(QsConfigC), i32, C.POINTER(vp)]
    L.qs_destroy.argtypes = [vp]
    for n in ("qs_num_envs", "qs_num_agents", "qs_obs_dim", "qs_act_dim"):
        getattr(L, n).argtypes = [vp]
    L.qs_launch_count.argtypes = [vp]
    L.qs_launch_count.restype = C.c_int64
    L.qs_reset.argtypes = [vp, vp, vp, vp]
    L.qs_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.qs_reset_host.argtypes = [vp, vp, vp]
    L.qs_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.qs_get_state.argtypes = [vp, C.POINTER(QsStateViewC), vp]
    L.qs_set_state.argtypes = [vp, C.POINTER(QsStateViewC), vp]
    L.qs_set_param.argtypes = [vp, i32, C.c_double]
    L.qs_episode_stats.argtypes = [vp, C.POINTER(QsStatsC), i32, vp]
    L.qs_episode_records.argtypes = [vp, vp, vp, vp]
    L.qs_episode_records_host.argtypes = [vp, vp, vp, vp]
    L.qs_set_reward_info.argtypes = [vp, vp]
    L.qs_snapshot_size.argtypes = [vp]
    L.qs_snapshot_size.restype = C.c_size_t
    L.qs_snapshot.argtypes = [vp, vp, C.c_size_t, vp]
    L.qs_restore.argtypes = [vp, vp, C.c_size_t, vp]
    L.qs_restore_shards.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t), i32, vp]
    L.qs_philox_probe.argtypes = [C.c_uint32] * 6 + [C.POINTER(C.c_uint32), fp]
    # fused policy forward (include/quadpolicy.h)
    L.qp_config_size.restype = C.c_size_t
    L.qp_last_error.restype = C.c_char_p
    L.qp_last_error.argtypes = [vp]
    L.qp_create.argtypes = [vp, i32, C.POINTER(vp)]
    L.qp_create_encoder.argtypes = [vp, i32, i32, C.POINTER(vp)]
    L.qp_destroy.argtypes = [vp]
    L.qp_launch_count.argtypes = [vp]
    L.qp_launch_count.restype = C.c_int64
    L.qp_set_weights.argtypes = [vp, i32, vp, vp]
    L.qp_forward.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    L.qp_gae.argtypes = [vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, vp, vp, vp]
    L.qp_bias_tanh.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    L.qp_bias_tanh_backward.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp]
    L.qp_bias_tanh_backward_first.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]
    L.qp_bias_tanh_backward_first_workspace.argtypes = [i32, i32]
    L.qp_bias_tanh_backward_first_workspace.restype = C.c_size_t
    L.qp_bias_tanh_mean.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp]
    L.qp_bias_tanh_mean_backward.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp]
    if L.qs_config_size() != C.sizeof(QsConfigC) or L.qs_stats_size() != C.sizeof(QsStatsC):
        raise RuntimeError("qs_config / qs_stats layout mismatch between config.py and include/quadsim.h")
    _lib = L
    return L


def check(handle, rc: int, what: str):
    if rc != 0:
        msg = lib().qs_last_error(handle)
        raise RuntimeError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
