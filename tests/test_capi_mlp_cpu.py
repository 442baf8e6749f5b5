"""CPU-side checks of the MLP neighbour encoder's C-ABI (include/quadpolicy.h): qp_create_encoder is exported, the ctypes mirrors
follow the header (encoder kinds, the qp_tower_weights field order with nbr_w3 / nbr_b3 appended), and the configurations the kernel
does not build are rejected before any device is touched."""
import ctypes as C
import os
import re

import pytest

from quad_swarm_rl_stable_baselines3_b200 import _capi
from quad_swarm_rl_stable_baselines3_b200.fused_policy import QP_API_VERSION, QP_NBR, QpConfigC, QpTowerWeightsC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "quadpolicy.h")).read()


@pytest.fixture(scope="module")
def lib():
    _capi.build()
    return _capi.lib()


def test_create_encoder_exported(lib):
    assert "qp_create_encoder" in _capi.POLICY_EXPORTS and hasattr(lib, "qp_create_encoder")
    assert re.search(r"\bint qp_create_encoder\(const qp_config \*cfg, int nbr_encoder, int device, qp_policy \*\*out\);", HEADER)


def test_encoder_kinds_match_the_header():
    kinds = dict((k, int(v)) for k, v in re.findall(r"\b(QP_NBR_[A-Z]+) = (\d+)", HEADER))
    assert kinds == {"QP_NBR_DEEPSETS": 0, "QP_NBR_MLP": 1}
    assert QP_NBR == {"mean_embed": 0, "none": 0, "mlp": 1}


def test_tower_weights_mirror_the_header():
    body = re.search(r"typedef struct \{(.*?)\} qp_tower_weights;", HEADER, re.S).group(1)
    fields = re.findall(r"\*(\w+)", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    assert tuple(fields) == QpTowerWeightsC.FIELDS
    assert fields[-2:] == ["nbr_w3", "nbr_b3"] and C.sizeof(QpTowerWeightsC) == 18 * C.sizeof(C.c_void_p)


@pytest.mark.parametrize("cfg,kind,msg", [
    ((18, 6, 7, 256, 4, 0), 1, b"<= 40"),           # W * V = 42
    ((19, 6, 2, 256, 4, 9), 1, b"obst_dim"),        # with the obstacle encoder
    ((18, 6, 0, 256, 4, 0), 1, b"num_nbr"),         # no neighbours
    ((18, 6, 6, 256, 4, 0), 2, b"nbr_encoder"),     # unknown kind
    ((18, 6, 6, 256, 4, 0), -1, b"nbr_encoder"),
])
def test_unbuilt_mlp_configs_rejected(lib, cfg, kind, msg):
    h = C.c_void_p()
    assert lib.qp_create_encoder(C.byref(QpConfigC(QP_API_VERSION, *cfg)), kind, 0, C.byref(h)) == -2 and not h.value
    assert msg in lib.qp_last_error(None), lib.qp_last_error(None)


def test_create_encoder_without_gpu_fails_loudly(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = C.c_void_p()
    assert lib.qp_create_encoder(C.byref(QpConfigC(QP_API_VERSION, 18, 8, 5, 256, 4, 0)), 1, 0, C.byref(h)) < 0 and not h.value
    assert b"CUDA" in lib.qp_last_error(None)
