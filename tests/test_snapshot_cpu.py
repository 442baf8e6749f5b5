"""CPU-side checks of the snapshot entry points (include/quadsim.h: qs_snapshot_size / qs_snapshot / qs_restore): the NULL-handle
contract and the ctypes signatures, which decide whether a 64-bit size and host pointers cross the boundary intact."""
import ctypes as C

import pytest

from quad_swarm_rl_stable_baselines3_b200 import _capi

QS_ERR_NULL = -4


@pytest.fixture(scope="module")
def lib():
    _capi.build()
    return _capi.lib()


def test_snapshot_size_of_null_handle_is_zero(lib):
    assert lib.qs_snapshot_size(None) == 0


def test_snapshot_and_restore_reject_null_handle(lib):
    buf = (C.c_uint8 * 64)()
    assert lib.qs_snapshot(None, C.cast(buf, C.c_void_p), 64, None) == QS_ERR_NULL
    assert lib.qs_restore(None, C.cast(buf, C.c_void_p), 64, None) == QS_ERR_NULL
    assert lib.qs_snapshot(None, None, 0, None) == QS_ERR_NULL
    assert lib.qs_restore(None, None, 0, None) == QS_ERR_NULL


def test_snapshot_signatures_declared(lib):
    vp, sz = C.c_void_p, C.c_size_t
    assert lib.qs_snapshot_size.argtypes == [vp] and lib.qs_snapshot_size.restype is sz
    assert lib.qs_snapshot.argtypes == [vp, vp, sz, vp] and lib.qs_snapshot.restype is C.c_int
    assert lib.qs_restore.argtypes == [vp, vp, sz, vp] and lib.qs_restore.restype is C.c_int
    assert {"qs_snapshot_size", "qs_snapshot", "qs_restore"} <= set(_capi.EXPORTS)
