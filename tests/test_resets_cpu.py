"""CPU tests of the per-robot reset entry points (go2p_step_batch_ex, go2p_step_batch_host_ex, go2p_fleet_step_host_ex):
they are exported, refuse a null handle or fleet, and the Python layer validates a host reset mask before any call.
Everything that needs a handle -- the resets themselves -- is tested on the GPU (test_gpu_resets.py)."""
import numpy as np
import pytest

from go2_onnx_controller_b200 import actor, build, capi


@pytest.fixture(scope="module")
def lib():
    build.build()
    return capi.load()


def test_reset_entry_points_are_declared_and_exported(lib):
    for name in ("go2p_step_batch_ex", "go2p_step_batch_host_ex", "go2p_fleet_step_host_ex"):
        assert name in capi.SIGNATURES and hasattr(lib, name), name
    assert lib.go2p_abi_version() == 2                 # additive change: the ABI version stays


def test_null_handle_or_fleet_is_invalid(lib):
    raw = np.zeros((4, 156), np.uint8)
    act = np.zeros((4, 12), np.float32)
    mask = np.ones(4, np.uint8)
    # device form: every pointer argument non-null except the handle
    assert lib.go2p_step_batch_ex(None, raw.ctypes.data, mask.ctypes.data, act.ctypes.data, act.ctypes.data,
                                  act.ctypes.data, act.ctypes.data, None, 4, capi.PREC_FP16, None) == capi.ERR_INVALID
    assert lib.go2p_step_batch_host_ex(None, raw.ctypes.data, mask.ctypes.data, act.ctypes.data, None, 4,
                                       capi.PREC_FP16) == capi.ERR_INVALID
    assert lib.go2p_fleet_step_host_ex(None, raw.ctypes.data, mask.ctypes.data, act.ctypes.data, None, 4,
                                       capi.PREC_FP16) == capi.ERR_INVALID
    assert lib.go2p_last_error()                        # with a message


@pytest.mark.parametrize("mask", [np.zeros(5, np.bool_), np.arange(5, dtype=np.uint8)])
def test_host_reset_mask_accepts_bool_and_uint8(mask):
    assert actor.host_reset_mask(mask, 5) is mask


@pytest.mark.parametrize("mask,exc", [
    (np.zeros(5, np.int32), TypeError),                 # another dtype
    (np.zeros(5, np.float32), TypeError),
    ([0, 1, 0, 0, 1], TypeError),                       # not a numpy array
    (np.zeros(4, np.uint8), ValueError),                # another length
    (np.zeros((5, 1), np.bool_), ValueError),           # another shape
    (np.zeros(10, np.uint8)[::2], ValueError),          # strided: not one byte per robot
])
def test_host_reset_mask_rejects_other_arrays(mask, exc):
    with pytest.raises(exc):
        actor.host_reset_mask(mask, 5)
