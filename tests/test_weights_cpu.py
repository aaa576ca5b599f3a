"""CPU tests of the weight-update entry points (go2p_set_weights, go2p_set_weights_host, go2p_fleet_set_weights_host):
they are declared, exported and bound, refuse a null handle or fleet, and the Python layer validates the tensors against
the policy's layer widths before any native call.  The updates themselves are tested on the GPU (test_gpu_weights.py)."""
import re

import numpy as np
import pytest

from go2_onnx_controller_b200 import actor, build, capi

NAMES = ("go2p_set_weights", "go2p_set_weights_host", "go2p_fleet_set_weights_host")
DIMS = [98, 128, 128, 128, 12]


@pytest.fixture(scope="module")
def lib():
    build.build()
    return capi.load()


def test_weight_entry_points_are_declared_exported_and_bound(lib):
    with open(build.ROOT + "/include/go2policy.h") as fh:
        hdr = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    for name in NAMES:
        assert re.search(r"\bint " + name + r"\(", hdr), name
        assert name in capi.SIGNATURES and hasattr(lib, name), name
    assert lib.go2p_abi_version() == 2                 # additive change: the ABI version stays


def test_null_handle_or_fleet_is_invalid(lib):
    w = [np.zeros((o, i), np.float32) for i, o in zip(DIMS[:-1], DIMS[1:])]
    ptrs = actor._ptr_array(w)
    assert lib.go2p_set_weights(None, ptrs, None, 4, None, None, None) == capi.ERR_INVALID
    assert b"null handle" in lib.go2p_last_error()
    assert lib.go2p_set_weights_host(None, ptrs, None, 4, None, None) == capi.ERR_INVALID
    assert b"null handle" in lib.go2p_last_error()
    assert lib.go2p_fleet_set_weights_host(None, ptrs, None, 4, None, None) == capi.ERR_INVALID
    assert b"null fleet" in lib.go2p_last_error()


def _net(dims=DIMS):
    rng = np.random.default_rng(0)
    w = [rng.standard_normal((o, i)).astype(np.float32) for i, o in zip(dims[:-1], dims[1:])]
    b = [rng.standard_normal(o).astype(np.float32) for o in dims[1:]]
    return w, b


def test_validator_accepts_host_arrays():
    w, b = _net()
    mean, std = np.zeros(98, np.float32), np.ones(98, np.float32)
    assert actor.weight_arrays(DIMS, w, b) == "host"
    assert actor.weight_arrays(DIMS, tuple(w), None, mean, std) == "host"
    assert actor.weight_arrays(DIMS, w, [None, b[1], None, b[3]]) == "host"     # a missing bias is zero


class FakeDevice:
    def __init__(self, type_, index):
        self.type, self.index = type_, index

    def __str__(self):
        return f"{self.type}:{self.index}"


class FakeTensor:
    """What the validator reads of a torch tensor (duck typing: the product does not import torch)."""
    def __init__(self, a, device=("cuda", 0), contiguous=True, dtype="torch.float32"):
        self.shape, self.dtype, self.device, self._c = a.shape, dtype, FakeDevice(*device), contiguous

    def data_ptr(self):
        return 0x1000

    def is_contiguous(self):
        return self._c


def test_validator_accepts_device_tensors():
    w, b = _net()
    assert actor.weight_arrays(DIMS, [FakeTensor(x) for x in w], [FakeTensor(x) for x in b], device=0) == "device"


def _bad_cases():
    w, b = _net()
    t = [FakeTensor(x) for x in w]
    mean = np.zeros(98, np.float32)
    return [
        ("not a list", dict(weights=w[0]), TypeError),
        ("too few layers", dict(weights=w[:3]), ValueError),
        ("too many layers", dict(weights=w + [w[-1]]), ValueError),
        ("bias count", dict(weights=w, biases=b[:2]), ValueError),
        ("biases not a list", dict(weights=w, biases=b[0]), TypeError),
        ("transposed weight", dict(weights=[w[0].T.copy()] + w[1:]), ValueError),
        ("bias shape", dict(weights=w, biases=[b[0][:-1]] + b[1:]), ValueError),
        ("float64", dict(weights=[w[0].astype(np.float64)] + w[1:]), TypeError),
        ("float16 bias", dict(weights=w, biases=[b[0].astype(np.float16)] + b[1:]), TypeError),
        ("not C-contiguous", dict(weights=[np.asfortranarray(w[0])] + w[1:]), ValueError),
        ("strided bias", dict(weights=w, biases=[np.zeros(256, np.float32)[::2]] + b[1:]), ValueError),
        ("a python list", dict(weights=[w[0].tolist()] + w[1:]), TypeError),
        ("mean without std", dict(weights=w, obs_mean=mean), ValueError),
        ("std without mean", dict(weights=w, obs_std=mean), ValueError),
        ("mean shape", dict(weights=w, obs_mean=mean[:-1], obs_std=mean[:-1]), ValueError),
        ("host and device mixed", dict(weights=[t[0]] + w[1:]), TypeError),
        ("device bias, host weights", dict(weights=w, biases=[FakeTensor(x) for x in b]), TypeError),
        ("device tensor on another GPU", dict(weights=[FakeTensor(w[0], ("cuda", 1))] + t[1:], device=0), ValueError),
        ("CPU tensor", dict(weights=[FakeTensor(w[0], ("cpu", None))] + t[1:]), TypeError),
        ("non-contiguous tensor", dict(weights=[FakeTensor(w[0], contiguous=False)] + t[1:]), ValueError),
        ("float64 tensor", dict(weights=[FakeTensor(w[0], dtype="torch.float64")] + t[1:]), TypeError),
    ]


@pytest.mark.parametrize("case", _bad_cases(), ids=lambda c: c[0])
def test_validator_rejects_bad_input(case):
    _, kw, exc = case
    with pytest.raises(exc):
        actor.weight_arrays(DIMS, **kw)
