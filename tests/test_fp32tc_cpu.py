"""CPU tests of GO2P_PREC_FP32_TC: the header, the ctypes mirror and the Python layer agree on the value, 3 stays the
rejected tf32 slot, the ABI version stays, and the entry points pass the new value through their argument checks.  The
precision itself is tested on the GPU (test_gpu_fp32tc.py)."""
import ctypes as C
import re

import numpy as np
import pytest

from go2_onnx_controller_b200 import Fleet, PolicyBatch, build, capi


@pytest.fixture(scope="module")
def lib():
    build.build()
    return capi.load()


def _enum(name):
    with open(build.ROOT + "/include/go2policy.h") as fh:
        hdr = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    body = re.search(r"typedef enum go2p_precision \{(.*?)\} go2p_precision;", hdr, flags=re.S).group(1)
    return dict((k, int(v)) for k, v in re.findall(r"(GO2P_PREC_\w+)\s*=\s*(\d+)", body)).get(name), body


def test_header_enum_and_python_constant_agree(lib):
    value, body = _enum("GO2P_PREC_FP32_TC")
    assert value == capi.PREC_FP32_TC == 4
    assert 3 not in [int(v) for v in re.findall(r"=\s*(\d+)", body)]      # the rejected tf32 slot stays empty
    assert (capi.PREC_FP32, capi.PREC_BF16, capi.PREC_FP16) == (0, 1, 2)
    assert capi.PREC_NAMES == {"fp32": 0, "bf16": 1, "fp16": 2}          # what bench.py offers is unchanged
    assert lib.go2p_abi_version() == 2


def test_python_defaults_stay_fp32_and_docstrings_name_the_new_value():
    import inspect
    for fn in (PolicyBatch.infer_device, PolicyBatch.infer_host, PolicyBatch.step_device, PolicyBatch.step_device_cmd,
               PolicyBatch.step_fields, PolicyBatch.step_host, Fleet.infer_host, Fleet.step_host):
        assert inspect.signature(fn).parameters["precision"].default == capi.PREC_FP32, fn.__name__
    assert "PREC_FP32_TC" in PolicyBatch.__doc__ and "PREC_FP32_TC" in Fleet.__doc__


def test_precision_switch_accepts_the_new_value_and_rejects_the_tf32_slot(lib):
    """go2p_infer_batch's precision switch, reached without a device: a zeroed buffer stands in for a handle that serves
    no tensor-core path (every *_ok flag 0) and has no batch-1 or fleet state, and B > 0 with non-null buffers passes
    the argument checks.  3 (the rejected tf32 slot) and unknown values are GO2P_ERR_INVALID 'unknown precision';
    GO2P_PREC_FP32_TC is a known precision that this handle does not serve: GO2P_ERR_UNSUPPORTED, pointing to
    GO2P_PREC_FP32 -- nothing is launched in either case."""
    fake = np.zeros(1 << 20, np.uint8)
    h = C.c_void_p(fake.ctypes.data)
    buf = np.zeros(64, np.float32)
    p = buf.ctypes.data
    for bad in (3, 5, 99, -1):
        assert lib.go2p_infer_batch(h, p, p, 4, bad, None) == capi.ERR_INVALID, bad
        assert b"unknown precision" in lib.go2p_last_error(), bad
    assert lib.go2p_infer_batch(h, p, p, 4, capi.PREC_FP32_TC, None) == capi.ERR_UNSUPPORTED
    msg = lib.go2p_last_error()
    assert b"GO2P_PREC_FP32_TC" in msg and b"use GO2P_PREC_FP32" in msg
    assert lib.go2p_last_launch_count(h) == 0
