"""CPU tests of the per-field step (go2p_step_batch_fields, PolicyBatch.step_fields): the entry point is declared,
exported and bound, refuses a null handle, struct or field with a message, and the Python layer validates the tensors
before any native call.  The step itself is tested on the GPU (test_gpu_fields.py)."""
import ctypes as C
import re

import numpy as np
import pytest

from go2_onnx_controller_b200 import actor, build, capi


@pytest.fixture(scope="module")
def lib():
    build.build()
    return capi.load()


def test_fields_entry_point_is_declared_exported_and_bound(lib):
    with open(build.ROOT + "/include/go2policy.h") as fh:
        hdr = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    assert re.search(r"\bint go2p_step_batch_fields\(", hdr)
    assert "typedef struct go2p_raw_fields" in hdr
    assert "go2p_step_batch_fields" in capi.SIGNATURES and hasattr(lib, "go2p_step_batch_fields")
    assert C.sizeof(capi.RawFields) == 8 * C.sizeof(C.c_void_p)
    assert lib.go2p_abi_version() == 2                 # additive change: the ABI version stays


def _call(lib, h, f, buf):
    p = buf.ctypes.data
    return lib.go2p_step_batch_fields(h, f, None, p, p, p, p, None, 4, capi.PREC_FP16, None)


def test_null_handle_struct_or_field_is_invalid(lib):
    buf = np.zeros(4096, np.float32)
    names = [n for n, _ in capi.RawFields._fields_]
    full = capi.RawFields(*[buf.ctypes.data] * len(names))
    assert _call(lib, None, C.byref(full), buf) == capi.ERR_INVALID
    assert b"null handle" in lib.go2p_last_error()
    # the struct and field checks come before anything reads the handle: a non-null dummy stands in for one
    fake = C.c_void_p(buf.ctypes.data)
    assert _call(lib, fake, None, buf) == capi.ERR_INVALID
    assert b"null go2p_raw_fields" in lib.go2p_last_error()
    for name in names:
        f = capi.RawFields(*[buf.ctypes.data] * len(names))
        setattr(f, name, None)
        assert _call(lib, fake, C.byref(f), buf) == capi.ERR_INVALID, name
        assert f"null {name}".encode() in lib.go2p_last_error(), name


class FakeDevice:
    def __init__(self, type_, index):
        self.type, self.index = type_, index

    def __str__(self):
        return f"{self.type}:{self.index}"


class FakeTensor:
    """What the validator reads of a torch tensor (duck typing: the product does not import torch)."""
    def __init__(self, shape, dtype="torch.float32", device=("cuda", 0), contiguous=True):
        self.shape, self.dtype, self.device, self._c = tuple(shape), dtype, FakeDevice(*device), contiguous

    def data_ptr(self):
        return 0x1000

    def is_contiguous(self):
        return self._c


B, IN_DIM = 5, 98
WIDTH = dict(actor.RAW_FIELDS)


def _good():
    fields = {n: FakeTensor((B, w) if w else (B,), "torch.int16" if n == "foot_force" else
                            "torch.bool" if w is None else "torch.float32") for n, w in actor.RAW_FIELDS}
    return dict(fields=fields, vel_cmd=FakeTensor((B, 3)), obs=FakeTensor((B, IN_DIM)), action=FakeTensor((B, 12)),
                qdes=FakeTensor((B, 12), "torch.float64"), cmd=FakeTensor((B, 112), "torch.uint8"),
                reset=FakeTensor((B,), "torch.uint8"))


def _validate(kw):
    return actor.step_field_tensors(IN_DIM, 0, **kw)


def test_validator_accepts_good_tensors():
    assert _validate(_good()) == B
    kw = _good()
    kw["fields"]["joy_valid"] = FakeTensor((B,), "torch.uint8")
    kw.update(qdes=None, reset=None)
    assert _validate(kw) == B
    kw = _good()
    kw["cmd"] = None
    assert _validate(kw) == B


def _with(name, t=None, **top):
    kw = _good()
    if name is not None:
        kw["fields"][name] = t
    kw.update(top)
    return kw


def _dtype(name):
    return "torch.int16" if name == "foot_force" else "torch.uint8" if WIDTH[name] is None else "torch.float32"


def _bad_cases():
    cases = []
    for n, w in actor.RAW_FIELDS:
        shape, dt = ((B, w) if w else (B,)), _dtype(n)
        wrong = "torch.float32" if dt != "torch.float32" else "torch.float64"
        cases += [
            (f"{n} dtype", _with(n, FakeTensor(shape, wrong)), TypeError),
            (f"{n} width", _with(n, FakeTensor((B, (w or 1) + 1), dt)), ValueError),
            (f"{n} rows", _with(n, FakeTensor((B + 1,) + shape[1:], dt)), ValueError),
            (f"{n} non-contiguous", _with(n, FakeTensor(shape, dt, contiguous=False)), ValueError),
            (f"{n} CPU tensor", _with(n, FakeTensor(shape, dt, device=("cpu", None))), TypeError),
            (f"{n} another GPU", _with(n, FakeTensor(shape, dt, device=("cuda", 1))), ValueError),
            (f"{n} numpy array", _with(n, np.zeros(shape, np.float32)), TypeError),
        ]
    cases += [
        ("int32 foot_force", _with("foot_force", FakeTensor((B, 4), "torch.int32")), TypeError),
        ("int32 button0", _with("button0", FakeTensor((B,), "torch.int32")), TypeError),
        ("qdes float32", _with(None, qdes=FakeTensor((B, 12))), TypeError),
        ("cmd float32", _with(None, cmd=FakeTensor((B, 112))), TypeError),
        ("cmd shape", _with(None, cmd=FakeTensor((B, 14), "torch.uint8")), ValueError),
        ("obs width", _with(None, obs=FakeTensor((B, IN_DIM + 1))), ValueError),
        ("vel_cmd float64", _with(None, vel_cmd=FakeTensor((B, 3), "torch.float64")), TypeError),
        ("action rows", _with(None, action=FakeTensor((B - 1, 12))), ValueError),
        ("action non-contiguous", _with(None, action=FakeTensor((B, 12), contiguous=False)), ValueError),
        ("obs on CPU", _with(None, obs=FakeTensor((B, IN_DIM), device=("cpu", None))), TypeError),
        ("vel_cmd on another GPU", _with(None, vel_cmd=FakeTensor((B, 3), device=("cuda", 1))), ValueError),
        ("reset int32", _with(None, reset=FakeTensor((B,), "torch.int32")), TypeError),
        ("reset shape", _with(None, reset=FakeTensor((B + 1,), "torch.bool")), ValueError),
        ("qdes and cmd both None", _with(None, qdes=None, cmd=None), ValueError),
    ]
    return cases


@pytest.mark.parametrize("case", _bad_cases(), ids=lambda c: c[0])
def test_validator_rejects_bad_input(case):
    _, kw, exc = case
    with pytest.raises(exc):
        _validate(kw)
