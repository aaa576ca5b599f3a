"""CPU tests of the per-field step sequence (go2p_step_batch_fields_seq, PolicyBatch.step_fields_seq): the entry point is
declared, exported and bound, refuses null pointers with the argument named, negative T or B and a T*B that overflows,
and the Python validator checks the [T,B,w] tensors before any native call.  The sequence itself is tested on the GPU
(test_gpu_fields_seq.py)."""
import ctypes as C
import re

import numpy as np
import pytest

from go2_onnx_controller_b200 import actor, build, capi

from test_fields_cpu import FakeTensor


@pytest.fixture(scope="module")
def lib():
    build.build()
    return capi.load()


def test_seq_entry_point_is_declared_exported_and_bound(lib):
    with open(build.ROOT + "/include/go2policy.h") as fh:
        hdr = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    assert re.search(r"\bint go2p_step_batch_fields_seq\(", hdr)
    assert "go2p_step_batch_fields_seq" in capi.SIGNATURES and hasattr(lib, "go2p_step_batch_fields_seq")
    assert lib.go2p_abi_version() == 2


def _call(lib, h, f, buf, T=2, B=4, action_seq=True, state=None):
    p = buf.ctypes.data
    st = dict(d_vel_cmd=p, d_obs=p, d_action=p)
    st.update(state or {})
    return lib.go2p_step_batch_fields_seq(h, f, T, None, st["d_vel_cmd"], st["d_obs"], st["d_action"],
                                          p if action_seq else None, None, None, None, B, capi.PREC_FP16, None)


def _full(buf):
    return capi.RawFields(*[buf.ctypes.data] * len(capi.RawFields._fields_))


def test_null_arguments_are_named(lib):
    buf = np.zeros(4096, np.float32)
    assert _call(lib, None, C.byref(_full(buf)), buf) == capi.ERR_INVALID
    assert b"null handle" in lib.go2p_last_error()
    # every pointer check comes before anything reads the handle: a non-null dummy stands in for one
    fake = C.c_void_p(buf.ctypes.data)
    assert _call(lib, fake, None, buf) == capi.ERR_INVALID
    assert b"null go2p_raw_fields" in lib.go2p_last_error()
    for name, _ in capi.RawFields._fields_:
        f = _full(buf)
        setattr(f, name, None)
        assert _call(lib, fake, C.byref(f), buf) == capi.ERR_INVALID, name
        assert f"null {name}".encode() in lib.go2p_last_error(), name
    for name in ("d_vel_cmd", "d_obs", "d_action"):
        assert _call(lib, fake, C.byref(_full(buf)), buf, state={name: None}) == capi.ERR_INVALID, name
        assert f"null {name}".encode() in lib.go2p_last_error(), name
    assert _call(lib, fake, C.byref(_full(buf)), buf, action_seq=False) == capi.ERR_INVALID
    assert b"null d_action_seq" in lib.go2p_last_error()


@pytest.mark.parametrize("T,B", [(-1, 4), (2, -1), (-3, -3), (2**62, 2**3), (2**31, 2**31), (1, 2**62)])
def test_negative_or_overflowing_sizes_are_invalid(lib, T, B):
    buf = np.zeros(4096, np.float32)
    fake = C.c_void_p(buf.ctypes.data)
    assert _call(lib, fake, C.byref(_full(buf)), buf, T=T, B=B) == capi.ERR_INVALID
    assert re.search(rb"negative T or B|overflows int64", lib.go2p_last_error())


T, B, IN_DIM = 3, 5, 98
WIDTH = dict(actor.RAW_FIELDS)


def _dtype(name):
    return "torch.int16" if name == "foot_force" else "torch.uint8" if WIDTH[name] is None else "torch.float32"


def _good():
    fields = {n: FakeTensor((T, B, w) if w else (T, B), _dtype(n)) for n, w in actor.RAW_FIELDS}
    return dict(fields=fields, vel_cmd=FakeTensor((B, 3)), obs=FakeTensor((B, IN_DIM)), action=FakeTensor((B, 12)),
                qdes=FakeTensor((T, B, 12), "torch.float64"), cmd=FakeTensor((T, B, 112), "torch.uint8"),
                reset=FakeTensor((T, B), "torch.bool"), action_seq=FakeTensor((T, B, 12)),
                obs_seq=FakeTensor((T, B, IN_DIM)))


def _validate(kw):
    return actor.step_field_tensors(IN_DIM, 0, seq=True, **kw)


def test_validator_accepts_good_tensors():
    assert _validate(_good()) == (T, B)
    kw = _good()
    kw.update(qdes=None, cmd=None, reset=None, obs_seq=None)      # every per-step output but the action is optional
    assert _validate(kw) == (T, B)
    assert actor.step_field_tensors(IN_DIM, 0, **{k: v for k, v in _good().items()
                                                  if k not in ("action_seq", "obs_seq")} | dict(
        fields={n: FakeTensor((B, w) if w else (B,), _dtype(n)) for n, w in actor.RAW_FIELDS},
        qdes=FakeTensor((B, 12), "torch.float64"), cmd=None, reset=None)) == B     # the single step is unchanged


def _with(name, t=None, **top):
    kw = _good()
    if name is not None:
        kw["fields"][name] = t
    kw.update(top)
    return kw


def _bad_cases():
    cases = []
    for n, w in actor.RAW_FIELDS:
        shape, dt = ((T, B, w) if w else (T, B)), _dtype(n)
        wrong = "torch.float32" if dt != "torch.float32" else "torch.float64"
        cases += [
            (f"{n} dtype", _with(n, FakeTensor(shape, wrong)), TypeError),
            (f"{n} steps", _with(n, FakeTensor((T + 1,) + shape[1:], dt)), ValueError),
            (f"{n} rows", _with(n, FakeTensor((T, B + 1) + shape[2:], dt)), ValueError),
            (f"{n} without the step dimension", _with(n, FakeTensor(shape[1:], dt)), ValueError),
            (f"{n} non-contiguous", _with(n, FakeTensor(shape, dt, contiguous=False)), ValueError),
            (f"{n} CPU tensor", _with(n, FakeTensor(shape, dt, device=("cpu", None))), TypeError),
            (f"{n} numpy array", _with(n, np.zeros(shape, np.float32)), TypeError),
        ]
        if w:
            cases.append((f"{n} width", _with(n, FakeTensor((T, B, w + 1), dt)), ValueError))
    cases += [
        ("quat without the step dimension", _with("quat", FakeTensor((B, 4))), ValueError),
        ("action_seq missing", _with(None, action_seq=None), ValueError),
        ("action_seq steps", _with(None, action_seq=FakeTensor((T - 1, B, 12))), ValueError),
        ("action_seq rows", _with(None, action_seq=FakeTensor((T, B + 1, 12))), ValueError),
        ("action_seq width", _with(None, action_seq=FakeTensor((T, B, 13))), ValueError),
        ("action_seq float64", _with(None, action_seq=FakeTensor((T, B, 12), "torch.float64")), TypeError),
        ("action_seq non-contiguous", _with(None, action_seq=FakeTensor((T, B, 12), contiguous=False)), ValueError),
        ("action_seq on CPU", _with(None, action_seq=FakeTensor((T, B, 12), device=("cpu", None))), TypeError),
        ("obs_seq width", _with(None, obs_seq=FakeTensor((T, B, IN_DIM + 1))), ValueError),
        ("obs_seq steps", _with(None, obs_seq=FakeTensor((T + 1, B, IN_DIM))), ValueError),
        ("obs_seq float16", _with(None, obs_seq=FakeTensor((T, B, IN_DIM), "torch.float16")), TypeError),
        ("qdes_seq without the step dimension", _with(None, qdes=FakeTensor((B, 12), "torch.float64")), ValueError),
        ("qdes_seq float32", _with(None, qdes=FakeTensor((T, B, 12))), TypeError),
        ("cmd_seq shape", _with(None, cmd=FakeTensor((T, B, 14), "torch.uint8")), ValueError),
        ("reset without the step dimension", _with(None, reset=FakeTensor((B,), "torch.bool")), ValueError),
        ("reset int32", _with(None, reset=FakeTensor((T, B), "torch.int32")), TypeError),
        ("obs with a step dimension", _with(None, obs=FakeTensor((T, B, IN_DIM))), ValueError),
        ("action with a step dimension", _with(None, action=FakeTensor((T, B, 12))), ValueError),
        ("vel_cmd float64", _with(None, vel_cmd=FakeTensor((B, 3), "torch.float64")), TypeError),
        ("vel_cmd on another GPU", _with(None, vel_cmd=FakeTensor((B, 3), device=("cuda", 1))), ValueError),
    ]
    return cases


@pytest.mark.parametrize("case", _bad_cases(), ids=lambda c: c[0])
def test_validator_rejects_bad_input(case):
    _, kw, exc = case
    with pytest.raises(exc):
        _validate(kw)
