"""The batched controller step from per-field device tensors (go2p_step_batch_fields, PolicyBatch.step_fields).

Its contract is twin identity: from the same state and the same raw values, the per-field step leaves exactly the bits
the record step (go2p_step_batch_ex) leaves, on every path -- the one-launch fused kernel (fp16 / bf16, full and ragged
tiles), the two-kernel chain (fp32, the wide H = 5 policy, a misaligned field) -- and reports the same launch count.
The record step itself is checked against the oracle by test_gpu_resets.py and test_gpu_round2.py.  The records carry
joy_valid / button0 = 7 where the fields carry 1: both are only ever compared with 0."""
import ctypes as C

import numpy as np
import pytest

from go2_onnx_controller_b200 import PolicyBatch, actor, capi

from test_gpu_resets import _poison, _raws
from test_gpu_round2 import CMD_DT

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

PRECS = [capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16]


def _inputs(torch, golden_loop, rng, B):
    """Records (uint8 [B,156] on the device, flags 7) and the same values as eight field tensors (flags bool / uint8)."""
    raw, rv = _raws(golden_loop, rng, B)
    for f in ("joy_valid", "button0"):
        rv[f][rv[f] != 0] = 7
    fields = {n: torch.from_numpy(np.ascontiguousarray(rv[n])).cuda() for n, _ in actor.RAW_FIELDS[:6]}
    fields["joy_valid"] = torch.from_numpy(rv["joy_valid"] != 0).cuda()                       # torch.bool
    fields["button0"] = torch.from_numpy((rv["button0"] != 0).astype(np.uint8)).cuda()
    return torch.from_numpy(raw).cuda(), fields


def _state(rng, B, in_dim):
    return (rng.standard_normal((B, in_dim)).astype(np.float32), rng.standard_normal((B, 3)).astype(np.float32),
            rng.standard_normal((B, 12)).astype(np.float32))


def _raw_fields(fields):
    return capi.RawFields(*[fields[n].data_ptr() for n, _ in actor.RAW_FIELDS])


def _step(pb, torch, src, d_rst, state, prec):
    """One step from a copy of `state` (obs, vel, act); src: a record tensor or a dict of field tensors.  Returns every
    output as bytes-comparable numpy arrays plus the launch count."""
    B = state[0].shape[0]
    d_obs, d_vel, d_act = (torch.from_numpy(x).cuda() for x in state)
    d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
    d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
    rst = None if d_rst is None else d_rst.data_ptr()
    out = (d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(), d_cmd.data_ptr(), B, prec, None)
    lib, h = pb._hd.lib, pb._hd.h
    if isinstance(src, dict):
        capi.check(lib.go2p_step_batch_fields(h, C.byref(_raw_fields(src)), rst, *out))
    else:
        capi.check(lib.go2p_step_batch_ex(h, src.data_ptr(), rst, *out))
    torch.cuda.synchronize()
    return [t.cpu().numpy().view(np.uint8) for t in (d_obs, d_vel, d_act, d_q, d_cmd)] + [pb.last_launches()]


def _same(a, b, what):
    for name, x, y in zip(("obs", "vel_cmd", "action", "q_des", "cmd", "launches"), a, b):
        assert np.array_equal(x, y), (what, name)


def _mask(torch, kind, rng, B, state):
    if kind == "none":
        return None
    if kind == "zeros":
        return torch.zeros(B, device="cuda", dtype=torch.uint8)
    m = rng.random(B) < 0.15
    for x in state:
        x[m] = np.nan
    return torch.from_numpy(m).cuda()


@pytest.mark.parametrize("B", [333, 100_077, 1])
@pytest.mark.parametrize("prec", PRECS)
def test_fields_and_records_leave_identical_bits(torch_cuda, model_path, golden_loop, prec, B):
    torch = torch_cuda
    rng = np.random.default_rng(B + prec)
    d_raw, fields = _inputs(torch, golden_loop, rng, B)
    pb = PolicyBatch(model_path)
    try:
        for kind in ("none", "zeros", "random"):
            state = _state(rng, B, 98)
            d_rst = _mask(torch, kind, rng, B, state)
            rec = _step(pb, torch, d_raw, d_rst, state, prec)
            fld = _step(pb, torch, fields, d_rst, state, prec)
            _same(rec, fld, kind)
            assert fld[-1] == (5 if prec == capi.PREC_FP32 else 1)
    finally:
        pb.close()


@pytest.mark.parametrize("prec", PRECS)
def test_closed_loop_stays_identical(torch_cuda, model_path, golden_loop, prec):
    """8 steps fed back on the device's own state (history, command, action), ~15 % random resets with NaN-poisoned
    rows; B = 5,000 (39 full tiles + a ragged one)."""
    torch = torch_cuda
    B, steps = 5_000, 8
    rng = np.random.default_rng(40 + prec)
    pb = PolicyBatch(model_path)
    try:
        bufs = {}
        for src in ("rec", "fld"):
            bufs[src] = dict(obs=torch.zeros((B, 98), device="cuda"), vel=torch.zeros((B, 3), device="cuda"),
                             act=torch.zeros((B, 12), device="cuda"),
                             q=torch.zeros((B, 12), device="cuda", dtype=torch.float64),
                             cmd=torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8))
        for s in range(steps):
            d_raw, fields = _inputs(torch, golden_loop, rng, B)
            mask = rng.random(B) < 0.15
            launches = {}
            for src, b in bufs.items():
                _poison(torch, mask, b["obs"], b["vel"], b["act"])
                d_rst = torch.from_numpy(mask).cuda()
                if src == "rec":
                    pb.step_device_cmd(d_raw.data_ptr(), b["vel"].data_ptr(), b["obs"].data_ptr(), b["act"].data_ptr(),
                                       b["q"].data_ptr(), b["cmd"].data_ptr(), B, prec, d_reset=d_rst.data_ptr())
                else:
                    pb.step_fields(**fields, vel_cmd=b["vel"], obs=b["obs"], action=b["act"], qdes=b["q"], cmd=b["cmd"],
                                   precision=prec, reset=d_rst)
                torch.cuda.synchronize()
                launches[src] = pb.last_launches()
            assert launches["rec"] == launches["fld"] == (5 if prec == capi.PREC_FP32 else 1)
            for k in bufs["rec"]:
                assert torch.equal(bufs["rec"][k].view(torch.uint8), bufs["fld"][k].view(torch.uint8)), (s, k)
            assert torch.isfinite(bufs["fld"]["act"]).all(), s
    finally:
        pb.close()


@pytest.mark.parametrize("prec", [capi.PREC_FP16, capi.PREC_BF16])
def test_misaligned_field_takes_the_two_kernel_chain(torch_cuda, model_path, golden_loop, prec):
    """A field 4 bytes off a 16-byte boundary sends the step through assemble_batch_kernel + the policy kernel (2
    launches), matching records whose d_raw is misaligned the same way; with resets."""
    torch = torch_cuda
    B = 1_000
    rng = np.random.default_rng(55)
    d_raw, fields = _inputs(torch, golden_loop, rng, B)
    raw_buf = torch.zeros(B * d_raw.shape[1] + 4, device="cuda", dtype=torch.uint8)
    raw_off = raw_buf[4:].view(B, d_raw.shape[1])
    raw_off.copy_(d_raw)
    pb = PolicyBatch(model_path)
    try:
        for name in ("quat", "gyro", "q", "foot_force", "button0"):
            t = fields[name]
            buf = torch.zeros(t.numel() + 8, device="cuda", dtype=t.dtype)
            off = 4 // t.element_size()
            moved = buf[off:off + t.numel()].view(t.shape)
            moved.copy_(t)
            assert moved.data_ptr() % 16 == 4 and moved.is_contiguous()
            state = _state(rng, B, 98)
            d_rst = _mask(torch, "random", rng, B, state)
            rec = _step(pb, torch, raw_off, d_rst, state, prec)
            fld = _step(pb, torch, dict(fields, **{name: moved}), d_rst, state, prec)
            _same(rec, fld, name)
            assert fld[-1] == 2, name
            assert _step(pb, torch, fields, d_rst, state, prec)[-1] == 1      # aligned again: one launch
    finally:
        pb.close()


@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16])
def test_wide_policy(torch_cuda, wide_model_path, golden_loop, prec):
    """The 245-1024-512-256-12 policy at H = 5 (assemble_batch_kernel + the wide chain): fields and records agree."""
    torch = torch_cuda
    B = 333
    rng = np.random.default_rng(61)
    d_raw, fields = _inputs(torch, golden_loop, rng, B)
    pb = PolicyBatch(wide_model_path, history=5)
    try:
        for kind in ("none", "random"):
            state = _state(rng, B, 245)
            d_rst = _mask(torch, kind, rng, B, state)
            _same(_step(pb, torch, d_raw, d_rst, state, prec), _step(pb, torch, fields, d_rst, state, prec), kind)
    finally:
        pb.close()


def test_empty_batch_and_python_wrapper(torch_cuda, model_path, golden_loop):
    """B = 0 reads and writes nothing; PolicyBatch.step_fields leaves the bits of the direct C call."""
    torch = torch_cuda
    B = 333
    rng = np.random.default_rng(70)
    d_raw, fields = _inputs(torch, golden_loop, rng, B)
    pb = PolicyBatch(model_path)
    try:
        state = _state(rng, B, 98)
        d_obs, d_vel, d_act = (torch.from_numpy(x).cuda() for x in state)
        d_q = torch.full((B, 12), 3.0, device="cuda", dtype=torch.float64)
        assert pb._hd.lib.go2p_step_batch_fields(pb._hd.h, C.byref(_raw_fields(fields)), None, d_vel.data_ptr(),
                                                 d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(), None, 0,
                                                 capi.PREC_FP16, None) == capi.OK
        torch.cuda.synchronize()
        for got, exp in zip((d_obs, d_vel, d_act), state):
            assert np.array_equal(got.cpu().numpy().view(np.uint32), exp.view(np.uint32))
        assert (d_q == 3.0).all()
        empty = {n: t[:0] for n, t in fields.items()}
        pb.step_fields(**empty, vel_cmd=d_vel[:0], obs=d_obs[:0], action=d_act[:0], qdes=d_q[:0],
                       precision=capi.PREC_FP16)

        for prec in (capi.PREC_FP16, capi.PREC_FP32):
            d_rst = _mask(torch, "random", rng, B, state)
            direct = _step(pb, torch, fields, d_rst, state, prec)
            d_obs, d_vel, d_act = (torch.from_numpy(x).cuda() for x in state)
            d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
            d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
            pb.step_fields(**fields, vel_cmd=d_vel, obs=d_obs, action=d_act, qdes=d_q, cmd=d_cmd, precision=prec,
                           stream=torch.cuda.current_stream().cuda_stream, reset=d_rst)
            torch.cuda.synchronize()
            wrapped = [t.cpu().numpy().view(np.uint8) for t in (d_obs, d_vel, d_act, d_q, d_cmd)] + [pb.last_launches()]
            _same(direct, wrapped, prec)
        with pytest.raises(ValueError):
            pb.step_fields(**fields, vel_cmd=d_vel, obs=d_obs, action=d_act)
    finally:
        pb.close()
