"""Per-robot resets in the batched controller step (go2p_step_batch_ex, go2p_step_batch_host_ex, go2p_fleet_step_host_ex).

A robot whose reset byte is non-zero starts the step from the controller's initial state (controller.hpp:132-162:
histories 0, previous action 0, joystick command 0) and then steps as usual; the checker is the oracle's
ControllerState.reset() + controller_step.  Rows to be reset are poisoned with NaN first: nothing they held may reach
the outputs.  Robots with a zero byte step exactly as without a mask."""
import ctypes as C

import numpy as np
import pytest

from go2_onnx_controller_b200 import Fleet, PolicyBatch, capi
from oracle import coracle, oracle

from test_gpu_parity import TC_TOL, TOL_FP32, bits
from test_gpu_round2 import CMD_DT, RAW_DT, _raw_bytes, check_cmd

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


def _raw_py(rv, b):
    return oracle.RawState(quat=rv["quat"][b], gyro=rv["gyro"][b], q=rv["q"][b], dq=rv["dq"][b],
                           foot_force=rv["foot_force"][b], axes=rv["axes"][b], joy_valid=int(rv["joy_valid"][b]),
                           button0=int(rv["button0"][b]))


def _raws(g, rng, B, no_joy_every=3, button_p=0.1):
    """B golden raw states, joy_valid = 0 on every third robot, the dead-man button pressed on some."""
    raw = _raw_bytes(g, rng.integers(0, g["obs"].shape[0], B), rng.random(B) < button_p)
    rv = raw.view(RAW_DT).reshape(B)
    rv["joy_valid"][np.arange(B) % no_joy_every == 0] = 0
    return raw, rv


def _poison(torch, mask, *bufs):
    m = torch.from_numpy(mask).cuda()
    for t in bufs:
        t[m] = float("nan")


def _gravity_ok(got, exp, H):
    return np.abs(bits(got[:3 * H]).astype(np.int64) - bits(exp[:3 * H]).astype(np.int64)).max() <= 1


@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16])
def test_resets_closed_loop_vs_oracle(torch_cuda, model_path, policy, golden_loop, prec):
    """B = 333 (two full tiles + a ragged one), 8 closed-loop steps, ~15 % random resets per step (every robot at step
    0), the reset rows poisoned with NaN beforehand.  Observation (gravity <= 1 ulp) and joystick command bit-exact,
    action within the precision's bound, q_des and motor command bit-exact, launch count unchanged."""
    torch = torch_cuda
    B, steps, H = 333, 8, 2
    rng = np.random.default_rng(100 + prec)
    pb = PolicyBatch(model_path)
    tol = TOL_FP32 if prec == capi.PREC_FP32 else 1e-2 if prec == capi.PREC_FP16 else TC_TOL[capi.PREC_BF16]["d1"]
    states = [oracle.ControllerState(H=H) for _ in range(B)]
    try:
        d_obs = torch.zeros((B, 49 * H), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
        d_act = torch.zeros((B, 12), device="cuda"); d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
        d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
        n_reset = n_masked = 0
        for s in range(steps):
            raw, rv = _raws(golden_loop, rng, B)
            mask = np.ones(B, np.bool_) if s == 0 else rng.random(B) < 0.15
            _poison(torch, mask, d_obs, d_vel, d_act)
            d_raw = torch.from_numpy(raw).cuda(); d_rst = torch.from_numpy(mask).cuda()
            pb.step_device_cmd(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(),
                               d_cmd.data_ptr(), B, prec, d_reset=d_rst.data_ptr())
            torch.cuda.synchronize()
            assert pb.last_launches() == (5 if prec == capi.PREC_FP32 else 1)
            obs, vel, act, qd = d_obs.cpu().numpy(), d_vel.cpu().numpy(), d_act.cpu().numpy(), d_q.cpu().numpy()
            cmd = d_cmd.cpu().numpy().view(CMD_DT).reshape(B)
            assert np.isfinite(obs).all() and np.isfinite(vel).all() and np.isfinite(act).all(), s
            ref_act = oracle.forward(policy, obs, np.float64)
            for b in range(B):
                if mask[b]:
                    states[b].reset()
                so = oracle.controller_step(policy, states[b], _raw_py(rv, b), np.float64, act_fn=lambda o: ref_act[b])
                assert _gravity_ok(obs[b], so.obs, H), (s, b)
                assert np.array_equal(bits(obs[b, 3 * H:]), bits(so.obs[3 * H:])), (s, b, bool(mask[b]))
                assert np.array_equal(bits(vel[b]), bits(states[b].vel_cmd)), (s, b, bool(mask[b]))
                assert (np.abs(act[b] - so.action) / np.maximum(1, np.abs(so.action))).max() <= tol, (s, b)
                states[b].action = act[b].copy()          # closed loop on the device's own published action
                states[b].hist[0][:] = obs[b, :3 * H]     # keep the <= 1-ulp gravity difference from accumulating
            check_cmd(act, qd, cmd, rv["button0"])
            n_reset += int(mask.sum()); n_masked += int((rv["button0"] != 0).sum())
        assert n_reset > B + 200 and n_masked > 100
    finally:
        pb.close()


def _step_ex(pb, torch, d_raw, d_rst, state, B, prec, use):
    """One step from a copy of `state` (obs, vel, act) through one of the three entry points; returns the new state."""
    d_obs, d_vel, d_act = (torch.from_numpy(x).cuda() for x in state)
    d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
    lib, h = pb._hd.lib, pb._hd.h
    args = (d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), None, d_cmd.data_ptr(), B, prec, None)
    if use == "cmd":
        rc = lib.go2p_step_batch_cmd(h, d_raw.data_ptr(), *args)
    else:
        rc = lib.go2p_step_batch_ex(h, d_raw.data_ptr(), None if d_rst is None else d_rst.data_ptr(), *args)
    capi.check(rc)
    torch.cuda.synchronize()
    return d_obs.cpu().numpy(), d_vel.cpu().numpy(), d_act.cpu().numpy(), d_cmd.cpu().numpy(), pb.last_launches()


@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16])
def test_no_mask_zero_mask_and_old_entry_point_agree(torch_cuda, model_path, golden_loop, prec):
    """go2p_step_batch_cmd, _ex with NULL and _ex with an all-zero mask leave identical bits from the same random state;
    a mask byte of 0xFF resets a robot just as 1 does; argument errors and the empty batch."""
    torch = torch_cuda
    B = 100_000 + 77
    rng = np.random.default_rng(7)
    state = (rng.standard_normal((B, 98)).astype(np.float32), rng.standard_normal((B, 3)).astype(np.float32),
             rng.standard_normal((B, 12)).astype(np.float32))
    raw, _ = _raws(golden_loop, rng, B)
    d_raw = torch.from_numpy(raw).cuda()
    pb = PolicyBatch(model_path)
    try:
        ref = _step_ex(pb, torch, d_raw, None, state, B, prec, "cmd")
        for d_rst in (None, torch.zeros(B, device="cuda", dtype=torch.uint8)):
            got = _step_ex(pb, torch, d_raw, d_rst, state, B, prec, "ex")
            for x, y in zip(got[:4], ref[:4]):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
            assert got[4] == ref[4]
        sel = rng.random(B) < 0.3
        m1 = torch.from_numpy(sel.astype(np.uint8)).cuda()
        mff = torch.from_numpy(sel.astype(np.uint8) * np.uint8(0xFF)).cuda()
        a, b = _step_ex(pb, torch, d_raw, m1, state, B, prec, "ex"), _step_ex(pb, torch, d_raw, mff, state, B, prec, "ex")
        for x, y in zip(a[:4], b[:4]):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
        assert not np.array_equal(a[0][sel].view(np.uint32), ref[0][sel].view(np.uint32))   # the mask did something
        assert np.array_equal(a[0][~sel].view(np.uint32), ref[0][~sel].view(np.uint32))     # ... only on its rows
        # argument errors: null raw states, negative batch; B = 0 touches nothing
        lib, h = pb._hd.lib, pb._hd.h
        d_obs = torch.full((4, 98), 7.0, device="cuda"); d_vel = torch.full((4, 3), 7.0, device="cuda")
        d_act = torch.full((4, 12), 7.0, device="cuda"); d_q = torch.zeros((4, 12), device="cuda", dtype=torch.float64)
        ptrs = (d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(), None)
        assert lib.go2p_step_batch_ex(h, None, m1.data_ptr(), *ptrs, 4, prec, None) == capi.ERR_INVALID
        assert lib.go2p_step_batch_ex(h, d_raw.data_ptr(), m1.data_ptr(), *ptrs, -1, prec, None) == capi.ERR_INVALID
        assert lib.go2p_step_batch_ex(h, d_raw.data_ptr(), m1.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(),
                                      None, None, 4, prec, None) == capi.ERR_INVALID        # neither q_des nor commands
        assert lib.go2p_step_batch_ex(h, d_raw.data_ptr(), m1.data_ptr(), *ptrs, 0, prec, None) == capi.OK
        torch.cuda.synchronize()
        assert bool((d_obs == 7).all()) and bool((d_vel == 7).all()) and bool((d_act == 7).all())
    finally:
        pb.close()


def test_fused_resets_under_stage_reuse(torch_cuda, model_path, golden_loop):
    """B = 100,077: 5-6 tiles per CTA and a ragged last tile, so the fused kernel's observation and raw stages are
    reused.  From a random N(0,1) state with 50 % resets (their rows NaN) and a third of the robots without joystick,
    the fused fp16 step and the fp32 two-kernel chain leave the same observation rows and joystick commands, and the
    reset rows equal the same raw states stepped from all-zero buffers.  Repeated: a stage race would be timing
    dependent."""
    torch = torch_cuda
    B = 100_000 + 77
    rng = np.random.default_rng(13)
    mask = rng.random(B) < 0.5
    obs0 = rng.standard_normal((B, 98)).astype(np.float32); vel0 = rng.standard_normal((B, 3)).astype(np.float32)
    act0 = rng.standard_normal((B, 12)).astype(np.float32)
    for x in (obs0, vel0, act0):
        x[mask] = np.nan
    raw, rv = _raws(golden_loop, rng, B)
    d_raw = torch.from_numpy(raw).cuda(); d_rst = torch.from_numpy(mask).cuda()
    zero = (np.zeros_like(obs0), np.zeros_like(vel0), np.zeros_like(act0))
    pb = PolicyBatch(model_path)
    try:
        obs_ref, vel_ref, _, _, n = _step_ex(pb, torch, d_raw, d_rst, (obs0, vel0, act0), B, capi.PREC_FP32, "ex")
        assert n > 1
        obs_z, vel_z, act_z, cmd_z, _ = _step_ex(pb, torch, d_raw, None, zero, B, capi.PREC_FP16, "ex")
        for rep in range(3):
            obs, vel, act, cmd, n = _step_ex(pb, torch, d_raw, d_rst, (obs0, vel0, act0), B, capi.PREC_FP16, "ex")
            assert n == 1, rep
            assert np.array_equal(bits(obs), bits(obs_ref)), rep
            assert np.array_equal(bits(vel), bits(vel_ref)), rep
            assert np.array_equal(bits(obs[mask]), bits(obs_z[mask])), rep
            assert np.array_equal(bits(vel[mask]), bits(vel_z[mask])), rep
            assert np.array_equal(bits(act[mask]), bits(act_z[mask])), rep
            assert np.array_equal(cmd[mask], cmd_z[mask]), rep
            assert np.isfinite(act[mask]).all()
    finally:
        pb.close()


def test_host_and_fleet_forms_apply_the_same_resets(torch_cuda, model_path, golden_loop):
    """step_host(reset=...) with more than one 65,536-row pipeline chunk against step_device_cmd(d_reset=...) on caller
    buffers, and a Fleet (two devices, or two handles on one) against one handle: identical bits step after step."""
    torch = torch_cuda
    g = golden_loop
    B = 70_000
    rng = np.random.default_rng(17)
    host, dev = PolicyBatch(model_path), PolicyBatch(model_path)
    try:
        d_obs = torch.zeros((B, 98), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
        d_act = torch.zeros((B, 12), device="cuda"); d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
        h_act = np.zeros((B, 12), np.float32); h_cmd = np.zeros((B, CMD_DT.itemsize), np.uint8)
        for s in range(4):
            raw, _ = _raws(g, rng, B)
            mask = rng.random(B) < 0.2
            host.step_host(raw, h_act, h_cmd, capi.PREC_FP16, reset=mask)
            d_raw = torch.from_numpy(raw).cuda(); d_rst = torch.from_numpy(mask).cuda()
            dev.step_device_cmd(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), None, d_cmd.data_ptr(), B,
                                capi.PREC_FP16, d_reset=d_rst.data_ptr())
            torch.cuda.synchronize()
            assert np.array_equal(bits(h_act), bits(d_act.cpu().numpy())), s
            assert np.array_equal(h_cmd, d_cmd.cpu().numpy()), s
        with pytest.raises(TypeError):
            host.step_host(raw, h_act, None, capi.PREC_FP16, reset=mask.astype(np.int32))
        with pytest.raises(ValueError):
            host.step_host(raw, h_act, None, capi.PREC_FP16, reset=mask[:-1])
    finally:
        host.close(); dev.close()

    devices = (0, 1) if torch.cuda.device_count() >= 2 else (0, 0)
    Bf = 5001
    one, fl = PolicyBatch(model_path), Fleet(model_path, devices=devices)
    try:
        a1, a2 = np.zeros((Bf, 12), np.float32), np.zeros((Bf, 12), np.float32)
        c1, c2 = np.zeros((Bf, CMD_DT.itemsize), np.uint8), np.zeros((Bf, CMD_DT.itemsize), np.uint8)
        for s in range(4):
            raw, _ = _raws(g, rng, Bf)
            mask = (rng.random(Bf) < 0.2).astype(np.uint8)
            one.step_host(raw, a1, c1, capi.PREC_FP16, reset=mask)
            fl.step_host(raw, a2, c2, capi.PREC_FP16, reset=mask)
            assert np.array_equal(bits(a1), bits(a2)), s
            assert np.array_equal(c1, c2), s
    finally:
        fl.close(); one.close()


def test_wide_policy_resets_through_the_assembly_kernel(torch_cuda, wide_model_path, golden_loop):
    """The 245-1024-512-256-12 policy at H = 5 is served by assemble_batch_kernel + the wide tcgen05 GEMMs (fp16):
    observations and joystick commands bit-exact against ControllerState(H=5) with resets, actions within 2e-2 abs of
    the C oracle's fp64 forward (the bound of test_wide_policy_tensor_core_path)."""
    torch = torch_cuda
    B, steps, H = 333, 6, 5
    rng = np.random.default_rng(19)
    cm = coracle.CModel(wide_model_path)
    pb = PolicyBatch(wide_model_path, history=H)
    states = [oracle.ControllerState(H=H) for _ in range(B)]
    try:
        d_obs = torch.zeros((B, 49 * H), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
        d_act = torch.zeros((B, 12), device="cuda"); d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
        for s in range(steps):
            raw, rv = _raws(golden_loop, rng, B)
            mask = np.ones(B, np.bool_) if s == 0 else rng.random(B) < 0.15
            _poison(torch, mask, d_obs, d_vel, d_act)
            d_raw = torch.from_numpy(raw).cuda(); d_rst = torch.from_numpy(mask).cuda()
            pb.step_device(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(), B,
                           capi.PREC_FP16, d_reset=d_rst.data_ptr())
            torch.cuda.synchronize()
            assert pb.last_launches() == 1 + 5                 # assembly + the wide chain
            obs, vel, act = d_obs.cpu().numpy(), d_vel.cpu().numpy(), d_act.cpu().numpy()
            ref = oracle.clamp_mask(cm.forward_f64(obs, 8).astype(np.float32), rv["button0"])
            assert np.abs(act - ref).max() <= 2e-2, (s, np.abs(act - ref).max())
            for b in range(B):
                if mask[b]:
                    states[b].reset()
                exp = oracle.assemble_observation(states[b], _raw_py(rv, b))
                assert _gravity_ok(obs[b], exp, H), (s, b)
                assert np.array_equal(bits(obs[b, 3 * H:]), bits(exp[3 * H:])), (s, b, bool(mask[b]))
                assert np.array_equal(bits(vel[b]), bits(states[b].vel_cmd)), (s, b, bool(mask[b]))
                states[b].action = act[b].copy()
                states[b].hist[0][:] = obs[b, :3 * H]
    finally:
        pb.close()
