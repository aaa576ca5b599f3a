"""GPU parity tests of the round-2 additions (run on a B200 with -m gpu), all through the C ABI:
  * send_command arguments in Unitree motor order from every output epilogue   (controller.cpp:235-251)
  * ObservationAction ring on the device                                       (ObservationAction.msg:1-2)
  * closed-loop fleet step from host buffers, several handles / devices in one process
The oracle (oracle/) is only the checker."""
import ctypes as C

import numpy as np
import pytest

from go2_onnx_controller_b200 import Fleet, Go2Controller, PolicyBatch, capi
from oracle import coracle, oracle

from test_gpu_parity import bits, raw_struct

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]

CMD_DT = np.dtype([("q_des", np.float64, 12), ("kp", np.float64), ("kd", np.float64)])


def run_cmd(torch, pb, X, prec, button0, flags):
    B = X.shape[0]
    d_obs = torch.from_numpy(np.ascontiguousarray(X, np.float32)).cuda()
    d_act = torch.zeros((B, pb.out_dim), device="cuda")
    d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
    d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
    d_b = torch.from_numpy(np.ascontiguousarray(button0, np.int32)).cuda()
    pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), B, prec, 0, d_b.data_ptr(), d_q.data_ptr(), flags, d_cmd.data_ptr())
    torch.cuda.synchronize()
    return d_act.cpu().numpy(), d_q.cpu().numpy(), d_cmd.cpu().numpy().view(CMD_DT).reshape(B)


def check_cmd(act, qd, cmd, button0, kp=28.0, kd=0.5):
    exp_q, exp_kp, exp_kd = oracle.joint_targets(act, button0[:, None], kp, kd)
    assert np.array_equal(qd.view(np.uint64), exp_q.view(np.uint64))                       # A11 bit-exact given the action
    mq, _, _ = oracle.motor_command(exp_q, None, None)
    assert np.array_equal(cmd["q_des"].view(np.uint64), mq.view(np.uint64))                # same doubles, motor order
    assert np.array_equal(cmd["kp"], np.where(button0 == 0, np.float64(np.float32(kp)), 5.0))
    assert np.array_equal(cmd["kd"], np.full(len(button0), np.float64(np.float32(kd))))


@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16])
def test_motor_cmd_from_the_fused_epilogues(torch_cuda, model_path, golden, prec):
    """Unitree-order q_des/kp/kd next to the Isaac-order q_des: identical doubles, permuted; kp follows button0."""
    pb = PolicyBatch(model_path)
    try:
        rng = np.random.default_rng(3)
        X = np.concatenate([golden["d3_obs"], oracle.make_obs_d1(1000, 98, seed=4)]).astype(np.float32)
        b0 = (rng.random(X.shape[0]) < 0.2).astype(np.int32)
        act, qd, cmd = run_cmd(torch_cuda, pb, X, prec, b0, capi.F_CLAMP_MASK | capi.F_QDES | capi.F_MOTOR_CMD)
        fin = np.isfinite(act).all(axis=1)
        check_cmd(act[fin], qd[fin], cmd[fin], b0[fin])
        assert not act[b0 == 1][np.isfinite(act[b0 == 1])].any()
        # gains changed at run time (ROS parameters, controller.cpp:254-277) reach the batched epilogue
        capi.check(pb._hd.lib.go2p_set_gains(pb._hd.h, 31.5, 0.75))
        act, qd, cmd = run_cmd(torch_cuda, pb, X[:300], prec, b0[:300], capi.F_CLAMP_MASK | capi.F_QDES | capi.F_MOTOR_CMD)
        fin = np.isfinite(act).all(axis=1)
        check_cmd(act[fin], qd[fin], cmd[fin], b0[:300][fin], 31.5, 0.75)
        # motor command without the Isaac-order q_des and without the clamp
        d = run_cmd(torch_cuda, pb, X[256:400], prec, b0[256:400], capi.F_MOTOR_CMD)
        exp_q, _, _ = oracle.joint_targets(d[0], 0)
        assert np.array_equal(d[2]["q_des"].view(np.uint64), oracle.motor_command(exp_q, 0, 0)[0].view(np.uint64))
        assert np.array_equal(d[2]["kp"], np.where(b0[256:400] == 0, np.float64(np.float32(31.5)), 5.0))
    finally:
        pb.close()


def test_motor_cmd_other_epilogues(torch_cuda, tmp_path, wide_model_path):
    """generic tcgen05 output epilogue (activation on the last layer), the wide per-layer GEMM path, and the fp32
    GEMM + elementwise A9/A11 kernel that serves last hidden layers too wide for the staged output kernel."""
    from oracle import onnx_mini
    rng = np.random.default_rng(11)
    cases = []
    dims = (64, 128, 12)
    ws = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for k, n in zip(dims[:-1], dims[1:])]
    bs = [rng.normal(0, 0.2, n).astype(np.float32) for n in dims[1:]]
    p1 = tmp_path / "act_last.onnx"
    p1.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0, final_activation=True))
    cases.append((str(p1), 64, (capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16)))
    cases.append((wide_model_path, 245, (capi.PREC_FP32, capi.PREC_FP16)))
    dims = (40, 640, 12)        # 128 staged rows of 640 floats do not fit in shared memory -> GEMM + post kernel
    ws = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for k, n in zip(dims[:-1], dims[1:])]
    bs = [rng.normal(0, 0.2, n).astype(np.float32) for n in dims[1:]]
    p3 = tmp_path / "wide_last.onnx"
    p3.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0))
    cases.append((str(p3), 40, (capi.PREC_FP32,)))
    for path, in_dim, precs in cases:
        pb = PolicyBatch(path)
        cm = coracle.CModel(path)
        try:
            X = rng.normal(0, 1, (333, in_dim)).astype(np.float32)
            b0 = (rng.random(333) < 0.3).astype(np.int32)
            for prec in precs:
                act, qd, cmd = run_cmd(torch_cuda, pb, X, prec, b0, capi.F_CLAMP_MASK | capi.F_QDES | capi.F_MOTOR_CMD)
                check_cmd(act, qd, cmd, b0)
                if prec == capi.PREC_FP32:
                    ref = oracle.clamp_mask(cm.forward_f64(X, 4).astype(np.float32), b0[:, None])
                    assert (np.abs(act - ref) / np.maximum(1, np.abs(ref))).max() <= 1e-5
        finally:
            pb.close()


def test_step_fused_cmd_and_observation_action_ring(torch_cuda, model_path, golden_loop):
    """Every control step's ObservationAction record (ObservationAction.msg:1-2, controller.cpp:226-229) lands in the
    device ring byte-equal to what go2p_step_out returned; the ring drops the oldest records when it is lapped."""
    g = golden_loop
    ctl = Go2Controller(model_path)
    try:
        ctl.log_enable(64)
        outs = []
        for i in range(40):
            out, cmd = ctl.step_cmd(raw_struct(g, i))
            q = np.frombuffer(out.q_des, np.float64, 12)
            assert np.array_equal(np.frombuffer(cmd.q_des, np.float64, 12), q[oracle.ISAAC_OF_MOTOR])
            assert cmd.kp == out.kp and cmd.kd == out.kd
            outs.append((np.frombuffer(out.observation, np.float32, 98).copy(), np.frombuffer(out.action, np.float32, 12).copy()))
        obs, act, dropped = ctl.log_drain(25)            # partial drain: the oldest 25
        assert obs.shape == (25, 98) and dropped == 0
        for k in range(25):
            assert np.array_equal(bits(obs[k]), bits(outs[k][0])) and np.array_equal(bits(act[k]), bits(outs[k][1]))
        obs, act, dropped = ctl.log_drain()
        assert obs.shape[0] == 15 and dropped == 0
        assert np.array_equal(bits(obs[-1]), bits(outs[39][0])) and np.array_equal(bits(act[-1]), bits(outs[39][1]))
        for i in range(40, 140):                           # 100 more steps lap the 64-record ring
            out = ctl.step(raw_struct(g, i))
            outs.append((np.frombuffer(out.observation, np.float32, 98).copy(), np.frombuffer(out.action, np.float32, 12).copy()))
        obs, act, dropped = ctl.log_drain()
        assert obs.shape[0] == 64 and dropped == 36
        for k in range(64):
            assert np.array_equal(bits(obs[k]), bits(outs[76 + k][0])) and np.array_equal(bits(act[k]), bits(outs[76 + k][1]))
        ctl.log_enable(0)                                  # off again: steps still work, drain is refused
        ctl.step(raw_struct(g, 0))
        with pytest.raises(capi.Go2PolicyError):
            ctl.log_drain()
    finally:
        ctl.close()


RAW_DT = np.dtype([("quat", np.float32, 4), ("gyro", np.float32, 3), ("q", np.float32, 12), ("dq", np.float32, 12),
                   ("axes", np.float32, 4), ("foot_force", np.int16, 4), ("joy_valid", np.int32), ("button0", np.int32)])
assert RAW_DT.itemsize == C.sizeof(capi.RawState)


def _raw_bytes(g, idx, button=None):
    """go2p_raw_state records of the golden raw states idx, as uint8 [n, 156] (vectorised: no per-robot ctypes)."""
    idx = np.asarray(idx)
    r = np.zeros(len(idx), RAW_DT)
    for f in ("quat", "gyro", "q", "dq", "axes", "foot_force", "joy_valid", "button0"):
        r[f] = g["raw_" + f][idx]
    if button is not None:
        r["button0"] = np.asarray(button).astype(np.int32)
    return r.view(np.uint8).reshape(len(idx), RAW_DT.itemsize).copy()


@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16])
def test_step_batch_host_matches_device_step(torch_cuda, model_path, golden_loop, prec):
    """go2p_step_batch_host (raw states in, actions + motor commands out, history resident in the handle) against
    go2p_step_batch_cmd on caller-owned device buffers: identical bits step after step, ragged chunking included."""
    torch = torch_cuda
    g = golden_loop
    n_g = g["obs"].shape[0]
    B = 70_000                       # more than one 65,536-row pipeline chunk
    host, dev = PolicyBatch(model_path), PolicyBatch(model_path)
    try:
        d_obs = torch.zeros((B, 98), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
        d_act = torch.zeros((B, 12), device="cuda"); d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
        h_act = np.zeros((B, 12), np.float32); h_cmd = np.zeros((B, CMD_DT.itemsize), np.uint8)
        rng = np.random.default_rng(5)
        for s in range(4):
            idx = rng.integers(0, n_g, B)
            raw = _raw_bytes(g, idx, rng.random(B) < 0.1)
            host.step_host(raw, h_act, h_cmd, prec)
            d_raw = torch.from_numpy(raw).cuda()
            dev.step_device_cmd(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), None, d_cmd.data_ptr(), B, prec)
            torch.cuda.synchronize()
            assert np.array_equal(bits(h_act), bits(d_act.cpu().numpy())), s
            assert np.array_equal(h_cmd, d_cmd.cpu().numpy()), s
        c = h_cmd.view(CMD_DT).reshape(B)
        exp_q, _, _ = oracle.joint_targets(h_act, 0)
        assert np.array_equal(c["q_des"].view(np.uint64), oracle.motor_command(exp_q, 0, 0)[0].view(np.uint64))
        host.step_host_reset()       # zeroed histories again: first step equals a fresh handle's
        fresh = PolicyBatch(model_path)
        a1, a2 = np.zeros((256, 12), np.float32), np.zeros((256, 12), np.float32)
        raw = _raw_bytes(g, list(range(256)))
        host.step_host(raw, a1, None, prec); fresh.step_host(raw, a2, None, prec)
        fresh.close()
        assert np.array_equal(bits(a1), bits(a2))
    finally:
        host.close(); dev.close()


def test_fused_step_with_many_tiles_per_cta_matches_the_two_kernel_chain(torch_cuda, model_path, golden_loop):
    """The fused fleet step (assembly inside the tcgen05 kernel) where every CTA walks several tiles per slot, i.e. where
    observation stages, the raw stage and the copy-back of updated rows are REUSED: from identical state, one step of the
    fused fp16 kernel must leave the same observation rows and joystick commands (bit for bit) as the fp32 path's
    assembly kernel (controller.cpp:173-212 is precision-free), and actions within the tensor-core tolerance.  Repeated,
    because a stage-reuse race would be timing dependent."""
    torch = torch_cuda
    g = golden_loop
    n_g = g["obs"].shape[0]
    B = 100_000 + 77                 # 782 tiles over 148 CTAs: 5-6 tiles per CTA, ragged last tile
    rng = np.random.default_rng(11)
    obs0 = rng.standard_normal((B, 98)).astype(np.float32)
    act0 = rng.standard_normal((B, 12)).astype(np.float32)
    vel0 = rng.standard_normal((B, 3)).astype(np.float32)
    raw = _raw_bytes(g, rng.integers(0, n_g, B), rng.random(B) < 0.1)
    raw.view(RAW_DT)["joy_valid"][::3] = 0           # a third of the robots keep their last joystick command
    d_raw = torch.from_numpy(raw).cuda()
    pb = PolicyBatch(model_path)
    try:
        def step(prec):
            d_obs = torch.from_numpy(obs0).cuda(); d_act = torch.from_numpy(act0).cuda(); d_vel = torch.from_numpy(vel0).cuda()
            d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
            pb.step_device(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(), B, prec)
            torch.cuda.synchronize()
            return d_obs.cpu().numpy(), d_vel.cpu().numpy(), d_act.cpu().numpy(), d_q.cpu().numpy(), pb.last_launches()
        obs_ref, vel_ref, act_ref, q_ref, n_ref = step(capi.PREC_FP32)
        assert n_ref > 1                               # assembly + policy launches
        for rep in range(3):
            obs, vel, act, q, n = step(capi.PREC_FP16)
            assert n == 1                              # ONE launch
            assert np.array_equal(bits(obs), bits(obs_ref)), rep
            assert np.array_equal(bits(vel), bits(vel_ref)), rep
            assert np.abs(act - act_ref).max() <= 5e-2, rep          # a tail statistic over 1.2 M actions of N(0,1) rows; precision is tested elsewhere
            exp_q, _, _ = oracle.joint_targets(act, raw.view(RAW_DT)["button0"].reshape(B, 1))
            assert np.array_equal(q.view(np.uint64), exp_q.view(np.uint64)), rep
    finally:
        pb.close()


def test_fleet_shards_rows_over_handles(torch_cuda, model_path, golden_loop):
    """One process, several handles, one host thread each: the result equals a single handle's, row for row.  With one
    GPU visible both shards run on device 0; with more the shards run on different devices."""
    torch = torch_cuda
    ndev = torch.cuda.device_count()
    devices = (0, 1) if ndev >= 2 else (0, 0)
    X = oracle.make_obs_d1(100_001, 98, seed=21)
    one = PolicyBatch(model_path)
    fl = Fleet(model_path, devices=devices)
    try:
        ref = one.infer_host(X, None, capi.PREC_FP16)
        got = np.zeros_like(ref)
        fl.infer_host(X, got, capi.PREC_FP16)
        assert np.array_equal(bits(got), bits(ref))
        g = golden_loop
        raw = _raw_bytes(g, [i % 400 for i in range(5001)])
        a1, a2 = np.zeros((5001, 12), np.float32), np.zeros((5001, 12), np.float32)
        for _ in range(3):
            one.step_host(raw, a1, None, capi.PREC_FP32)
            fl.step_host(raw, a2, None, capi.PREC_FP32)
            assert np.array_equal(bits(a1), bits(a2))
    finally:
        fl.close(); one.close()


def test_one_thread_two_devices(torch_cuda, model_path, golden):
    """The dynamic shared memory opt-in is a per-device function attribute: a second handle on another device, driven
    from the same host thread, must launch the tcgen05 kernels as well (regression for a cache keyed by size only)."""
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    X = golden["d1_obs"]
    outs = []
    pbs = [PolicyBatch(model_path, device=d) for d in (0, 1)]
    try:
        for d, pb in enumerate(pbs):
            with torch.cuda.device(d):
                d_obs = torch.from_numpy(X).to(f"cuda:{d}"); d_act = torch.zeros((X.shape[0], 12), device=f"cuda:{d}")
                for prec in (capi.PREC_FP16, capi.PREC_FP32):
                    pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), X.shape[0], prec)
                    torch.cuda.synchronize(d)
                outs.append(d_act.cpu().numpy())
        assert np.array_equal(bits(outs[0]), bits(outs[1]))
    finally:
        for pb in pbs:
            pb.close()


def test_relu_policy_with_observation_normaliser_all_paths(torch_cuda, tmp_path):
    """SURVEY 8f-4: a Relu policy with a Sub/Div observation normaliser in the graph (folded by the reader) agrees with
    the oracle, which evaluates the graph as written, on the fp32 path (1e-5), the tcgen05 path and batch-1 act()."""
    from go2_onnx_controller_b200 import ONNXActor
    from oracle import onnx_mini
    torch = torch_cuda
    rng = np.random.default_rng(8)
    dims = (60, 128, 128, 128, 12)
    ws = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for k, n in zip(dims[:-1], dims[1:])]
    bs = [rng.normal(0, 0.2, n).astype(np.float32) for n in dims[1:]]
    mean, std = rng.normal(0, 2, 60).astype(np.float32), rng.uniform(0.5, 3, 60).astype(np.float32)
    path = tmp_path / "norm_relu.onnx"
    path.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0, act_op="Relu", pre=[("Sub", mean), ("Div", std)]))
    pol = oracle.load_policy(str(path))
    X = (rng.normal(0, 1, (1500, 60)) * std + mean).astype(np.float32)
    ref = oracle.forward(pol, X)
    pb = PolicyBatch(str(path))
    try:
        d_obs = torch.from_numpy(X).cuda(); d_act = torch.zeros((1500, 12), device="cuda")
        for prec, tol in ((capi.PREC_FP32, 1e-5), (capi.PREC_FP16, 1e-2), (capi.PREC_BF16, 7e-2)):
            pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), 1500, prec)
            torch.cuda.synchronize()
            err = (np.abs(d_act.cpu().numpy() - ref) / np.maximum(1, np.abs(ref))).max()
            assert err <= tol, (prec, err)
    finally:
        pb.close()
    obs, act = np.zeros(60, np.float32), np.zeros(12, np.float32)
    a = ONNXActor(str(path), obs, act)
    try:
        for i in range(5):
            obs[:] = X[i]
            a.act()
            assert (np.abs(act - ref[i]) / np.maximum(1, np.abs(ref[i]))).max() <= 1e-5
    finally:
        a.close()


def _scaled_operands(pol, X):
    """The fp16 kernel's Gemm operands in its own (base-2 exponent) domain: the observation, then every hidden
    activation h' = log2(e) * elu(z), fp64 evaluation -- what cvt.rn.satfinite.f16x2 sees, up to rounding."""
    ops = [X.astype(np.float64)]
    h = X.astype(np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        for layer in pol.layers[:-1]:
            z = h @ layer.weight.astype(np.float64).T + layer.bias.astype(np.float64)
            h = oracle.elu(z, layer.elu_alpha)
            ops.append(h * np.log2(np.e))
    return ops


def test_fp16_saturation_is_counted_and_clean_rows_clip_like_the_reference(torch_cuda, model_path, golden, policy):
    """fp16 operands saturate at +-65504 where the fp32 reference does not (the x3000 stress set D3 reaches 1e6).
    GO2P_F_SAT_COUNT reports how many (row, 32-column operand block) pairs were clipped; on the rows the oracle
    predicts clean, the clip / mask decisions (controller.cpp:217-223) are the reference's."""
    torch = torch_cuda
    pb = PolicyBatch(model_path)
    try:
        # realistic observations never saturate: the counter stays at zero
        X2 = golden["d2_obs"]
        d_obs = torch.from_numpy(X2).cuda(); d_act = torch.zeros((X2.shape[0], 12), device="cuda")
        pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), X2.shape[0], capi.PREC_FP16, 0, None, None, capi.F_SAT_COUNT)
        assert pb.saturation_count() == 0
        # stress set x4 (its own activations stay below 31k): finite rows only -- NaN / Inf rows are covered by the
        # NaN-propagation test.  An operand block certainly saturates if it exceeds the format in the FIRST stage where
        # the row saturates at all (everything upstream of it is then exactly what the oracle predicts).
        X, b0 = golden["d3_obs"], golden["d3_button0"]
        fin = np.isfinite(X).all(axis=1)
        X, b0 = np.ascontiguousarray(X[fin] * np.float32(4.0)), np.ascontiguousarray(b0[fin])
        ops = _scaled_operands(policy, X)
        clean = np.ones(X.shape[0], bool)
        undecided = np.ones(X.shape[0], bool)          # rows not yet saturated in an earlier stage
        certain = 0
        for o in ops:
            pad = np.zeros((o.shape[0], 128)); pad[:, : o.shape[1]] = np.abs(o)
            blk = pad.reshape(o.shape[0], 4, 32).max(axis=2)          # per (row, 32-column block)
            certain += int((blk[undecided] > 66000).sum())
            undecided &= (blk < 65000).all(axis=1)
            clean &= (blk < 60000).all(axis=1)
        assert certain > 50 and clean.sum() > 20, (certain, clean.sum())
        d_obs = torch.from_numpy(X).cuda(); d_act = torch.zeros((X.shape[0], 12), device="cuda")
        d_b = torch.from_numpy(b0.astype(np.int32)).cuda()
        pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), X.shape[0], capi.PREC_FP16, 0, d_b.data_ptr(), None,
                        capi.F_CLAMP_MASK | capi.F_SAT_COUNT)
        n = pb.saturation_count()
        assert certain <= n <= int((~clean).sum()) * 16, (certain, n)
        assert pb.saturation_count() == 0                             # reading resets
        # the clean rows alone: nothing is counted
        Xc = np.ascontiguousarray(X[clean]); d_c = torch.from_numpy(Xc).cuda(); d_ac = torch.zeros((Xc.shape[0], 12), device="cuda")
        pb.infer_device(d_c.data_ptr(), d_ac.data_ptr(), Xc.shape[0], capi.PREC_FP16, 0, None, None, capi.F_SAT_COUNT)
        assert pb.saturation_count() == 0
        # rows without any clipped operand: same clip / mask decisions as the fp64 oracle, away from the clip edge
        got = d_act.cpu().numpy()[clean]
        ref = oracle.forward(policy, X[clean])
        exp = oracle.clamp_mask(ref.astype(np.float32), b0[clean][:, None])
        decided = (np.abs(np.abs(ref) - 1000) > 50.0)
        assert np.array_equal(np.abs(got[decided]) == 1000, np.abs(exp[decided]) == 1000)
        assert np.array_equal(got[decided] == 0, exp[decided] == 0)
        assert np.array_equal(np.signbit(got[decided]), np.signbit(exp[decided]))
    finally:
        pb.close()
