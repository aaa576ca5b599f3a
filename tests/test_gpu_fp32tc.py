"""GO2P_PREC_FP32_TC: fp32 accuracy on the tensor cores (every operand as three bf16 pieces, six products per K step).

Its contract is GO2P_PREC_FP32's against the fp64 oracle (assert_fp32_parity: |a - ref| <= 1e-5 * max(|ref|, 1) and row
rel-L2 <= 1e-5), with fp32's range (no saturation), the oracle's NaN pattern on +-Inf / NaN inputs, and results that do
not depend on batch size or entry point.  It is not bit-identical to GO2P_PREC_FP32 (another summation order), so
identities are checked between the new precision's own paths."""
import ctypes as C

import numpy as np
import pytest

from go2_onnx_controller_b200 import Fleet, PolicyBatch, capi
from oracle import coracle, onnx_mini, oracle

from test_gpu_parity import TOL_FP32, assert_fp32_parity, bits, run_batch
from test_gpu_resets import _poison
from test_gpu_round2 import CMD_DT, RAW_DT, _raw_bytes
from test_gpu_weights import _noisy, _update

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

TC32 = capi.PREC_FP32_TC
CH = 4 * 148 * 128                   # rows per pass of the per-layer GEMM chain


def _launches(B, n_layers=4):
    """one conversion launch + one GEMM launch per layer, per pass"""
    return (1 + n_layers) * ((B + CH - 1) // CH)


def _rel(y, ref):
    fin = np.isfinite(ref)
    return float((np.abs(y[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))).max())


@pytest.fixture(scope="module")
def pb(torch_cuda, model_path):
    p = PolicyBatch(model_path)
    yield p
    p.close()


@pytest.mark.parametrize("name", ["kat", "d1", "d2"])
def test_golden_sets_meet_the_fp32_contract(torch_cuda, pb, golden, name):
    y, _ = run_batch(torch_cuda, pb, golden[f"{name}_obs"], TC32)
    ref = golden[f"{name}_action_f64"]
    print(f"fp32_tc {name}: max rel err {_rel(y, ref):.3e}")
    assert_fp32_parity(y.astype(np.float64), ref)
    assert pb.last_launches() == _launches(len(y))


@pytest.mark.parametrize("B", [1, 2, 127, 128, 129, 255, 1000, 4096, 148 * 128 * 2 + 77, CH + 77])
def test_ragged_sizes(torch_cuda, pb, cmodel, B):
    X = oracle.make_obs_d1(B, 98, seed=B)
    y, _ = run_batch(torch_cuda, pb, X, TC32)
    assert_fp32_parity(y.astype(np.float64), cmodel.forward_f64(X, threads=8))
    assert pb.last_launches() == _launches(B)


def test_full_size_rows_are_batch_independent(torch_cuda, pb, cmodel):
    torch = torch_cuda
    B = 1_048_576
    g = torch.Generator(device="cuda").manual_seed(0)
    d_obs = torch.randn((B, 98), device="cuda", dtype=torch.float32, generator=g)
    d_act = torch.empty((B, 12), device="cuda", dtype=torch.float32)
    pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), B, TC32)
    torch.cuda.synchronize()
    idx = torch.randint(0, B, (3000,), device="cuda", generator=g)
    sub = d_obs[idx].contiguous()
    sub_act = torch.empty((3000, 12), device="cuda", dtype=torch.float32)
    pb.infer_device(sub.data_ptr(), sub_act.data_ptr(), 3000, TC32)
    torch.cuda.synchronize()
    assert torch.equal(d_act[idx].view(torch.int32), sub_act.view(torch.int32))
    assert_fp32_parity(sub_act.cpu().numpy().astype(np.float64), cmodel.forward_f64(sub.cpu().numpy(), threads=8))
    d_act2 = torch.empty_like(d_act)
    pb.infer_device(d_obs.data_ptr(), d_act2.data_ptr(), B, TC32)
    torch.cuda.synchronize()
    assert torch.equal(d_act.view(torch.int32), d_act2.view(torch.int32))


def test_stress_set_nan_pattern_clamp_and_published_values(torch_cuda, pb, golden):
    """D3 (x3000 rows, +-Inf and NaN entries): no piece saturates, +-Inf observations give the oracle's NaN pattern,
    and the A9 / A11 epilogue follows from the kernel's own raw action bit for bit."""
    X, b0 = golden["d3_obs"], golden["d3_button0"]
    raw, _ = run_batch(torch_cuda, pb, X, TC32)
    pub, qd = run_batch(torch_cuda, pb, X, TC32, button0=b0, flags=capi.F_CLAMP_MASK | capi.F_QDES)
    ref_raw = golden["d3_action_f64"]
    assert np.isinf(X).any() and np.isnan(X).any()
    assert np.array_equal(np.isnan(raw), np.isnan(ref_raw))
    assert (np.abs(raw) > 1000).mean() > 0.1
    exp_pub = oracle.clamp_mask(raw, b0)
    assert np.array_equal(bits(pub), bits(exp_pub))
    exp_qd, _, _ = oracle.joint_targets(exp_pub, b0[:, None])
    assert np.array_equal(qd.view(np.uint64), exp_qd.view(np.uint64))
    fin = np.isfinite(ref_raw)
    print(f"fp32_tc d3: max rel err {_rel(raw, ref_raw):.3e} on finite actions")
    assert _rel(raw, ref_raw) <= 2e-3            # the bound the CUDA-core fp32 path meets on this set
    gold = golden["d3_published_from_f64"]
    decided = fin & (np.abs(np.abs(ref_raw) - 1000) > 5.0) & ((np.abs(gold) == 1000) | (gold == 0))
    assert decided.sum() > 500
    assert np.array_equal(bits(pub[decided]), bits(gold[decided]))


def _fleet_bufs(torch, B):
    return dict(obs=torch.zeros((B, 98), device="cuda"), vel=torch.zeros((B, 3), device="cuda"),
                act=torch.zeros((B, 12), device="cuda"), q=torch.zeros((B, 12), device="cuda", dtype=torch.float64),
                cmd=torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8))


@pytest.mark.parametrize("resets", [False, True])
def test_closed_loop_fleet_step_from_records_and_fields(torch_cuda, model_path, policy, golden_loop, resets):
    """400 closed-loop steps of a 1,000-robot fleet on the device's own state.  Even robots replay the recorded trace
    (tests/golden/ref_controller_trace.npz, from the reference's compiled controller) and are checked against it, the
    odd ones take other recorded raw states.  Every step: the same bytes from records and from fields, two-kernel chain
    launch count, observations bit-exact against the oracle's assembly from the device's own previous action, actions
    within the fp32 contract of the fp64 oracle on the device's own observations.  With resets: ~5 % of the odd robots
    per step, their rows poisoned with NaN first."""
    import os
    torch = torch_cuda
    g = golden_loop
    tr = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_controller_trace.npz"))
    B, steps = 1000, g["obs"].shape[0]
    even = np.arange(B) % 2 == 0
    rng = np.random.default_rng(7)
    pb = PolicyBatch(model_path)
    bufs = {"rec": _fleet_bufs(torch, B), "fld": _fleet_bufs(torch, B)}
    st = oracle.ControllerState(H=2)
    max_err, max_drift = 0.0, 0.0
    try:
        for s in range(steps):
            idx = np.where(even, s, rng.integers(0, steps, B))
            raw = _raw_bytes(g, idx)
            d_raw = torch.from_numpy(raw).cuda()
            r = raw.view(RAW_DT).reshape(B)
            fields = {"quat": r["quat"], "gyro": r["gyro"], "q": r["q"], "dq": r["dq"], "axes": r["axes"],
                      "foot_force": r["foot_force"]}
            fields = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in fields.items()}
            fields["joy_valid"] = torch.from_numpy(r["joy_valid"] != 0).cuda()
            fields["button0"] = torch.from_numpy((r["button0"] != 0).astype(np.uint8)).cuda()
            mask = (~even) & (rng.random(B) < 0.05) if resets else None
            out = {}
            for src, b in bufs.items():
                d_rst = None
                if mask is not None:
                    _poison(torch, mask, b["obs"], b["vel"], b["act"])
                    d_rst = torch.from_numpy(mask).cuda()
                args = (b["vel"].data_ptr(), b["obs"].data_ptr(), b["act"].data_ptr(), b["q"].data_ptr(), b["cmd"].data_ptr(),
                        B, TC32, None)
                rst = None if d_rst is None else d_rst.data_ptr()
                lib, h = pb._hd.lib, pb._hd.h
                if src == "rec":
                    capi.check(lib.go2p_step_batch_ex(h, d_raw.data_ptr(), rst, *args))
                else:
                    f = capi.RawFields(*[fields[n].data_ptr() for n in ("quat", "gyro", "q", "dq", "axes", "foot_force",
                                                                         "joy_valid", "button0")])
                    capi.check(lib.go2p_step_batch_fields(h, C.byref(f), rst, *args))
                torch.cuda.synchronize()
                assert pb.last_launches() == 1 + _launches(B), s
                out[src] = [b[k].cpu().numpy() for k in ("obs", "vel", "act", "q", "cmd")]
            for x, y in zip(out["rec"], out["fld"]):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), s
            obs, _, act, qd, _ = out["rec"]
            # the trace robots are one robot: identical rows, checked against the oracle and the recorded trace
            assert np.array_equal(bits(obs[even]), np.broadcast_to(bits(obs[0]), obs[even].shape)), s
            so = oracle.controller_step(policy, st, oracle.RawState(
                quat=g["raw_quat"][s], gyro=g["raw_gyro"][s], q=g["raw_q"][s], dq=g["raw_dq"][s],
                foot_force=g["raw_foot_force"][s], axes=g["raw_axes"][s], joy_valid=int(g["raw_joy_valid"][s]),
                button0=int(g["raw_button0"][s])), np.float64, act_fn=lambda o: oracle.forward(policy, obs[0], np.float64))
            assert np.abs(bits(obs[0, :6]).astype(np.int64) - bits(so.obs[:6]).astype(np.int64)).max() <= 1, s
            assert np.array_equal(bits(obs[0, 6:]), bits(so.obs[6:])), s
            st.hist[0][:] = obs[0, :6]
            st.action = act[0].copy()
            ro = tr["obs"][s]
            assert np.array_equal(bits(obs[0, 6:66]), bits(ro[6:66])) and np.array_equal(bits(obs[0, 90:]), bits(ro[90:])), s
            assert np.abs(obs[0, 66:90] - ro[66:90]).max() <= 1e-4, s
            max_drift = max(max_drift, float(np.abs(act[0] - tr["action"][s]).max()))
            # every robot: the published action is clamp/mask of an action within the contract of its own observation
            ref = oracle.forward(policy, obs, np.float64)
            btn = r["button0"].reshape(B, 1) != 0
            exp = np.where(btn, 0.0, np.clip(ref, -1000, 1000))
            err = np.abs(act - exp) / np.maximum(1.0, np.abs(exp))
            max_err = max(max_err, float(err.max()))
            assert err.max() <= TOL_FP32, s
            exp_q, _, _ = oracle.joint_targets(act, r["button0"].reshape(B, 1))
            assert np.array_equal(qd.view(np.uint64), exp_q.view(np.uint64)), s
        print(f"fp32_tc fleet closed loop: {steps} steps, max rel err {max_err:.2e}, drift vs recorded trace {max_drift:.2e}")
        assert max_drift <= 1e-3
    finally:
        pb.close()


def test_host_pipeline_step_host_and_fleet_match_the_device_path(torch_cuda, model_path, golden_loop):
    torch = torch_cuda
    g = golden_loop
    X = oracle.make_obs_d1(200_001, 98, seed=9)
    B = 70_000                       # more than one 65,536-row pipeline chunk
    dev, host = PolicyBatch(model_path), PolicyBatch(model_path)
    fl = Fleet(model_path, devices=(0,))
    try:
        y_dev, _ = run_batch(torch, dev, X, TC32)
        assert np.array_equal(bits(host.infer_host(X, None, TC32)), bits(y_dev))
        y_fl = np.zeros_like(y_dev)
        fl.infer_host(X, y_fl, TC32)
        assert np.array_equal(bits(y_fl), bits(y_dev))
        d_obs = torch.zeros((B, 98), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
        d_act = torch.zeros((B, 12), device="cuda"); d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
        h_act = np.zeros((B, 12), np.float32); h_cmd = np.zeros((B, CMD_DT.itemsize), np.uint8)
        f_act = np.zeros((B, 12), np.float32); f_cmd = np.zeros((B, CMD_DT.itemsize), np.uint8)
        rng = np.random.default_rng(5)
        for s in range(3):
            raw = _raw_bytes(g, rng.integers(0, g["obs"].shape[0], B), rng.random(B) < 0.1)
            reset = rng.random(B) < 0.05 if s == 2 else None
            host.step_host(raw, h_act, h_cmd, TC32, reset=reset)
            fl.step_host(raw, f_act, f_cmd, TC32, reset=reset)
            d_raw = torch.from_numpy(raw).cuda()
            d_rst = None if reset is None else torch.from_numpy(reset).cuda().data_ptr()
            dev.step_device_cmd(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), None, d_cmd.data_ptr(),
                                B, TC32, d_reset=d_rst)
            torch.cuda.synchronize()
            assert np.array_equal(bits(h_act), bits(d_act.cpu().numpy())), s
            assert np.array_equal(h_cmd, d_cmd.cpu().numpy()), s
            assert np.array_equal(bits(f_act), bits(h_act)) and np.array_equal(f_cmd, h_cmd), s
    finally:
        fl.close(); dev.close(); host.close()


@pytest.mark.parametrize("form", ["device", "host"])
def test_set_weights_gives_the_bits_of_a_handle_created_from_the_tensors(torch_cuda, model_path, policy, tmp_path, form):
    torch = torch_cuda
    ws, bs = _noisy(policy.layers, seed=43)
    path = tmp_path / "b.onnx"
    path.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0))
    X = oracle.make_obs_d1(5000, 98, seed=3)
    upd, fresh = PolicyBatch(model_path), PolicyBatch(str(path))
    try:
        before, _ = run_batch(torch, upd, X, TC32)
        _update(torch, upd, ws, bs, form)
        y, _ = run_batch(torch, upd, X, TC32)
        y_fresh, _ = run_batch(torch, fresh, X, TC32)
        assert np.array_equal(bits(y), bits(y_fresh))
        assert not np.array_equal(bits(y), bits(before))
        assert_fp32_parity(y.astype(np.float64), coracle.CModel(str(path)).forward_f64(X, 8))
    finally:
        upd.close(); fresh.close()


def test_wide_policy(torch_cuda, wide_model_path):
    cm = coracle.CModel(wide_model_path)
    p = PolicyBatch(wide_model_path, history=5)
    try:
        for B in (1, 129, 3001, CH + 77):
            X = oracle.make_obs_d1(B, 245, seed=B)
            y, _ = run_batch(torch_cuda, p, X, TC32)
            ref = cm.forward_f64(X, 8)
            print(f"fp32_tc wide B={B}: max rel err {_rel(y, ref):.3e}")
            assert_fp32_parity(y.astype(np.float64), ref)
            assert p.last_launches() == _launches(B)
        y1, _ = run_batch(torch_cuda, p, X[CH - 100:CH + 200], TC32)
        assert np.array_equal(bits(y1), bits(y[CH - 100:CH + 200]))
        assert np.array_equal(bits(p.infer_host(X, None, TC32)), bits(y))
    finally:
        p.close()


def _model(tmp_path, dims, alpha, final_act, seed):
    rng = np.random.default_rng(seed)
    ws = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for k, n in zip(dims[:-1], dims[1:])]
    bs = [rng.normal(0, 0.2, n).astype(np.float32) for n in dims[1:]]
    path = tmp_path / f"m{len(dims)}_{dims[1]}.onnx"
    path.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, alpha, final_activation=final_act))
    return str(path)


def test_final_activation_model_and_unserved_shape(torch_cuda, tmp_path):
    path = _model(tmp_path, (64, 128, 12), 1.0, True, seed=204)
    p = PolicyBatch(path)
    try:
        X = np.random.default_rng(1).normal(0, 1, (1000, 64)).astype(np.float32)
        y, _ = run_batch(torch_cuda, p, X, TC32)
        assert_fp32_parity(y.astype(np.float64), coracle.CModel(path).forward_f64(X, 4))
        assert p.last_launches() == _launches(1000, 2)
    finally:
        p.close()
    path = _model(tmp_path, (98, 100, 12), 1.0, False, seed=7)        # hidden width not a multiple of 64
    p = PolicyBatch(path)
    try:
        with pytest.raises(capi.Go2PolicyError) as e:
            run_batch(torch_cuda, p, np.zeros((10, 98), np.float32), TC32)
        assert e.value.code == capi.ERR_UNSUPPORTED and "GO2P_PREC_FP32" in str(e.value)
        run_batch(torch_cuda, p, np.zeros((10, 98), np.float32), capi.PREC_FP32)     # the fp32 path still serves it
    finally:
        p.close()


def test_empty_batch_launches_nothing(torch_cuda, pb):
    y, _ = run_batch(torch_cuda, pb, np.zeros((0, 98), np.float32), TC32)
    assert y.shape == (0, 12) and pb.last_launches() == 0


def test_inf_input_meets_every_weight_piece_with_one_sign_and_no_zero(torch_cuda, tmp_path):
    """The non-finite rule of the weight split (DESIGN.md §3.3c).  Layer 0's weights on input column 0 are all negative;
    a third of them are exactly bf16 (their mid and lo pieces would be 0) and a third have 16 significand bits (their lo
    piece would be 0).  +Inf in that column makes every hidden unit -Inf in the reference, the ELU maps it to -alpha, and
    the action is finite.  A split with a zero piece (Inf * 0) or pieces of mixed sign (Inf - Inf) gives NaN there
    instead.  -Inf in that column, and NaN inputs, give NaN in the reference and here."""
    dims = (32, 128, 128, 12)
    rng = np.random.default_rng(17)
    ws = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for k, n in zip(dims[:-1], dims[1:])]
    bs = [rng.normal(0, 0.2, n).astype(np.float32) for n in dims[1:]]
    col = (-np.abs(ws[0][:, 0]) - 0.05).astype(np.float32).view(np.uint32)
    col[0::3] &= np.uint32(0xFFFF0000)
    col[1::3] &= np.uint32(0xFFFFFF00)
    ws[0][:, 0] = col.view(np.float32)
    path = tmp_path / "neg_column.onnx"
    path.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0))
    X = rng.normal(0, 1, (1000, dims[0])).astype(np.float32)
    X[0::4, 0] = np.inf
    X[1::4, 0] = -np.inf
    X[2::4, 5] = np.nan
    ref = coracle.CModel(str(path)).forward_f64(X, 4)
    assert np.isfinite(ref[0::4]).all() and np.isnan(ref[1::4]).all() and np.isnan(ref[2::4]).all()
    p = PolicyBatch(str(path))
    try:
        y, _ = run_batch(torch_cuda, p, X, TC32)
    finally:
        p.close()
    assert np.array_equal(np.isnan(y), np.isnan(ref))
    assert_fp32_parity(y.astype(np.float64), ref)
    assert_fp32_parity(y[0::4].astype(np.float64), ref[0::4])     # the +Inf rows alone, row rel-L2 included
