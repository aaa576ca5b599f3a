"""Pins the restated observation assembly / action post-processing (A1-A6, A9, A11) and the ONNXActor wrapper
semantics to the reference's OWN code: onnx_controller/src/controller.cpp and onnx_inference/src/cpp/onnx_actor.cpp,
compiled from /root/reference against stub ROS / Eigen / ONNX-Runtime headers (oracle/Makefile -> oracle/_ref).
Inside that build Session::Run is the C fp32 restatement, so A7 itself stays "parity unpinned" (DESIGN.md)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import coracle, oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HAVE_REF = os.path.exists(coracle.REF_LIB_PATH)
NEEDS_REF = "needs oracle/_ref, which oracle/Makefile builds only where the reference sources are present"
MODEL_SHA256 = "9bdcb0f47be89417dbf3f7fb46522ecb3ec42ca65458a905f191aff933a18eae"   # the reference's model.onnx


@pytest.fixture
def ref_share_dir(model_path, tmp_path, monkeypatch):
    """The compiled controller reads <GO2_REF_ROOT>/onnx_inference/data/model.onnx (ament share directory stub): point
    it at a copy of the bundled model, which is the reference's file byte for byte, so no reference tree is needed."""
    data = open(model_path, "rb").read()
    assert hashlib.sha256(data).hexdigest() == MODEL_SHA256
    d = tmp_path / "onnx_inference" / "data"
    d.mkdir(parents=True)
    (d / "model.onnx").write_bytes(data)
    monkeypatch.setenv("GO2_REF_ROOT", str(tmp_path))


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _raw(g, i):
    return oracle.RawState(quat=g["raw_quat"][i], gyro=g["raw_gyro"][i], q=g["raw_q"][i], dq=g["raw_dq"][i],
                           foot_force=g["raw_foot_force"][i], axes=g["raw_axes"][i],
                           joy_valid=int(g["raw_joy_valid"][i]), button0=int(g["raw_button0"][i]))


def test_c_oracle_matches_committed_reference_trace(cmodel, golden_loop):
    """Always runs (also where /root/reference is absent): the C restatement, fp32 policy arithmetic, reproduces the
    trace recorded from the reference's compiled controller bit for bit -- observation layout and history, clamp,
    dead-man mask (incl. -0.0), q_des in double, kp/kd selection."""
    tr = np.load(os.path.join(GOLD, "ref_controller_trace.npz"))
    g = golden_loop
    cc = coracle.CController(cmodel, H=2)
    for i in range(tr["obs"].shape[0]):
        co = cc.step(coracle.raw_from_py(_raw(g, i)), use_f64=False)
        assert np.array_equal(bits(np.frombuffer(co.obs, np.float32, 98)), bits(tr["obs"][i])), i
        assert np.array_equal(bits(np.frombuffer(co.action, np.float32, 12)), bits(tr["action"][i])), i
        assert np.array_equal(np.frombuffer(co.q_des, np.float64, 12), tr["q_des"][i]), i
        assert (tr["kp"][i] == co.kp).all() and (tr["kd"][i] == co.kd).all(), i


def test_numpy_oracle_obs_and_post_match_reference_trace(policy, golden_loop):
    tr = np.load(os.path.join(GOLD, "ref_controller_trace.npz"))
    g = golden_loop
    st = oracle.ControllerState(H=2)
    for i in range(150):
        raw_action = None

        def act_fn(obs, _i=i):
            return oracle.forward(policy, obs, np.float32).astype(np.float32)

        so = oracle.controller_step(policy, st, _raw(g, i), np.float32, act_fn=act_fn)
        assert np.array_equal(bits(so.obs), bits(tr["obs"][i])), i
        # numpy's fp32 matmul may round differently from the C loop: compare the post-processing on the reference's action
        pub = tr["action"][i]
        st.action = pub.copy()
        qd, kp, kd = oracle.joint_targets(pub, int(g["raw_button0"][i]))
        assert np.array_equal(qd, tr["q_des"][i]) and float(kp) == tr["kp"][i][0] and float(kd) == tr["kd"][i][0]
        assert np.abs(so.action - pub).max() < 1e-4


@pytest.mark.skipif(not HAVE_REF, reason=NEEDS_REF)
def test_reference_controller_live_vs_oracle_and_fixture(cmodel, golden_loop, ref_share_dir):
    tr = np.load(os.path.join(GOLD, "ref_controller_trace.npz"))
    g = golden_loop
    rc = coracle.RefController()
    try:
        for i in range(200):
            axes = g["raw_axes"][i] if g["raw_joy_valid"][i] else np.zeros(0, np.float32)
            rc.feed(g["raw_quat"][i], g["raw_gyro"][i], g["raw_foot_force"][i], g["raw_q"][i].astype(np.float64),
                    g["raw_dq"][i].astype(np.float64), axes, [int(g["raw_button0"][i])])
            obs, act, qd, kp, kd = rc.step()
            assert np.array_equal(bits(obs), bits(tr["obs"][i])) and np.array_equal(bits(act), bits(tr["action"][i]))
            assert np.array_equal(qd, tr["q_des"][i])
    finally:
        rc.close()


@pytest.mark.skipif(not HAVE_REF, reason=NEEDS_REF)
def test_reference_controller_gates_and_params(golden_loop, ref_share_dir):
    """publish() is skipped while the robot is not ready / not safe (controller.cpp:158-171) and kp/kd follow the ROS
    parameters (controller.cpp:254-277); the dead-man button forces kp = 5 (controller.cpp:246)."""
    g = golden_loop
    rc = coracle.RefController()
    try:
        args = (g["raw_quat"][0], g["raw_gyro"][0], g["raw_foot_force"][0], g["raw_q"][0].astype(np.float64),
                g["raw_dq"][0].astype(np.float64), g["raw_axes"][0])
        rc.feed(*args, [0], ready=False)
        assert rc.step() is None
        rc.feed(*args, [0], safe=False)
        assert rc.step() is None
        rc.feed(*args, [0])
        obs, act, qd, kp, kd = rc.step()
        assert (kp == 28.0).all() and (kd == 0.5).all()
        assert rc.set_param("kp", 31.5) and rc.set_param("kd", 0.75) and not rc.set_param("bogus", 1.0)
        rc.feed(*args, [0])
        assert (rc.step()[3] == 31.5).all()
        rc.feed(*args, [1])
        obs, act, qd, kp, kd = rc.step()
        assert (kp == 5.0).all() and (kd == 0.75).all() and (act == 0).all()
    finally:
        rc.close()
