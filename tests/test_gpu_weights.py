"""Replacing a live handle's policy weights (go2p_set_weights, go2p_set_weights_host, go2p_fleet_set_weights_host).

Model B is the bundled policy with seeded noise, written to an .onnx by the test-side writer.  A handle created from the
bundled model and updated to B must compute exactly what a handle created from B's file computes, on every path and in
both forms (device tensors ordered on a stream, host arrays); robot state kept by the handle carries across the update."""
import numpy as np
import pytest

from go2_onnx_controller_b200 import Fleet, Go2Controller, ONNXActor, PolicyBatch, actor, capi
from oracle import onnx_mini, oracle

from test_gpu_parity import TOL_FP32, bits, raw_py, raw_struct
from test_gpu_resets import _raws
from test_gpu_round2 import CMD_DT

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

PRECS = [capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16]
MODES = [capi.B1_PERSISTENT, capi.B1_GRAPH, capi.B1_LAUNCH]
ALL_FLAGS = capi.F_CLAMP_MASK | capi.F_QDES | capi.F_MOTOR_CMD


def _noisy(layers, seed):
    rng = np.random.default_rng(seed)
    ws = [(L.weight * (1 + 0.1 * rng.standard_normal(L.weight.shape)) + 0.01 * rng.standard_normal(L.weight.shape))
          .astype(np.float32) for L in layers]
    bs = [(L.bias + 0.05 * rng.standard_normal(L.bias.shape)).astype(np.float32) for L in layers]
    return ws, bs


@pytest.fixture(scope="module")
def model_b(tmp_path_factory, policy):
    assert [L.elu_alpha for L in policy.layers] == [1.0, 1.0, 1.0, None]
    ws, bs = _noisy(policy.layers, seed=41)
    p = tmp_path_factory.mktemp("weights") / "b.onnx"
    p.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0))
    return ws, bs, str(p)


def _cuda(torch, ws, bs, mean=None, std=None):
    """The update's tensors on the device, made before anything is queued (a copy from pageable memory waits for the
    stream it is issued on)."""
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = ([t(w) for w in ws], None if bs is None else [t(b) for b in bs], t(mean), t(std))
    torch.cuda.synchronize()
    return out


def _update(torch, obj, ws, bs, form, mean=None, std=None):
    """obj's weights replaced in the host form, or in the device form from CUDA tensors on the current stream."""
    if form == "host":
        obj._hd.set_weights(ws, bs, mean, std, 0, host_only=False)
        return
    obj._hd.set_weights(*_cuda(torch, ws, bs, mean, std), torch.cuda.current_stream().cuda_stream, host_only=False)
    torch.cuda.synchronize()


def _infer(torch, pb, X, button, prec, flags):
    B = X.shape[0]
    d_obs = torch.from_numpy(X).cuda(); d_btn = torch.from_numpy(button).cuda()
    d_act = torch.zeros((B, pb.out_dim), device="cuda")
    d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
    d_cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)
    q = d_q.data_ptr() if flags & capi.F_QDES else None
    c = d_cmd.data_ptr() if flags & capi.F_MOTOR_CMD else None
    pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), B, prec, d_button0=d_btn.data_ptr(), d_qdes=q, flags=flags, d_cmd=c)
    torch.cuda.synchronize()
    return d_act.cpu().numpy(), d_q.cpu().numpy(), d_cmd.cpu().numpy()


def _inputs(golden, in_dim, big, seed):
    """333 rows (golden D3 stress rows first, two full tiles + a ragged one) and a multi-tile batch."""
    rng = np.random.default_rng(seed)
    if in_dim == 98:
        small = np.concatenate([golden["d3_obs"], golden["d1_obs"][:77]]).astype(np.float32)
        btn_small = np.concatenate([golden["d3_button0"], np.zeros(77)]).astype(np.int32)
    else:
        small = rng.standard_normal((333, in_dim)).astype(np.float32)
        btn_small = (rng.random(333) < 0.1).astype(np.int32)
    base = np.tile(small, (big // 333 + 1, 1))[:big]
    large = (base + 0.1 * rng.standard_normal(base.shape)).astype(np.float32)
    return [(small, btn_small), (large, (rng.random(big) < 0.1).astype(np.int32))]


def _same_batched(torch, got, ref, golden, big, flags_set, precs=PRECS, seed=0):
    for X, btn in _inputs(golden, got.in_dim, big, seed):
        for prec in precs:
            for flags in flags_set:
                a, r = _infer(torch, got, X, btn, prec, flags), _infer(torch, ref, X, btn, prec, flags)
                for x, y in zip(a, r):
                    assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (X.shape[0], prec, flags)


class _State:
    def __init__(self, torch, B, H=2):
        self.obs = torch.zeros((B, 49 * H), device="cuda"); self.vel = torch.zeros((B, 3), device="cuda")
        self.act = torch.zeros((B, 12), device="cuda"); self.q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
        self.cmd = torch.zeros((B, CMD_DT.itemsize), device="cuda", dtype=torch.uint8)

    def step(self, pb, d_raw, B, prec, d_rst=None, stream=0):
        pb.step_device_cmd(d_raw.data_ptr(), self.vel.data_ptr(), self.obs.data_ptr(), self.act.data_ptr(), self.q.data_ptr(),
                           self.cmd.data_ptr(), B, prec, stream=stream, d_reset=None if d_rst is None else d_rst.data_ptr())

    def numpy(self):
        return [t.cpu().numpy().view(np.uint8) for t in (self.obs, self.vel, self.act, self.q, self.cmd)]


def _same_states(a, b, *ctx):
    for x, y in zip(a.numpy(), b.numpy()):
        assert np.array_equal(x, y), ctx


# ------------------------------------------------------------------------------------------ 1. update == create
@pytest.mark.parametrize("form", ["device", "host"])
def test_update_equals_create_infer(torch_cuda, model_path, golden, model_b, form):
    """infer_device, fp32 / fp16 / bf16, without and with clamp/mask + q_des + motor commands, at B = 333 (golden D3
    stress rows) and B = 40,000 (many tiles per CTA): identical bytes."""
    ws, bs, path_b = model_b
    got, ref = PolicyBatch(model_path), PolicyBatch(path_b)
    try:
        _update(torch_cuda, got, ws, bs, form)
        _same_batched(torch_cuda, got, ref, golden, 40_000, (0, ALL_FLAGS))
    finally:
        got.close(); ref.close()


@pytest.mark.parametrize("form", ["device", "host"])
def test_update_equals_create_fused_step(torch_cuda, model_path, golden_loop, model_b, form):
    """The batched controller step (fused tensor-core step for fp16 / bf16, assembly + fp32 chain for fp32), four
    closed-loop steps on caller buffers, every other one with ~20 % resets: identical bytes in every buffer."""
    torch = torch_cuda
    ws, bs, path_b = model_b
    got, ref = PolicyBatch(model_path), PolicyBatch(path_b)
    rng = np.random.default_rng(3)
    try:
        _update(torch, got, ws, bs, form)
        for B in (333, 40_000):
            for prec in PRECS:
                sg, sr = _State(torch, B), _State(torch, B)
                for s in range(4):
                    raw, _ = _raws(golden_loop, rng, B)
                    d_raw = torch.from_numpy(raw).cuda()
                    d_rst = torch.from_numpy(rng.random(B) < 0.2).cuda() if s % 2 else None
                    sg.step(got, d_raw, B, prec, d_rst); sr.step(ref, d_raw, B, prec, d_rst)
                    torch.cuda.synchronize()
                    _same_states(sg, sr, B, prec, s)
    finally:
        got.close(); ref.close()


@pytest.mark.parametrize("form", ["device", "host"])
def test_update_equals_create_host_step_and_fleet(torch_cuda, model_path, golden_loop, model_b, form):
    """step_host (two 65,536-row pipeline chunks) from zeroed state, fp16 then fp32; Fleet.step_host (host form only:
    two devices, or two handles on one)."""
    torch = torch_cuda
    ws, bs, path_b = model_b
    rng = np.random.default_rng(5)
    B = 70_000
    got, ref = PolicyBatch(model_path), PolicyBatch(path_b)
    try:
        _update(torch, got, ws, bs, form)
        a1, a2 = np.zeros((B, 12), np.float32), np.zeros((B, 12), np.float32)
        c1, c2 = np.zeros((B, CMD_DT.itemsize), np.uint8), np.zeros((B, CMD_DT.itemsize), np.uint8)
        for s, prec in enumerate([capi.PREC_FP16] * 3 + [capi.PREC_FP32] * 2):
            raw, _ = _raws(golden_loop, rng, B)
            got.step_host(raw, a1, c1, prec); ref.step_host(raw, a2, c2, prec)
            assert np.array_equal(bits(a1), bits(a2)), s
            assert np.array_equal(c1, c2), s
    finally:
        got.close(); ref.close()
    if form != "host":
        return
    devices = (0, 1) if torch.cuda.device_count() >= 2 else (0, 0)
    Bf = 5001
    fg, fr = Fleet(model_path, devices=devices), Fleet(path_b, devices=devices)
    try:
        fg.set_weights(ws, bs)
        a1, a2 = np.zeros((Bf, 12), np.float32), np.zeros((Bf, 12), np.float32)
        for s in range(3):
            raw, _ = _raws(golden_loop, rng, Bf)
            fg.step_host(raw, a1, None, capi.PREC_FP16); fr.step_host(raw, a2, None, capi.PREC_FP16)
            assert np.array_equal(bits(a1), bits(a2)), s
        with pytest.raises(TypeError):
            fg.set_weights([torch.from_numpy(w).cuda() for w in ws], None)
    finally:
        fg.close(); fr.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("form", ["device", "host"])
def test_update_equals_create_batch1(torch_cuda, model_path, golden, golden_loop, model_b, mode, form):
    """ONNXActor.act (updated after its kernel has served a request, so a resident kernel is stopped and relaunched)
    and Go2Controller.step (30 closed-loop steps from the initial state) in every batch-1 mode: identical bits."""
    ws, bs, path_b = model_b
    oa, aa, orf, ar = (np.zeros(98, np.float32), np.zeros(12, np.float32), np.zeros(98, np.float32), np.zeros(12, np.float32))
    got, ref = ONNXActor(model_path, oa, aa, b1_mode=mode), ONNXActor(path_b, orf, ar, b1_mode=mode)
    try:
        got.act()
        _update(torch_cuda, got, ws, bs, form)
        for x in np.concatenate([golden["kat_obs"], golden["d1_obs"][:32]]):
            oa[:] = x; orf[:] = x
            got.act(); ref.act()
            assert np.array_equal(bits(aa), bits(ar))
    finally:
        got.close(); ref.close()
    cg, cr = Go2Controller(model_path, b1_mode=mode), Go2Controller(path_b, b1_mode=mode)
    try:
        _update(torch_cuda, cg, ws, bs, form)
        for i in range(30):
            o1, o2 = cg.step(raw_struct(golden_loop, i)), cr.step(raw_struct(golden_loop, i))
            for f in ("observation", "action_raw", "action", "q_des"):
                assert bytes(getattr(o1, f)) == bytes(getattr(o2, f)), (i, f)
            assert (o1.kp, o1.kd) == (o2.kp, o2.kd)
    finally:
        cg.close(); cr.close()


# ------------------------------------------------------------------------------------------ 2. wide policy
@pytest.mark.parametrize("form", ["device", "host"])
def test_wide_policy_update_equals_create(torch_cuda, tmp_path, wide_model_path, golden, form):
    """245-1024-512-256-12 (per-layer tcgen05 GEMMs with blocked weight tiles): a second seeded policy, fp32 / fp16 /
    bf16 at B = 333 and 20,000, with clamp/mask + q_des."""
    ws, bs = onnx_mini.make_wide_policy(seed=6)
    p = tmp_path / "wide_b.onnx"
    p.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0, batch="batch"))
    got, ref = PolicyBatch(wide_model_path), PolicyBatch(str(p))
    try:
        assert got.info.tensor_core_path == 1
        _update(torch_cuda, got, ws, bs, form)
        _same_batched(torch_cuda, got, ref, golden, 20_000, (capi.F_CLAMP_MASK | capi.F_QDES,), seed=1)
    finally:
        got.close(); ref.close()


# ------------------------------------------------------------------------------------------ 3. normaliser
@pytest.mark.parametrize("form", ["device", "host"])
def test_normaliser_update_equals_sub_div_prefix(torch_cuda, tmp_path, model_path, golden, golden_loop, model_b, form):
    """set_weights(B, mean, std) against a handle created from B with a Sub(mean) -> Div(std) prefix: the batched
    inference paths and the fused step, identical bytes."""
    torch = torch_cuda
    ws, bs, _ = model_b
    rng = np.random.default_rng(23)
    mean = (0.5 * rng.standard_normal(98)).astype(np.float32)
    std = rng.uniform(0.3, 3.0, 98).astype(np.float32)
    p = tmp_path / "norm.onnx"
    p.write_bytes(onnx_mini.write_mlp_onnx(ws, bs, 1.0, pre=[("Sub", mean), ("Div", std)]))
    got, ref = PolicyBatch(model_path), PolicyBatch(str(p))
    try:
        _update(torch, got, ws, bs, form, mean, std)
        _same_batched(torch, got, ref, golden, 40_000, (0, ALL_FLAGS), seed=2)
        B = 5000
        for prec in (capi.PREC_FP32, capi.PREC_FP16):
            sg, sr = _State(torch, B), _State(torch, B)
            for s in range(3):
                raw, _ = _raws(golden_loop, rng, B)
                d_raw = torch.from_numpy(raw).cuda()
                sg.step(got, d_raw, B, prec); sr.step(ref, d_raw, B, prec)
                torch.cuda.synchronize()
                _same_states(sg, sr, prec, s)
    finally:
        got.close(); ref.close()


# ------------------------------------------------------------------------------------------ 4. ordering
def test_step_update_step_on_one_stream(torch_cuda, model_path, policy, golden_loop, model_b):
    """fp16 fused step (A) -> set_weights(B) -> step -> set_weights(A) -> step, all queued on one torch stream with no
    host synchronisation; the step after each update is the tensor-core launch without programmatic serialization.
    Each step's buffers equal the reference handles' (A, B, A) run of the same sequence."""
    torch = torch_cuda
    ws, bs, path_b = model_b
    wa, ba = [L.weight for L in policy.layers], [L.bias for L in policy.layers]
    B = 100_077
    rng = np.random.default_rng(29)
    raws = [torch.from_numpy(_raws(golden_loop, rng, B)[0]).cuda() for _ in range(3)]
    got, ref_a, ref_b = PolicyBatch(model_path), PolicyBatch(model_path), PolicyBatch(path_b)
    try:
        st = torch.cuda.Stream()
        sg = _State(torch, B)
        tb, ta = _cuda(torch, ws, bs), _cuda(torch, wa, ba)
        snaps = []
        with torch.cuda.stream(st):
            sid = st.cuda_stream
            sg.step(got, raws[0], B, capi.PREC_FP16, stream=sid)
            snaps.append([t.clone() for t in (sg.obs, sg.vel, sg.act, sg.q, sg.cmd)])
            got.set_weights(*tb, stream=sid)
            sg.step(got, raws[1], B, capi.PREC_FP16, stream=sid)
            snaps.append([t.clone() for t in (sg.obs, sg.vel, sg.act, sg.q, sg.cmd)])
            got.set_weights(*ta, stream=sid)
            sg.step(got, raws[2], B, capi.PREC_FP16, stream=sid)
            snaps.append([t.clone() for t in (sg.obs, sg.vel, sg.act, sg.q, sg.cmd)])
        st.synchronize()
        sr = _State(torch, B)
        for s, h in enumerate((ref_a, ref_b, ref_a)):
            sr.step(h, raws[s], B, capi.PREC_FP16)
            torch.cuda.synchronize()
            for x, y in zip(snaps[s], sr.numpy()):
                assert np.array_equal(x.cpu().numpy().view(np.uint8), y), s
    finally:
        got.close(); ref_a.close(); ref_b.close()


def test_async_device_update_then_host_step_and_batch1_step(torch_cuda, model_path, golden_loop, model_b):
    """A device-form update queued behind ~20 ms of other work on a torch stream, followed at once (no host sync) by
    step_host and, on another handle, by Go2Controller.step: both already compute with B."""
    torch = torch_cuda
    ws, bs, path_b = model_b
    rng = np.random.default_rng(31)
    B = 70_000
    raw, _ = _raws(golden_loop, rng, B)
    st = torch.cuda.Stream()
    tb = _cuda(torch, ws, bs)
    got, ref = PolicyBatch(model_path), PolicyBatch(path_b)
    try:
        with torch.cuda.stream(st):
            torch.cuda._sleep(40_000_000)
            got.set_weights(*tb, stream=st.cuda_stream)
        a1, a2 = np.zeros((B, 12), np.float32), np.zeros((B, 12), np.float32)
        got.step_host(raw, a1, None, capi.PREC_FP16)
        ref.step_host(raw, a2, None, capi.PREC_FP16)
        assert np.array_equal(bits(a1), bits(a2))
    finally:
        got.close(); ref.close()
    for mode in MODES:
        cg, cr = Go2Controller(model_path, b1_mode=mode), Go2Controller(path_b, b1_mode=mode)
        try:
            with torch.cuda.stream(st):
                torch.cuda._sleep(40_000_000)
                cg._hd.set_weights(*tb, st.cuda_stream, host_only=False)
            for i in range(10):
                o1, o2 = cg.step(raw_struct(golden_loop, i)), cr.step(raw_struct(golden_loop, i))
                assert bytes(o1.action_raw) == bytes(o2.action_raw), (mode, i)
                assert bytes(o1.observation) == bytes(o2.observation), (mode, i)
        finally:
            cg.close(); cr.close()


# ------------------------------------------------------------------------------------------ 5. state survives
@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16])
def test_host_step_state_survives_an_update(torch_cuda, model_path, golden_loop, model_b, prec):
    """step_host robots keep history, joystick command and previous action across an update: six steps with the
    update before the fourth equal the device-form step over caller buffers run by A for three steps, then by B."""
    torch = torch_cuda
    ws, bs, path_b = model_b
    rng = np.random.default_rng(37)
    B = 70_000
    host, dev_a, dev_b = PolicyBatch(model_path), PolicyBatch(model_path), PolicyBatch(path_b)
    try:
        sd = _State(torch, B)
        h_act, h_cmd = np.zeros((B, 12), np.float32), np.zeros((B, CMD_DT.itemsize), np.uint8)
        for s in range(6):
            if s == 3:
                host.set_weights(ws, bs)
            raw, _ = _raws(golden_loop, rng, B)
            mask = rng.random(B) < 0.1
            host.step_host(raw, h_act, h_cmd, prec, reset=mask)
            sd.step(dev_a if s < 3 else dev_b, torch.from_numpy(raw).cuda(), B, prec, torch.from_numpy(mask).cuda())
            torch.cuda.synchronize()
            assert np.array_equal(bits(h_act), bits(sd.act.cpu().numpy())), s
            assert np.array_equal(h_cmd, sd.cmd.cpu().numpy()), s
    finally:
        host.close(); dev_a.close(); dev_b.close()


@pytest.mark.parametrize("mode", MODES)
def test_batch1_history_survives_an_update(torch_cuda, model_path, policy, golden_loop, model_b, mode):
    """Go2Controller: 40 closed-loop steps, the weights replaced (host form) before step 20 while the controller runs.
    Against the oracle's controller_step with A's forward, then B's: the observation (history included) bit-exact but
    gravity <= 1 ulp, published action and q_des bit-exact, raw action within the fp32 tolerance of the right policy."""
    ws, bs, path_b = model_b
    pol_b = oracle.load_policy(path_b)
    ctl = Go2Controller(model_path, b1_mode=mode)
    st = oracle.ControllerState(H=2)
    try:
        for i in range(40):
            if i == 20:
                ctl.set_weights(ws, bs)
            pol = policy if i < 20 else pol_b
            out = ctl.step(raw_struct(golden_loop, i))
            d_obs = np.frombuffer(out.observation, np.float32, 98).copy()
            d_raw = np.frombuffer(out.action_raw, np.float32, 12).copy()
            d_act = np.frombuffer(out.action, np.float32, 12).copy()
            so = oracle.controller_step(pol, st, raw_py(golden_loop, i), np.float64, act_fn=lambda o: d_raw)
            assert np.abs(bits(d_obs[:6]).astype(np.int64) - bits(so.obs[:6]).astype(np.int64)).max() <= 1, i
            assert np.array_equal(bits(d_obs[6:]), bits(so.obs[6:])), i
            assert np.array_equal(bits(d_act), bits(so.action)), i
            assert np.array_equal(np.frombuffer(out.q_des, np.float64, 12), so.q_des), i
            ref = oracle.forward(pol, d_obs, np.float64)
            assert (np.abs(d_raw - ref) / np.maximum(1, np.abs(ref))).max() <= TOL_FP32, i
            st.hist[0][:] = d_obs[:6]
    finally:
        ctl.close()


# ------------------------------------------------------------------------------------------ 6. errors
def test_rejected_updates_leave_the_handle_working(torch_cuda, model_path, golden, policy):
    """Wrong n_layers, a null weight pointer, a mean without std: GO2P_ERR_INVALID with a message, and the handle
    still computes exactly what a fresh handle of the same model computes."""
    ws = [L.weight for L in policy.layers]
    junk = [np.full_like(w, 7.0) for w in ws]
    got, ref = PolicyBatch(model_path), PolicyBatch(model_path)
    try:
        lib, h = got._hd.lib, got._hd.h
        t = [torch_cuda.from_numpy(w).cuda() for w in junk]
        assert lib.go2p_set_weights(h, actor._ptr_array(t), None, 3, None, None, None) == capi.ERR_INVALID
        assert b"n_layers" in lib.go2p_last_error()
        assert lib.go2p_set_weights_host(h, actor._ptr_array(junk[:3] + [None]), None, 4, None, None) == capi.ERR_INVALID
        assert b"null weight pointer" in lib.go2p_last_error()
        assert lib.go2p_set_weights_host(h, None, None, 4, None, None) == capi.ERR_INVALID
        mean = np.zeros(98, np.float32)
        assert lib.go2p_set_weights_host(h, actor._ptr_array(junk), None, 4, mean.ctypes.data, None) == capi.ERR_INVALID
        assert b"obs_mean and obs_std" in lib.go2p_last_error()
        with pytest.raises(ValueError):
            got.set_weights(junk[:3])
        _same_batched(torch_cuda, got, ref, golden, 2000, (ALL_FLAGS,), seed=3)
    finally:
        got.close(); ref.close()
