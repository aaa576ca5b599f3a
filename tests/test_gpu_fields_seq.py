"""T closed-loop controller steps from per-field sensor streams in one call (go2p_step_batch_fields_seq,
PolicyBatch.step_fields_seq).

Its contract is twin identity: the call leaves exactly the bytes that T calls of go2p_step_batch_fields leave on the
step-t slices of the fields and of the reset mask, with d_action copied to d_action_seq[t] and d_obs to d_obs_seq[t]
after each.  fp16 / bf16 at B % 16 == 0 take one launch (the observation history stays in shared memory for all T
steps); every other case steps T times.  The single step itself is checked against the oracle by test_gpu_fields.py,
test_gpu_resets.py and test_gpu_parity.py; one sequence is checked against the oracle here as well."""
import ctypes as C

import numpy as np
import pytest

from go2_onnx_controller_b200 import PolicyBatch, actor, capi
from oracle import oracle

from test_gpu_parity import TC_TOL, TOL_FP32, bits
from test_gpu_resets import _raw_py, _raws
from test_gpu_round2 import CMD_DT

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

PRECS = [capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16, capi.PREC_FP32_TC]


def _streams(torch, T, B, seed):
    """T*B rows of every field, step-major ([T,B,w]), drawn on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev = dict(device="cuda", generator=g)
    quat = torch.randn((T, B, 4), **dev)
    quat /= quat.norm(dim=-1, keepdim=True)
    return dict(quat=quat, gyro=torch.randn((T, B, 3), **dev), q=0.3 * torch.randn((T, B, 12), **dev),
                dq=2.0 * torch.randn((T, B, 12), **dev), axes=2.0 * torch.rand((T, B, 4), **dev) - 1.0,
                foot_force=torch.randint(0, 60, (T, B, 4), dtype=torch.int16, **dev),
                joy_valid=torch.rand((T, B), **dev) < 0.6,
                button0=(torch.rand((T, B), **dev) < 0.1).to(torch.uint8))


def _state(torch, B, in_dim, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(shape, device="cuda", generator=g) for shape in ((B, in_dim), (B, 3), (B, 12))]


def _mask(torch, kind, T, B, seed, state):
    """None, all zeros, or ~15 % resets per step; the state rows of robots reset at step 0 are NaN-poisoned."""
    if kind == "none":
        return None
    if kind == "zeros":
        return torch.zeros((T, B), device="cuda", dtype=torch.uint8)
    g = torch.Generator(device="cuda").manual_seed(seed)
    m = torch.rand((T, B), device="cuda", generator=g) < 0.15
    for x in state:
        x[m[0]] = float("nan")
    return m


def _fields_ptr(fields, t=None):
    return capi.RawFields(*[(fields[n] if t is None else fields[n][t]).data_ptr() for n, _ in actor.RAW_FIELDS])


def _outputs(torch, T, B, in_dim, on):
    """action_seq always; qdes_seq, cmd_seq and obs_seq when `on`."""
    z = dict(device="cuda")
    return dict(act=torch.full((T, B, 12), 7.0, **z),
                q=torch.full((T, B, 12), 7.0, dtype=torch.float64, **z) if on else None,
                cmd=torch.full((T, B, CMD_DT.itemsize), 7, dtype=torch.uint8, **z) if on else None,
                obs=torch.full((T, B, in_dim), 7.0, **z) if on else None)


def _ptr(t):
    return None if t is None else t.data_ptr()


def _seq(pb, fields, T, B, mask, state, out, prec, t0=0):
    """One go2p_step_batch_fields_seq call over steps t0..t0+T-1 of the streams; state (obs, vel, act) updated in place.
    out: the per-step outputs of these T steps.  Returns the launch count."""
    obs, vel, act = state
    f = _fields_ptr({n: fields[n][t0:t0 + T] for n in fields})
    rst = None if mask is None else mask[t0:t0 + T].data_ptr()
    capi.check(pb._hd.lib.go2p_step_batch_fields_seq(pb._hd.h, C.byref(f), T, rst, vel.data_ptr(), obs.data_ptr(),
                                                     act.data_ptr(), out["act"].data_ptr(), _ptr(out["q"]),
                                                     _ptr(out["cmd"]), _ptr(out["obs"]), B, prec, None))
    return pb.last_launches()


def _loop(torch, pb, fields, T, B, mask, state, out, prec):
    """The twin: T calls of go2p_step_batch_fields on the step-t slices, copies of action / obs after each."""
    obs, vel, act = state
    q_scratch = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
    launches = 0
    for t in range(T):
        q = out["q"][t] if out["q"] is not None else q_scratch
        rst = None if mask is None else mask[t].data_ptr()
        capi.check(pb._hd.lib.go2p_step_batch_fields(pb._hd.h, C.byref(_fields_ptr(fields, t)), rst, vel.data_ptr(),
                                                     obs.data_ptr(), act.data_ptr(), q.data_ptr(),
                                                     _ptr(None if out["cmd"] is None else out["cmd"][t]), B, prec,
                                                     None))
        launches += pb.last_launches()
        out["act"][t].copy_(act)
        if out["obs"] is not None:
            out["obs"][t].copy_(obs)
    return launches


def _same_bytes(torch, a, b, what):
    for k in a:
        if a[k] is None:
            assert b[k] is None
            continue
        assert torch.equal(a[k].contiguous().view(torch.uint8), b[k].contiguous().view(torch.uint8)), (what, k)


def _compare(torch, pb, fields, T, B, in_dim, kind, on, prec, seed, one_launch=None):
    """one_launch: whether the sequence takes the one-launch kernel (default: fp16 / bf16 at B % 16 == 0)."""
    state0 = _state(torch, B, in_dim, seed)
    mask = _mask(torch, kind, T, B, seed + 1, state0)
    s_ref = [x.clone() for x in state0]
    s_seq = [x.clone() for x in state0]
    o_ref, o_seq = _outputs(torch, T, B, in_dim, on), _outputs(torch, T, B, in_dim, on)
    n_ref = _loop(torch, pb, fields, T, B, mask, s_ref, o_ref, prec)
    n_seq = _seq(pb, fields, T, B, mask, s_seq, o_seq, prec)
    torch.cuda.synchronize()
    what = (kind, on)
    _same_bytes(torch, dict(obs=s_ref[0], vel=s_ref[1], act=s_ref[2]), dict(obs=s_seq[0], vel=s_seq[1], act=s_seq[2]),
                what)
    _same_bytes(torch, o_ref, o_seq, what)
    if one_launch is None:
        one_launch = prec in (capi.PREC_FP16, capi.PREC_BF16) and B % 16 == 0
    assert n_seq == (1 if one_launch else n_ref), what
    return s_seq


# B = 16: one ragged tile; 5,008: 39 full tiles + a ragged one; 131,072: full tiles only, odd and even tile counts per
# CTA.  1, 333 and 100,077 are not multiples of 16: the step loop.
@pytest.mark.parametrize("T", [1, 2, 7, 33])
@pytest.mark.parametrize("B", [1, 16, 333, 5_008, 100_077, 131_072])
@pytest.mark.parametrize("prec", PRECS)
def test_sequence_leaves_the_bytes_of_T_single_steps(torch_cuda, model_path, prec, B, T):
    torch = torch_cuda
    fields = _streams(torch, T, B, seed=1000 * T + B)
    pb = PolicyBatch(model_path)
    try:
        for i, (kind, on) in enumerate((("none", True), ("zeros", False), ("random", True), ("random", False))):
            s = _compare(torch, pb, fields, T, B, 98, kind, on, prec, seed=7 * i + B + T)
            assert torch.isfinite(s[2]).all(), kind
    finally:
        pb.close()


@pytest.mark.parametrize("B", [333, 336])
@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16, capi.PREC_BF16])
def test_sequence_against_the_oracle(torch_cuda, model_path, policy, golden_loop, prec, B):
    """test_gpu_parity.py's closed loop (6 steps) as one sequence call with obs_seq: every step against the restated
    publish() re-synchronised to the device's own published action.  Observation bit-exact (gravity <= 1 ulp), action
    within the precision's bound, q_des bit-exact, masked rows zero.  B = 336 takes the one-launch kernel (two full tiles
    and a ragged one), B = 333 the step loop."""
    torch = torch_cuda
    g = golden_loop
    T, H = 6, 2
    rng = np.random.default_rng(200 + prec + B)
    rvs = [_raws(g, rng, B)[1] for _ in range(T)]
    fields = {n: torch.from_numpy(np.ascontiguousarray(np.stack([rv[n] for rv in rvs]))).cuda()
              for n, _ in actor.RAW_FIELDS[:6]}
    fields["joy_valid"] = torch.from_numpy(np.stack([rv["joy_valid"] != 0 for rv in rvs])).cuda()
    fields["button0"] = torch.from_numpy(np.stack([(rv["button0"] != 0).astype(np.uint8) for rv in rvs])).cuda()
    d_obs, d_vel, d_act = (torch.zeros(s, device="cuda") for s in ((B, 98), (B, 3), (B, 12)))
    out = _outputs(torch, T, B, 98, True)
    pb = PolicyBatch(model_path)
    try:
        pb.step_fields_seq(**fields, vel_cmd=d_vel, obs=d_obs, action=d_act, action_seq=out["act"], qdes_seq=out["q"],
                           cmd_seq=out["cmd"], obs_seq=out["obs"], precision=prec)
        torch.cuda.synchronize()
        if prec != capi.PREC_FP32 and B % 16 == 0:
            assert pb.last_launches() == 1
    finally:
        pb.close()
    obs_s, act_s, q_s = out["obs"].cpu().numpy(), out["act"].cpu().numpy(), out["q"].cpu().numpy()
    tol = TOL_FP32 if prec == capi.PREC_FP32 else 1e-2 if prec == capi.PREC_FP16 else TC_TOL[capi.PREC_BF16]["d1"]
    states = [oracle.ControllerState(H=H) for _ in range(B)]
    masked = 0
    for t in range(T):
        obs, act, qd = obs_s[t], act_s[t], q_s[t]
        for b in range(B):
            raw = _raw_py(rvs[t], b)
            so = oracle.controller_step(policy, states[b], raw, np.float64,
                                        act_fn=lambda o: oracle.forward(policy, obs[b], np.float64))
            assert np.abs(bits(obs[b, :6]).astype(np.int64) - bits(so.obs[:6]).astype(np.int64)).max() <= 1, (t, b)
            assert np.array_equal(bits(obs[b, 6:]), bits(so.obs[6:])), (t, b)
            assert (np.abs(act[b] - so.action) / np.maximum(1, np.abs(so.action))).max() <= tol, (t, b)
            if raw.button0:
                masked += 1
                assert not act[b].any()
            exp_q, _, _ = oracle.joint_targets(act[b], raw.button0)
            assert np.array_equal(qd[b].view(np.uint64), exp_q.view(np.uint64)), (t, b)
            states[b].action = act[b].copy()
            states[b].hist[0][:] = obs[b, :6]
    assert masked > 20
    assert np.array_equal(d_obs.cpu().numpy(), obs_s[-1]) and np.array_equal(d_act.cpu().numpy(), act_s[-1])


@pytest.mark.parametrize("B", [131_072, 5_008, 1_000])
@pytest.mark.parametrize("prec", [capi.PREC_FP16, capi.PREC_BF16, capi.PREC_FP32])
def test_chained_sequences_equal_one_sequence(torch_cuda, model_path, prec, B):
    """seq(3) then seq(5) on the state it left == seq(8), every output and the final state, with random resets."""
    torch = torch_cuda
    T1, T2 = 3, 5
    fields = _streams(torch, T1 + T2, B, seed=B + 3)
    pb = PolicyBatch(model_path)
    try:
        state0 = _state(torch, B, 98, seed=B)
        mask = _mask(torch, "random", T1 + T2, B, B + 1, state0)
        whole, parts = [x.clone() for x in state0], [x.clone() for x in state0]
        o_whole, o_parts = _outputs(torch, T1 + T2, B, 98, True), _outputs(torch, T1 + T2, B, 98, True)
        _seq(pb, fields, T1 + T2, B, mask, whole, o_whole, prec)
        _seq(pb, fields, T1, B, mask, parts, {k: v[:T1] for k, v in o_parts.items()}, prec)
        _seq(pb, fields, T2, B, mask, parts, {k: v[T1:] for k, v in o_parts.items()}, prec, t0=T1)
        torch.cuda.synchronize()
        _same_bytes(torch, dict(obs=whole[0], vel=whole[1], act=whole[2]), dict(obs=parts[0], vel=parts[1], act=parts[2]),
                    "state")
        _same_bytes(torch, o_whole, o_parts, "outputs")
    finally:
        pb.close()


@pytest.mark.parametrize("prec", [capi.PREC_FP16, capi.PREC_BF16])
def test_launch_count_and_fallbacks(torch_cuda, model_path, prec):
    """One launch at B % 16 == 0; B = 5,000 and a field 16 bytes plus 4 off its boundary take the step loop, identical
    to T single steps either way."""
    torch = torch_cuda
    T = 4
    pb = PolicyBatch(model_path)
    try:
        fields = _streams(torch, T, 4096, seed=5)
        _compare(torch, pb, fields, T, 4096, 98, "random", True, prec, seed=6)
        assert pb.last_launches() == 1
        fields = _streams(torch, T, 5_000, seed=7)
        _compare(torch, pb, fields, T, 5_000, 98, "random", True, prec, seed=8)
        assert pb.last_launches() > 1
        fields = _streams(torch, T, 4096, seed=9)
        for name in ("quat", "foot_force", "button0"):
            t = fields[name]
            buf = torch.zeros(t.numel() + 32, device="cuda", dtype=t.dtype)
            off = 20 // t.element_size()
            moved = buf[off:off + t.numel()].view(t.shape)
            moved.copy_(t)
            assert moved.data_ptr() % 16 == 4
            _compare(torch, pb, dict(fields, **{name: moved}), T, 4096, 98, "random", True, prec, seed=10, one_launch=False)
            assert pb.last_launches() > 1, name
    finally:
        pb.close()


@pytest.mark.parametrize("prec", [capi.PREC_FP32, capi.PREC_FP16])
def test_wide_policy(torch_cuda, wide_model_path, prec):
    """The 245-1024-512-256-12 policy at H = 5 steps T times through the two-kernel chain, identical to single steps."""
    torch = torch_cuda
    T, B = 5, 336
    fields = _streams(torch, T, B, seed=11)
    pb = PolicyBatch(wide_model_path, history=5)
    try:
        _compare(torch, pb, fields, T, B, 245, "random", True, prec, seed=12, one_launch=False)
    finally:
        pb.close()


def test_empty_sequence_and_batch(torch_cuda, model_path):
    """T = 0 or B = 0 reads and writes nothing."""
    torch = torch_cuda
    B = 64
    pb = PolicyBatch(model_path)
    try:
        fields = _streams(torch, 2, B, seed=13)
        state = _state(torch, B, 98, seed=14)
        before = [x.clone() for x in state]
        out = _outputs(torch, 2, B, 98, True)
        for T, b in ((0, B), (2, 0)):
            f = _fields_ptr(fields)
            assert pb._hd.lib.go2p_step_batch_fields_seq(pb._hd.h, C.byref(f), T, None, state[1].data_ptr(),
                                                         state[0].data_ptr(), state[2].data_ptr(),
                                                         out["act"].data_ptr(), None, None, None, b, capi.PREC_FP16,
                                                         None) == capi.OK
        pb.step_fields_seq(**{n: t[:0] for n, t in fields.items()}, vel_cmd=state[1], obs=state[0], action=state[2],
                           action_seq=out["act"][:0], precision=capi.PREC_FP16)
        torch.cuda.synchronize()
        for x, y in zip(state, before):
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8))
        assert (out["act"] == 7.0).all()
    finally:
        pb.close()
