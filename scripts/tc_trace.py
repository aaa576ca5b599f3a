"""Timeline of one CTA of tc_mlp_kernel (trace build: -DGO2P_TC_TRACE, lib/libgo2policy_trace.so).
usage: tc_trace.py [rows] [first event] [count] [warps, comma separated]
GO2P_TRACE_STEP=1 traces the fused controller step; GO2P_TRACE_RESET=p adds a mask resetting a fraction p of the robots.
GO2P_TRACE_SEQ=T traces T steps from per-field streams in one launch (go2p_step_batch_fields_seq); GO2P_TRACE_SEQ=F the
single per-field step (go2p_step_batch_fields).  Every run also prints, per traced pool warp, the cycles per output job
(one output job per tile-step)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("GO2P_LIB", os.path.join(ROOT, "go2_onnx_controller_b200", "lib", "libgo2policy_trace.so"))
import numpy as np, torch
trace = torch.zeros(34 * 2048, dtype=torch.int64, device="cuda")
os.environ["GO2P_TC_TRACE_PTR"] = str(trace.data_ptr())
import go2_onnx_controller_b200 as pkg
from go2_onnx_controller_b200 import capi
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1_048_576
lo = int(sys.argv[2]) if len(sys.argv) > 2 else 320
cnt = int(sys.argv[3]) if len(sys.argv) > 3 else 64
warps = [int(w) for w in sys.argv[4].split(",")] if len(sys.argv) > 4 else [0, 16]
model, width = pkg.DEFAULT_MODEL, 98
if os.environ.get("GO2P_TIME_IN"):      # synthetic Go2-topology policy with another input width
    import tempfile
    from go2_onnx_controller_b200 import onnx_writer
    width = int(os.environ["GO2P_TIME_IN"])
    ws, bs = onnx_writer.wide_policy(seed=3, dims=(width, 128, 128, 128, 12))
    model = os.path.join(tempfile.mkdtemp(), "narrow.onnx")
    onnx_writer.write_policy(model, ws, bs)
pb = pkg.PolicyBatch(model)
d_obs = torch.randn((B, width), device="cuda"); d_act = torch.empty((B, 12), device="cuda")
FUSED = os.environ.get("GO2P_TRACE_STEP") == "1"      # trace the fused fleet step (go2p_step_batch) instead of the plain forward
if FUSED:
    import ctypes as C, bench
    arr = bench.synthetic_raw_states(capi, 4096, seed=3)
    raw_np = np.frombuffer(bytes(arr), np.uint8).reshape(4096, C.sizeof(capi.RawState))
    d_raw = torch.from_numpy(np.tile(raw_np, (B // 4096, 1)).copy()).cuda()
    d_obs = torch.zeros((B, 98), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
    d_act = torch.zeros((B, 12), device="cuda"); d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
    # GO2P_TRACE_RESET=p: the step with per-robot resets (go2p_step_batch_ex), a fraction p of the robots reset
    RESET = float(os.environ["GO2P_TRACE_RESET"]) if os.environ.get("GO2P_TRACE_RESET") else None
    d_rst = (torch.rand(B, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5)) < RESET) if RESET is not None else None
SEQ = os.environ.get("GO2P_TRACE_SEQ")
if SEQ:
    import ctypes as C
    from go2_onnx_controller_b200 import actor
    T = 1 if SEQ == "F" else int(SEQ)
    g = torch.Generator(device="cuda").manual_seed(5)
    fl = {n: (torch.rand((T, B) + ((w,) if w else ()), device="cuda", generator=g) * (60 if n == "foot_force" else 1)).to(
        torch.int16 if n == "foot_force" else torch.uint8 if w is None else torch.float32) for n, w in actor.RAW_FIELDS}
    f = capi.RawFields(*[fl[n].data_ptr() for n, _ in actor.RAW_FIELDS])
    d_obs = torch.zeros((B, 98), device="cuda"); d_vel = torch.zeros((B, 3), device="cuda")
    d_act = torch.zeros((B, 12), device="cuda"); d_q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
    d_aseq = torch.zeros((T, B, 12), device="cuda")
for _ in range(3):
    trace.zero_()
    torch.cuda.synchronize()
    if SEQ == "F":
        capi.check(pb._hd.lib.go2p_step_batch_fields(pb._hd.h, C.byref(f), None, d_vel.data_ptr(), d_obs.data_ptr(),
                                                     d_act.data_ptr(), d_q.data_ptr(), None, B, capi.PREC_FP16, None))
    elif SEQ:
        capi.check(pb._hd.lib.go2p_step_batch_fields_seq(pb._hd.h, C.byref(f), T, None, d_vel.data_ptr(), d_obs.data_ptr(),
                                                         d_act.data_ptr(), d_aseq.data_ptr(), None, None, None, B,
                                                         capi.PREC_FP16, None))
    elif FUSED:
        pb.step_device(d_raw.data_ptr(), d_vel.data_ptr(), d_obs.data_ptr(), d_act.data_ptr(), d_q.data_ptr(), B, capi.PREC_FP16,
                       d_reset=None if d_rst is None else d_rst.data_ptr())
    else:
        pb.infer_device(d_obs.data_ptr(), d_act.data_ptr(), B, capi.PREC_FP16)
    torch.cuda.synchronize()
t = trace.cpu().numpy().reshape(34, 2048)
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
np.save(os.path.join(ROOT, "gpurun_out", "tc_trace_raw.npy"), t)
names = {1: "C tma issue", 2: "C a_ready", 3: "C committed", 4: "W conv acquired", 6: "W E acquired", 7: "W arrived", 8: "W out acquired",
         9: "W out done", 10: "W raw landed", 11: "W terms updated", 12: "W quarter met", 15: "W fine"}
c0 = min(int(t[w, 1]) for w in range(17) if t[w, 2046] > 0)
for w in warps:
    n = int(t[w, 2046]); ev = t[w, 0:2 * n:2]; ck = t[w, 1:2 * n:2]
    print(f"--- warp {w}: {n} events, span {int(ck[-1] - ck[0])} cycles")
    outs = ck[(ev >> 8) == 9]
    if len(outs) > 2:
        print(f"    {np.diff(outs).mean() * 1.0:.0f} cycles per output job (median {np.median(np.diff(outs)):.0f}) over {len(outs)} jobs")
    prev = None
    for e, c in list(zip(ev, ck))[(lo if w < 16 else lo * 13 // 19):][:cnt]:
        e = int(e); k = e >> 8; l = (e >> 4) & 15; s = e & 3
        print(f"{int(c) - c0:9d} (+{(int(c) - prev) if prev else 0:5d}) {names.get(k, hex(e)):16s} slot {s} sub {l}")
        prev = int(c)
