"""Cost of stepping a fleet from per-field device tensors: 1,048,576 robots, fp16, device buffers.

Times, with CUDA events, in one process, three variants alternately over several rounds (after a warm-up of each):
  records  go2p_step_batch_ex from go2p_raw_state records packed beforehand
  fields   go2p_step_batch_fields from the eight field tensors (quat, gyro, q, dq, axes, foot_force, joy_valid,
           button0), the form a GPU simulator keeps
  pack     what a caller without go2p_step_batch_fields does every step: copy the eight tensors into a uint8 [B,156]
           record buffer through views at the record's byte offsets (eight copy kernels), then go2p_step_batch_ex
and prints the card's name, power limit and maximum SM clock next to the fastest and median time of each.  The working
set (~0.6 GB) is far larger than L2, so every step reads its state from HBM.  Before timing, one step of each variant
from the same state is checked to leave the same bits.

    python scripts/fields_step_time.py [--rounds 7] [--iters 20]
"""
import argparse
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import go2_onnx_controller_b200 as pkg  # noqa: E402
from go2_onnx_controller_b200 import actor, capi  # noqa: E402
from reset_step_time import ROWS, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20, help="steps per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (the library has no CPU path)")

    pb = pkg.PolicyBatch(pkg.DEFAULT_MODEL)
    lib, h = pb._hd.lib, pb._hd.h
    rec_size = C.sizeof(capi.RawState)
    arr = bench.synthetic_raw_states(capi, 4096, seed=3)
    raw_np = np.frombuffer(bytes(arr), np.uint8).reshape(4096, rec_size)
    d_raw = torch.from_numpy(np.tile(raw_np, (ROWS // 4096, 1)).copy()).cuda()

    # the same values as field tensors, and the views a packing caller writes them through
    words = d_raw.view(torch.float32)                                    # [B, 39]
    ints = d_raw.view(torch.int32)
    ff_off = capi.RawState.foot_force.offset
    packed = torch.empty_like(d_raw)
    pw, pi = packed.view(torch.float32), packed.view(torch.int32)
    offsets = {name: getattr(capi.RawState, name).offset // 4 for name, _ in actor.RAW_FIELDS}
    fields, views = {}, {}
    for name, w in actor.RAW_FIELDS:
        o = offsets[name]
        if name == "foot_force":
            fields[name] = d_raw[:, ff_off:ff_off + 8].contiguous().view(torch.int16)
            views[name] = packed[:, ff_off:ff_off + 8].view(torch.int16)
        elif w is None:
            fields[name] = ints[:, o] != 0                                  # torch.bool
            views[name] = pi[:, o]
        else:
            fields[name] = words[:, o:o + w].contiguous()
            views[name] = pw[:, o:o + w]
    f = capi.RawFields(*[fields[name].data_ptr() for name, _ in actor.RAW_FIELDS])

    obs = torch.zeros((ROWS, 98), device="cuda"); vel = torch.zeros((ROWS, 3), device="cuda")
    act = torch.zeros((ROWS, 12), device="cuda"); q = torch.zeros((ROWS, 12), device="cuda", dtype=torch.float64)
    stream = torch.cuda.current_stream().cuda_stream
    P = capi.PREC_FP16

    def step_records(src):
        capi.check(lib.go2p_step_batch_ex(h, src.data_ptr(), None, vel.data_ptr(), obs.data_ptr(), act.data_ptr(),
                                          q.data_ptr(), None, ROWS, P, stream))

    def step_fields():
        capi.check(lib.go2p_step_batch_fields(h, C.byref(f), None, vel.data_ptr(), obs.data_ptr(), act.data_ptr(),
                                              q.data_ptr(), None, ROWS, P, stream))

    def pack():
        for name, _ in actor.RAW_FIELDS:
            views[name].copy_(fields[name])
        step_records(packed)

    variants = {"records": lambda: step_records(d_raw), "fields": step_fields, "pack": pack}

    outs = {}
    for k, fn in variants.items():                   # one step of each from the same (zero) state: the same bits
        for t in (obs, vel, act, q):
            t.zero_()
        fn()
        torch.cuda.synchronize()
        outs[k] = [t.cpu().numpy().view(np.uint8) for t in (obs, vel, act, q)]
    for k in ("fields", "pack"):
        assert all(np.array_equal(a, b) for a, b in zip(outs["records"], outs[k])), k

    for fn in variants.values():                       # warm-up: module load, smem opt-in, clocks
        for _ in range(5):
            fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = {k: [] for k in variants}
    for r in range(args.rounds):
        order = list(variants) if r % 2 == 0 else list(reversed(variants))
        for k in order:
            fn = variants[k]
            fn()
            e0.record()
            for _ in range(args.iters):
                fn()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.iters)

    print(f"card: {card()}")
    print(f"{ROWS:,} robots, fp16, {args.rounds} rounds x {args.iters} steps; ms per step: fastest / median")
    base = float(np.median(ms["records"]))
    for k, v in ms.items():
        med = float(np.median(v))
        print(f"  {k:<8} {min(v):.4f} / {med:.4f}  {100.0 * (med / base - 1.0):+.2f} % vs records (median)")
    pb.close()


if __name__ == "__main__":
    main()
