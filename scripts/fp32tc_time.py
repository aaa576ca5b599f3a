"""What GO2P_PREC_FP32_TC costs next to the CUDA-core fp32 path and the fp16 tensor-core path.

Times, with CUDA events, in one process, GO2P_PREC_FP32, GO2P_PREC_FP32_TC and GO2P_PREC_FP16 alternately over several
rounds (after a warm-up of each) on three workloads:
  infer  the bundled policy, 1,048,576 rows of N(0,1) observations (400 MB in, larger than the 126 MB L2)
  step   the batched controller step (go2p_step_batch_ex) for 1,048,576 robots on device buffers
  wide   the 245-1024-512-256-12 policy, 151,552 rows (two passes of the per-layer GEMM chain)
and prints the card's name, power limit and maximum SM clock next to the fastest and median time of each, the launch
count of one call, and the maximum relative error of FP32_TC against FP32 on the inference rows.

    python scripts/fp32tc_time.py [--rounds 7] [--iters 10]
"""
import argparse
import os
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import go2_onnx_controller_b200 as pkg  # noqa: E402
from go2_onnx_controller_b200 import capi, onnx_writer  # noqa: E402
from reset_step_time import ROWS, card  # noqa: E402

WIDE_ROWS = 2 * 4 * 148 * 128
PRECS = {"fp32": capi.PREC_FP32, "fp32_tc": capi.PREC_FP32_TC, "fp16": capi.PREC_FP16}


def time_variants(variants, rounds, iters):
    for fn in variants.values():                       # warm-up: module load, smem opt-in, scratch, clocks
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = {k: [] for k in variants}
    for r in range(rounds):
        for k in (list(variants) if r % 2 == 0 else list(reversed(variants))):
            fn = variants[k]
            fn()
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1) / iters)
    return ms


def report(title, ms, launches):
    print(title)
    for k, v in ms.items():
        print(f"  {k:<8} {min(v):.4f} / {float(np.median(v)):.4f} ms  ({launches[k]} launches)")
    tc, fp = float(np.median(ms["fp32_tc"])), float(np.median(ms["fp32"]))
    print(f"  fp32_tc is {fp / tc:.2f}x the CUDA-core fp32 path (medians)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10, help="calls per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (the library has no CPU path)")
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}")
    print(f"{args.rounds} rounds x {args.iters} calls; fastest / median per call")

    pb = pkg.PolicyBatch(pkg.DEFAULT_MODEL)
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = torch.randn((ROWS, 98), device="cuda", dtype=torch.float32, generator=g)
    outs = {k: torch.empty((ROWS, 12), device="cuda") for k in PRECS}

    def infer(k):
        return lambda: pb.infer_device(obs.data_ptr(), outs[k].data_ptr(), ROWS, PRECS[k], stream)

    variants = {k: infer(k) for k in PRECS}
    launches = {}
    for k, fn in variants.items():
        fn()
        launches[k] = pb.last_launches()
    torch.cuda.synchronize()
    a, b = outs["fp32_tc"].double(), outs["fp32"].double()
    rel = ((a - b).abs() / b.abs().clamp(min=1.0)).max().item()
    report(f"infer: bundled policy, {ROWS:,} rows (max rel diff fp32_tc vs fp32 {rel:.2e})",
           time_variants(variants, args.rounds, args.iters), launches)

    # the batched controller step, each precision on its own robots' state
    arr = bench.synthetic_raw_states(capi, 4096, seed=3)
    raw = np.frombuffer(bytes(arr), np.uint8).reshape(4096, -1)
    d_raw = torch.from_numpy(np.tile(raw, (ROWS // 4096, 1)).copy()).cuda()
    del obs, outs
    state = {k: (torch.zeros((ROWS, 98), device="cuda"), torch.zeros((ROWS, 3), device="cuda"),
                 torch.zeros((ROWS, 12), device="cuda"), torch.zeros((ROWS, 12), device="cuda", dtype=torch.float64))
             for k in PRECS}

    def step(k):
        o, v, act, q = state[k]
        return lambda: pb.step_device(d_raw.data_ptr(), v.data_ptr(), o.data_ptr(), act.data_ptr(), q.data_ptr(), ROWS,
                                      PRECS[k], stream)

    variants = {k: step(k) for k in PRECS}
    for k, fn in variants.items():
        fn()
        launches[k] = pb.last_launches()
    report(f"step: controller step, {ROWS:,} robots", time_variants(variants, args.rounds, args.iters), launches)
    del state
    pb.close()

    wpath = os.path.join(tempfile.mkdtemp(prefix="go2p_wide_"), "wide.onnx")
    ws, bs = onnx_writer.wide_policy(seed=5)
    onnx_writer.write_policy(wpath, ws, bs)
    wp = pkg.PolicyBatch(wpath, history=5)
    w_obs = torch.randn((WIDE_ROWS, 245), device="cuda", dtype=torch.float32, generator=g)
    w_out = {k: torch.empty((WIDE_ROWS, 12), device="cuda") for k in PRECS}

    def wide(k):
        return lambda: wp.infer_device(w_obs.data_ptr(), w_out[k].data_ptr(), WIDE_ROWS, PRECS[k], stream)

    variants = {k: wide(k) for k in PRECS}
    for k, fn in variants.items():
        fn()
        launches[k] = wp.last_launches()
    torch.cuda.synchronize()
    a, b = w_out["fp32_tc"].double(), w_out["fp32"].double()
    rel = ((a - b).abs() / b.abs().clamp(min=1.0)).max().item()
    report(f"wide: 245-1024-512-256-12 policy, {WIDE_ROWS:,} rows (max rel diff fp32_tc vs fp32 {rel:.2e})",
           time_variants(variants, args.rounds, args.iters), launches)
    wp.close()


if __name__ == "__main__":
    main()
