"""Cost of per-robot resets in the fused controller step: 1,048,576 robots, fp16, device buffers.

Times, with CUDA events, in one process, the variants alternately over several rounds (after a warm-up of each):
  cmd        go2p_step_batch_cmd (no mask)
  ex_null    go2p_step_batch_ex with a NULL mask
  ex_zero    go2p_step_batch_ex with an all-zero mask
  ex_1pct    go2p_step_batch_ex with 1 % random resets
  ex_all     go2p_step_batch_ex with every robot reset
  torch_fill the alternative without the mask: masked_fill_ of d_obs / d_vel_cmd / d_action (the 1 % rows), then
             go2p_step_batch_cmd
and prints the card's name, power limit and maximum SM clock next to the numbers.  The working set (~0.6 GB) is far
larger than L2, so every step reads its state from HBM.

    python scripts/reset_step_time.py [--rounds 7] [--iters 20]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import go2_onnx_controller_b200 as pkg  # noqa: E402
from go2_onnx_controller_b200 import capi  # noqa: E402

ROWS = 1_048_576


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20, help="steps per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (the library has no CPU path)")

    pb = pkg.PolicyBatch(pkg.DEFAULT_MODEL)
    lib, h = pb._hd.lib, pb._hd.h
    arr = bench.synthetic_raw_states(capi, 4096, seed=3)
    raw_np = np.frombuffer(bytes(arr), np.uint8).reshape(4096, C.sizeof(capi.RawState))
    d_raw = torch.from_numpy(np.tile(raw_np, (ROWS // 4096, 1)).copy()).cuda()
    obs = torch.zeros((ROWS, 98), device="cuda"); vel = torch.zeros((ROWS, 3), device="cuda")
    act = torch.zeros((ROWS, 12), device="cuda"); q = torch.zeros((ROWS, 12), device="cuda", dtype=torch.float64)
    gen = torch.Generator(device="cuda").manual_seed(5)
    m_zero = torch.zeros(ROWS, device="cuda", dtype=torch.bool)
    m_1pct = torch.rand(ROWS, device="cuda", generator=gen) < 0.01
    m_all = torch.ones(ROWS, device="cuda", dtype=torch.bool)
    stream = torch.cuda.current_stream().cuda_stream
    P = capi.PREC_FP16

    def cmd():
        capi.check(lib.go2p_step_batch_cmd(h, d_raw.data_ptr(), vel.data_ptr(), obs.data_ptr(), act.data_ptr(), q.data_ptr(),
                                           None, ROWS, P, stream))

    def ex(mask):
        ptr = None if mask is None else mask.data_ptr()
        return lambda: capi.check(lib.go2p_step_batch_ex(h, d_raw.data_ptr(), ptr, vel.data_ptr(), obs.data_ptr(),
                                                         act.data_ptr(), q.data_ptr(), None, ROWS, P, stream))

    rows_1pct = m_1pct.unsqueeze(1)

    def torch_fill():
        obs.masked_fill_(rows_1pct, 0.0); vel.masked_fill_(rows_1pct, 0.0); act.masked_fill_(rows_1pct, 0.0)
        cmd()

    variants = {"cmd": cmd, "ex_null": ex(None), "ex_zero": ex(m_zero), "ex_1pct": ex(m_1pct), "ex_all": ex(m_all),
                "torch_fill": torch_fill}
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
    print(f"{ROWS:,} robots, fp16, {args.rounds} rounds x {args.iters} steps; ms per step (median, min-max over rounds)")
    base = float(np.median(ms["cmd"]))
    for k, v in ms.items():
        med = float(np.median(v))
        print(f"  {k:<11} {med:.4f}  ({min(v):.4f}-{max(v):.4f})  {100.0 * (med / base - 1.0):+.2f} % vs cmd")
    pb.close()


if __name__ == "__main__":
    main()
