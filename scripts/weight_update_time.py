"""Cost of replacing a live handle's policy weights (go2p_set_weights / go2p_set_weights_host) against re-creating it.

For the Go2 policy (98-128-128-128-12, bundled model) and the wide 245-1024-512-256-12 policy, in one process:
  set_weights     go2p_set_weights from CUDA tensors: CUDA events around each call on one stream (median of --calls)
  set_weights_host  go2p_set_weights_host from numpy arrays: host wall time of the synchronous call (median)
  create+destroy  go2p_create + go2p_destroy of the same model from its .onnx: host wall time (median)
and, for the Go2 policy, the 1,048,576-robot fp16 fused controller step launched right after an update (that launch goes
without programmatic serialization) against the same step in steady state, alternately (median of --rounds).
Prints the card's name, power limit and maximum SM clock next to the numbers.

    python scripts/weight_update_time.py [--calls 200] [--rounds 50]
"""
import argparse
import ctypes as C
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import go2_onnx_controller_b200 as pkg  # noqa: E402
from go2_onnx_controller_b200 import capi  # noqa: E402
from oracle import onnx_mini  # noqa: E402

from reset_step_time import card  # noqa: E402

ROWS = 1_048_576


def tensors(dims, seed):
    rng = np.random.default_rng(seed)
    ws = [rng.uniform(-0.1, 0.1, (o, i)).astype(np.float32) for i, o in zip(dims[:-1], dims[1:])]
    bs = [rng.uniform(-0.1, 0.1, o).astype(np.float32) for o in dims[1:]]
    return ws, bs


def wall_ms(fn, n):
    t = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def update_times(name, path, calls):
    pb = pkg.PolicyBatch(path)
    ws, bs = tensors(pb._hd.dims, seed=1)
    tw, tb = [torch.from_numpy(w).cuda() for w in ws], [torch.from_numpy(b).cuda() for b in bs]
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(5):
        pb.set_weights(tw, tb, stream=stream)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
    for e0, e1 in ev:
        e0.record()
        pb.set_weights(tw, tb, stream=stream)
        e1.record()
    torch.cuda.synchronize()
    dev = float(np.median([e0.elapsed_time(e1) for e0, e1 in ev]))
    host = wall_ms(lambda: pb.set_weights(ws, bs), max(10, calls // 10))
    pb.close()
    create = wall_ms(lambda: pkg.PolicyBatch(path).close(), 5)
    n = sum(w.size + b.size for w, b in zip(ws, bs))
    print(f"  {name:<22} {n:>9,} params  set_weights {dev * 1e3:8.1f} us   set_weights_host {host:7.3f} ms   "
          f"create+destroy {create:7.2f} ms")


def step_after_update(rounds):
    pb = pkg.PolicyBatch(pkg.DEFAULT_MODEL)
    lib, h = pb._hd.lib, pb._hd.h
    ws, bs = tensors(pb._hd.dims, seed=2)
    tw, tb = [torch.from_numpy(w).cuda() for w in ws], [torch.from_numpy(b).cuda() for b in bs]
    arr = bench.synthetic_raw_states(capi, 4096, seed=3)
    raw_np = np.frombuffer(bytes(arr), np.uint8).reshape(4096, C.sizeof(capi.RawState))
    d_raw = torch.from_numpy(np.tile(raw_np, (ROWS // 4096, 1)).copy()).cuda()
    obs = torch.zeros((ROWS, 98), device="cuda"); vel = torch.zeros((ROWS, 3), device="cuda")
    act = torch.zeros((ROWS, 12), device="cuda"); q = torch.zeros((ROWS, 12), device="cuda", dtype=torch.float64)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        capi.check(lib.go2p_step_batch_cmd(h, d_raw.data_ptr(), vel.data_ptr(), obs.data_ptr(), act.data_ptr(), q.data_ptr(),
                                           None, ROWS, capi.PREC_FP16, stream))

    for _ in range(10):
        step()
    pb.set_weights(tw, tb, stream=stream)
    step()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    after, steady = [], []
    for r in range(rounds):
        for kind in (("after", "steady") if r % 2 == 0 else ("steady", "after")):
            step()
            if kind == "after":
                pb.set_weights(tw, tb, stream=stream)
            e[0].record()
            step()
            e[1].record()
            e[1].synchronize()
            (after if kind == "after" else steady).append(e[0].elapsed_time(e[1]))
    pb.close()
    print(f"  fused fp16 step, {ROWS:,} robots: right after an update {np.median(after):.4f} ms "
          f"({min(after):.4f}-{max(after):.4f}), steady state {np.median(steady):.4f} ms ({min(steady):.4f}-{max(steady):.4f})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (the library has no CPU path)")
    print(f"card: {card()}")
    with tempfile.TemporaryDirectory() as tmp:
        wide = os.path.join(tmp, "wide.onnx")
        ws, bs = onnx_mini.make_wide_policy(seed=5)
        with open(wide, "wb") as fh:
            fh.write(onnx_mini.write_mlp_onnx(ws, bs, 1.0, batch="batch"))
        update_times("Go2 98-128x3-12", pkg.DEFAULT_MODEL, args.calls)
        update_times("wide 245-1024-512-256-12", wide, args.calls)
    step_after_update(args.rounds)


if __name__ == "__main__":
    main()
