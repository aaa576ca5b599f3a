#!/usr/bin/env python
"""Headline benchmark of the Go2 policy hot path (BASELINE.json: policy inferences/s, batch-1 latency).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the batched hot path (A7 with the fused A9 clamp+mask epilogue) over BASELINE.json configs[3]:
ONE batch of 1,048,576 rollouts of the bundled Go2 policy, SHARDED over the N GPUs in contiguous row blocks
(go2p_shard_rows; strong scaling: 131,072 rows per GPU at N=8).  Rows are independent, every rank owns its block and
its own copy of the weights; there is no collective on the data path.
`value`    device-timed throughput of the whole job, observations already resident in HBM.  Every rank cycles through
           enough distinct input/output blocks that consecutive steps never find their rows in the 126 MB L2.
`weak`     the same kernel with 1,048,576 rows on EVERY GPU (what round 1 reported as the headline).
`e2e`      the same metric through go2p_infer_batch_host with pinned HOST buffers (H2D + kernel + D2H inside).
`e2e_step` closed-loop control steps from host buffers through go2p_step_batch_host: 156 B of raw state in and 48 B of
           action out per robot, history resident on the device (SURVEY.md 8d, fused pre/post variant).
`roofline` algorithmic 440 B/inference (SURVEY.md 8d) over the kernel's measured launch duration vs measured HBM.
`wide_mlp` BASELINE.json configs[4]: synthetic 245-1024-512-256-12 policy, 262,144 rows sharded the same way.
`cpu_baseline` the oracle's C port of the reference path on the box's host cores (ORT itself is not available), and a
           torch-CPU (MKL/oneDNN) batched arm beside it.
Prints ONE JSON line on rank 0.

--dump-outputs DIR writes the published actions of the last timed step (this rank's rows, float32) to
DIR/action.npy, or DIR/action_rank<r>.npy with several ranks; beyond 64 MB in all, every k-th row.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.  The two --impl arms draw
their inputs differently (CUDA generator seeded with the rank / oracle.make_obs_d1 on the host), so compare dumps of
the same arm only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GLOBAL_ROWS = 1_048_576                       # BASELINE.json configs[3]
WIDE_ROWS = 262_144                           # BASELINE.json configs[4]
ALGO_BYTES_PER_INF = 98 * 4 + 12 * 4          # SURVEY.md 8(d): obs in + action out, weights amortised
ALGO_FLOP_PER_INF = 93696
WIDE_FLOP_PER_INF = 2 * (245 * 1024 + 1024 * 512 + 512 * 256 + 256 * 12)
RAW_BYTES = 156                               # sizeof(go2p_raw_state)
# dram__bytes_read.sum + dram__bytes_write.sum of one tc_mlp_kernel launch over 1,048,576 rows, from the ncu --set full
# capture of the shipped kernel (profiles/r02_tc_mlp_kernel_raw.csv)
NCU_TRAFFIC_BYTES_PER_ROW = (415.403520e6 + 41.018112e6) / 1048576
L2_BYTES = 126e6
DUMP_BYTES = 64_000_000                       # --dump-outputs: all ranks' files together
METRIC = "policy_inferences_per_sec"
UNIT = "inferences/s"


def workload_config(precision):
    """The configuration both arms (ours and --impl reference) run: identical dictionaries."""
    return {"workload": "configs[3]: bundled Go2 policy 98-128-128-128-12, ONE batch of 1,048,576 rollouts per step "
                        "(N(0,1) observations), A7 + A9 clamp/mask, rows sharded over the GPUs in contiguous blocks",
            "global_rows": GLOBAL_ROWS, "precision": precision if precision != "cpu" else "fp32"}


def shard(total, n, i):
    q, r = divmod(total, n)
    b = i * q + min(i, r)
    return b, b + q + (1 if i < r else 0)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 0))), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_raw_states(capi, n, seed):
    """Closed-loop raw-state distribution of SURVEY.md 8(d) (small-angle attitude, joints around the default pose,
    uniform joystick, rare dead-man press) as an array of go2p_raw_state -- bench input only, generated here so the
    timed paths never touch oracle/."""
    import numpy as np
    rng = np.random.default_rng(seed)
    q0 = np.array([0.1, -0.1, 0.1, -0.1, 0.8, 0.8, 1.0, 1.0, -1.5, -1.5, -1.5, -1.5], np.float32)   # controller.hpp:119-120
    arr = (capi.RawState * n)()
    for i in range(n):
        axis = rng.standard_normal(3)
        axis /= np.linalg.norm(axis) + 1e-12
        ang = rng.normal(0.0, 0.2)
        r = arr[i]
        r.quat[:] = [float(np.cos(ang / 2))] + [float(v) for v in np.sin(ang / 2) * axis]
        r.gyro[:] = [float(v) for v in rng.normal(0, 0.5, 3)]
        r.q[:] = [float(v) for v in q0 + rng.normal(0, 0.3, 12)]
        r.dq[:] = [float(v) for v in rng.normal(0, 2.0, 12)]
        r.foot_force[:] = [int(v) for v in rng.integers(0, 61, 4)]
        r.axes[:] = [float(v) for v in rng.uniform(-1, 1, 4)]
        r.joy_valid = 1
        r.button0 = int(rng.random() < 0.01)
    return arr


def dump_outputs(dirname, name, array, rank, world):
    """Saves `array` (rows x cols) for --dump-outputs.  All ranks together write at most DUMP_BYTES: a larger output is
    sampled at a fixed row stride, so runs with the same arguments write the same rows."""
    import numpy as np
    stride = -(-array.nbytes * world // DUMP_BYTES)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, f"{name}.npy" if world == 1 else f"{name}_rank{rank}.npy"), array[::max(1, stride)])


def cpu_reference_rate(rows_per_step, steps, warmup, threads=None, blocked=False):
    """The reference path on host cores: B independent batch-1 forwards (the static-batch model's semantics,
    onnx_actor.cpp:38-48) + A9 clamp/mask, rows split over all cores -- C port in oracle/ (test infrastructure).
    Returns (rows/s, seconds, threads, published actions of the last step)."""
    from oracle import coracle, oracle
    from go2_onnx_controller_b200 import DEFAULT_MODEL
    cm = coracle.CModel(DEFAULT_MODEL)             # liboracle.so is built by build(): the tree may be read-only here
    # all host cores this process may use (torchrun exports OMP_NUM_THREADS=1, so do not ask OpenMP)
    threads = threads or len(os.sched_getaffinity(0))
    X = oracle.make_obs_d1(rows_per_step, 98, seed=0)
    for _ in range(warmup):
        cm.forward_f32(X[: max(1, rows_per_step // 8)], threads, blocked)
    t0 = time.perf_counter()
    for _ in range(steps):
        y = cm.forward_f32(X, threads, blocked)
        published = oracle.clamp_mask(y, 0)
    dt = time.perf_counter() - t0
    return rows_per_step * steps / dt, dt, threads, published


def torch_cpu_rate(rows, seconds=4.0):
    """The "generous" CPU arm of SURVEY.md 8d: the same Gemm/Elu chain as batched torch-CPU (MKL / oneDNN) GEMMs over
    all host cores -- a batched implementation the reference does not have; weights read by the oracle's ONNX reader."""
    import numpy as np
    import torch
    from oracle import oracle
    from go2_onnx_controller_b200 import DEFAULT_MODEL
    pol = oracle.load_policy(DEFAULT_MODEL)
    threads = len(os.sched_getaffinity(0))
    torch.set_num_threads(threads)
    ws = [torch.from_numpy(np.ascontiguousarray(l.weight, np.float32)) for l in pol.layers]
    bs = [torch.from_numpy(np.ascontiguousarray(l.bias, np.float32)) for l in pol.layers]
    x = torch.randn((rows, 98), dtype=torch.float32)

    def fwd():
        h = x
        for i, (w, b) in enumerate(zip(ws, bs)):
            h = torch.nn.functional.linear(h, w, b)
            if i + 1 < len(ws):
                h = torch.nn.functional.elu(h)
        return torch.clamp(h, -1000.0, 1000.0)
    with torch.no_grad():
        fwd()
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            fwd()
            n += 1
        dt = time.perf_counter() - t0
    return rows * n / dt, threads, n, dt


def run_reference(args, rank):
    if rank != 0:
        return
    rows = GLOBAL_ROWS
    rate, dt, threads, published = cpu_reference_rate(rows, args.steps, min(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "action", published, 0, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.precision),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{rows} rows x {args.steps} steps (the whole 1,048,576-row step), C restatement of the Gemm/Elu "
                                   "chain + clamp/mask, batch-1 semantics per row, OpenMP over all host cores; ONNX Runtime itself "
                                   "is not installable here (no wheel, no network)"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=GLOBAL_ROWS, help="rows of the global batch per step")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--b1-steps", type=int, default=100_000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-b1", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline + e2e only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's actions to DIR/action.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import ctypes as C
    import numpy as np
    import torch
    import go2_onnx_controller_b200 as pkg
    from go2_onnx_controller_b200 import capi, onnx_writer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    prec = capi.PREC_NAMES[args.precision]
    total = args.rows
    r_begin, r_end = shard(total, world, rank)          # the same split go2p_shard_rows makes
    rows = r_end - r_begin
    pb = pkg.PolicyBatch(pkg.DEFAULT_MODEL, device=local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    flags = capi.F_CLAMP_MASK
    # enough distinct blocks that two consecutive steps can never share L2 contents: 2 x L2 of inputs in rotation
    n_buf = max(1, int(np.ceil(2 * L2_BYTES / (rows * 98 * 4))))
    n_buf_timed = n_buf                                  # what the headline loop rotates over (reported in `sharding.l2`)
    g = torch.Generator(device="cuda").manual_seed(rank)
    d_obs = [torch.randn((rows, 98), device="cuda", dtype=torch.float32, generator=g) for _ in range(n_buf)]   # D1, seed = rank
    d_act = [torch.empty((rows, 12), device="cuda", dtype=torch.float32) for _ in range(n_buf)]
    d_b0 = torch.zeros((rows,), device="cuda", dtype=torch.int32)

    def step(i):
        k = i % n_buf
        pb.infer_device(d_obs[k].data_ptr(), d_act[k].data_ptr(), rows, prec, stream, d_b0.data_ptr(), None, flags)

    def timed_loop(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for i in range(args.warmup):
        step(i)
    launches_per_step = pb.last_launches()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    time.sleep(0.3 if rank == 0 else 0)
    barrier()
    t_wall0 = time.time()
    ms_local = timed_loop(step, args.steps)
    barrier()
    # later untimed launches reuse these buffers: keep the last timed step's output as it was
    last_action = d_act[(args.steps - 1) % n_buf].clone() if args.dump_outputs else None
    ms = max_over_ranks(ms_local)
    # keep the device busy a little longer for short runs so that the 100 ms clock sampler sees it under load
    if rank == 0 and time.time() - t_wall0 < 0.6:
        tb, i = time.time(), 0
        while time.time() - tb < 0.6:
            step(i); i += 1
        torch.cuda.synchronize()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    value = total * args.steps / (ms * 1e-3)
    kernel_ms = ms / args.steps

    # parity spot check of what was just timed (oracle = checker only)
    if rank == 0:
        from oracle import oracle
        pol = oracle.load_policy(pkg.DEFAULT_MODEL)
        idx = torch.randint(0, rows, (256,), device="cuda")
        ref = oracle.clamp_mask(oracle.forward(pol, d_obs[0][idx].cpu().numpy()).astype(np.float32), 0)
        step(0); torch.cuda.synchronize()
        parity_err = float(np.abs(d_act[0][idx].cpu().numpy() - ref).max())

    # ---- weak scaling: 1,048,576 rows on every GPU (fits the buffers only at world > 1 if re-allocated; short run)
    weak = None
    if not args.no_extras:
        if world == 1:
            weak = {"rows_per_gpu": rows, "value": value, "ms_per_step": kernel_ms}
        else:
            del d_obs, d_act
            w_obs = torch.randn((GLOBAL_ROWS, 98), device="cuda", dtype=torch.float32, generator=g)
            w_act = torch.empty((GLOBAL_ROWS, 12), device="cuda", dtype=torch.float32)
            w_b0 = torch.zeros((GLOBAL_ROWS,), device="cuda", dtype=torch.int32)
            wfn = lambda i: pb.infer_device(w_obs.data_ptr(), w_act.data_ptr(), GLOBAL_ROWS, prec, stream, w_b0.data_ptr(), None, flags)
            for i in range(3):
                wfn(i)
            barrier()
            wms = max_over_ranks(timed_loop(wfn, 20)) / 20
            weak = {"rows_per_gpu": GLOBAL_ROWS, "value": world * GLOBAL_ROWS / (wms * 1e-3), "ms_per_step": wms}
            del w_obs, w_act, w_b0
            d_obs = [torch.randn((rows, 98), device="cuda", dtype=torch.float32, generator=g)]
            d_act = [torch.empty((rows, 12), device="cuda", dtype=torch.float32)]
            n_buf = 1

    # ---- BASELINE.json configs[2]: batch 4096 on one GPU -- single-launch latency and pipelined throughput
    small = None
    if rank == 0 and not args.no_extras:
        sb = 4096
        lat = []
        for _ in range(200):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            pb.infer_device(d_obs[0].data_ptr(), d_act[0].data_ptr(), sb, prec, stream, d_b0.data_ptr(), None, flags)
            a1.record()
            a1.synchronize()
            lat.append(a0.elapsed_time(a1) * 1e3)
        ms_pipe = pb.time_device(d_obs[0].data_ptr(), d_act[0].data_ptr(), sb, prec, 200, stream, d_b0.data_ptr(), None, flags)
        # 4096 rows are 32 tiles = 32 CTAs on 148 SMs: independent batches on four streams run side by side
        n_str, per = 4, 100
        streams = [torch.cuda.Stream() for _ in range(n_str)]
        so = [torch.randn((sb, 98), device="cuda") for _ in range(n_str)]
        sa = [torch.empty((sb, 12), device="cuda") for _ in range(n_str)]
        torch.cuda.synchronize()
        def multi(n):
            for it in range(n):
                for k, st_ in enumerate(streams):
                    pb.infer_device(so[k].data_ptr(), sa[k].data_ptr(), sb, prec, st_.cuda_stream, d_b0.data_ptr(), None, flags)
        multi(5); torch.cuda.synchronize()
        tm0 = time.perf_counter(); multi(per); torch.cuda.synchronize(); tm = time.perf_counter() - tm0
        small = {"batch": sb, "single_launch_us_p50": float(np.percentile(lat, 50)), "single_launch_us_p99": float(np.percentile(lat, 99)),
                 "pipelined_inferences_per_sec": sb * 200 / (ms_pipe * 1e-3),
                 "pipelined_4_streams_inferences_per_sec": sb * n_str * per / tm,
                 "note": "L2-resident (1.8 MB); one launch = 32 CTAs, latency bound by the 4-layer chain of one tile; four "
                         "streams fill 128 of the 148 SMs with independent batches"}

    # ---- the fp32 contract path (1e-5 vs the reference) on the same rows: its throughput beside the tensor-core one
    fp32_path = None
    if rank == 0 and not args.no_extras and args.precision != "fp32":
        n32 = 3
        ms32 = pb.time_device(d_obs[0].data_ptr(), d_act[0].data_ptr(), rows, capi.PREC_FP32, n32, stream, d_b0.data_ptr(), None, flags)
        ms32 = pb.time_device(d_obs[0].data_ptr(), d_act[0].data_ptr(), rows, capi.PREC_FP32, n32, stream, d_b0.data_ptr(), None, flags) / n32
        fp32_path = {"rows": rows, "ms_per_step": ms32, "inferences_per_sec": rows / (ms32 * 1e-3), "launches_per_step": pb.last_launches() // n32,
                     "note": "CUDA-core FFMA path, <= 1e-5 vs the fp64 oracle (the reference's precision)"}

    # ---- e2e: HOST buffers through the C ABI, copies inside the timed region; this rank's shard of the global batch
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    hx = pb.pinned((rows, 98))
    hy = pb.pinned((rows, 12))
    hx[:] = d_obs[0].cpu().numpy()
    for _ in range(2):
        pb.infer_host(hx, hy, prec)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        pb.infer_host(hx, hy, prec)          # synchronous: returns when the actions are in host memory
    dt_local = time.perf_counter() - t0
    e2e_launches = pb.last_launches()
    barrier()
    dt = max_over_ranks(dt_local)
    e2e_value = total * e2e_steps / dt

    # ---- pinned-copy ceiling of this box at this N (H2D and D2H at the same time, all ranks at once): e2e's own roofline
    pcie = None
    if not args.no_extras:
        nb = 256 << 20
        h_a, h_b = torch.empty(nb, dtype=torch.uint8).pin_memory(), torch.empty(nb, dtype=torch.uint8).pin_memory()
        d_a, d_b = torch.empty(nb, dtype=torch.uint8, device="cuda"), torch.empty(nb, dtype=torch.uint8, device="cuda")
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        def both():
            with torch.cuda.stream(s1):
                d_a.copy_(h_a, non_blocking=True)
            with torch.cuda.stream(s2):
                h_b.copy_(d_b, non_blocking=True)
        both(); torch.cuda.synchronize()
        barrier()
        tc0 = time.perf_counter()
        for _ in range(4):
            both()
        torch.cuda.synchronize()
        dtc = max_over_ranks(time.perf_counter() - tc0)
        pcie = {"h2d_gbs_per_gpu": 4 * nb / dtc / 1e9, "d2h_gbs_per_gpu": 4 * nb / dtc / 1e9, "n_gpus_at_once": world,
                "note": "256 MiB pinned cudaMemcpyAsync each way concurrently on every rank; e2e cannot exceed "
                        "h2d_gbs / bytes-in-per-row"}
        del h_a, h_b, d_a, d_b

    # ---- closed-loop fleet step from host buffers: 156 B in, 48 B out per robot, history on the device
    e2e_step = None
    if not args.no_extras:
        arr = synthetic_raw_states(capi, 4096, seed=3 + rank)
        raw_np = np.frombuffer(bytes(arr), np.uint8).reshape(4096, C.sizeof(capi.RawState))
        h_raw = pb.pinned((rows, RAW_BYTES), np.uint8)
        h_raw[:] = np.tile(raw_np, (rows // 4096 + 1, 1))[:rows]
        for _ in range(2):
            pb.step_host(h_raw, hy, None, prec)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            pb.step_host(h_raw, hy, None, prec)
        dts = max_over_ranks(time.perf_counter() - t0)
        barrier()
        e2e_step = {"value": total * e2e_steps / dts, "unit": "robot-steps/s", "h2d_bytes_per_step": rows * RAW_BYTES,
                    "d2h_bytes_per_step": rows * 12 * 4, "steps": e2e_steps, "ms_per_step": dts / e2e_steps * 1e3,
                    "algorithmic_bytes_per_robot_step": RAW_BYTES + 48,
                    "api": "go2p_step_batch_host (pinned raw states in, published actions out, per-robot history resident in HBM)"}

    hbm_peak, tf_peak, peak_src = measured_peaks()
    achieved_gbs = ALGO_BYTES_PER_INF * rows / (kernel_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": args.precision, "data": "synthetic",
        "config": workload_config(args.precision),
        "sharding": {"rows_per_gpu": rows, "split": f"dp{world}, contiguous row blocks (go2p_shard_rows), no data-path collective",
                     "l2": f"{n_buf_timed} distinct input/output blocks of {rows * 98 * 4 / 1e6:.0f} MB per GPU in rotation "
                           f"(> 2 x 126 MB L2 between reuses), no flush needed"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": rows * 98 * 4, "d2h_bytes_per_step": rows * 12 * 4,
                "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3, "api": "go2p_infer_batch_host (pinned host buffers)"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                     "traffic": (NCU_TRAFFIC_BYTES_PER_ROW * rows if args.precision != "fp32" else None), "peak_source": peak_src,
                     "kernel": "tc_mlp_kernel" if args.precision != "fp32" else "sgemm_bias_act_kernel",
                     "algorithmic_bytes_per_inference": ALGO_BYTES_PER_INF, "rows_per_launch": rows,
                     "tensor_frac": ALGO_FLOP_PER_INF * rows / (kernel_ms * 1e-3) / 1e12 / tf_peak},
        "clocks": clocks,
    }
    if weak:
        line["weak"] = weak
    if e2e_step:
        line["e2e_step"] = e2e_step
    if pcie:
        line["pinned_copy_peak"] = pcie
    if rank == 0:
        line["parity_max_abs_err_vs_oracle"] = parity_err
        if small:
            line["batch4096"] = small
        if fp32_path:
            line["fp32_path"] = fp32_path

    # ---- BASELINE.json configs[4]: wide policy, 262,144 rows sharded over the GPUs
    if not args.no_extras:
        wb, we = shard(WIDE_ROWS, world, rank)
        wrows = we - wb
        wpath = os.path.join(tempfile.mkdtemp(prefix="go2p_wide_"), "wide.onnx")
        ws_, bs_ = onnx_writer.wide_policy(seed=5)
        onnx_writer.write_policy(wpath, ws_, bs_)
        wp = pkg.PolicyBatch(wpath, device=local_rank)
        gw = torch.Generator(device="cuda").manual_seed(100 + rank)
        w_obs = torch.randn((wrows, 245), device="cuda", dtype=torch.float32, generator=gw)
        w_act = torch.empty((wrows, 12), device="cuda", dtype=torch.float32)
        wprec = capi.PREC_FP16 if args.precision == "fp32" else prec
        wfn = lambda i: wp.infer_device(w_obs.data_ptr(), w_act.data_ptr(), wrows, wprec, stream)
        for i in range(3):
            wfn(i)
        w_launches = wp.last_launches()
        barrier()
        n_w = 10
        wms = max_over_ranks(timed_loop(wfn, n_w)) / n_w
        if rank == 0:
            from oracle import oracle
            wpol = oracle.load_policy(wpath)
            wi = torch.randint(0, wrows, (128,), device="cuda")
            werr = float(np.abs(w_act[wi].cpu().numpy() - oracle.forward(wpol, w_obs[wi].cpu().numpy())).max())
            wrate = WIDE_ROWS / (wms * 1e-3)
            line["wide_mlp"] = {"workload": "configs[4]: synthetic 245-1024-512-256-12 ELU policy, 262,144 rows sharded over the GPUs",
                                "rows_per_gpu": wrows, "ms_per_step": wms, "inferences_per_sec": wrate,
                                "tflops": wrate * WIDE_FLOP_PER_INF / 1e12,
                                "frac_of_bf16_sustained_per_gpu": wrate * WIDE_FLOP_PER_INF / 1e12 / world / tf_peak,
                                "launches_per_step": w_launches, "parity_max_abs_err_vs_oracle": werr,
                                "precision": "fp16" if wprec == capi.PREC_FP16 else "bf16"}
        wp.close()
        del w_obs, w_act

    if rank == 0 and world == 1 and not args.no_extras:
        # SURVEY 8f-1: the whole publish() for `rows` robots (raw state -> history -> policy -> clamp/mask -> q_des)
        d_raw = torch.from_numpy(np.asarray(h_raw)).to("cuda")
        s_obs = torch.zeros((rows, 98), device="cuda"); s_vel = torch.zeros((rows, 3), device="cuda")
        s_act = torch.zeros((rows, 12), device="cuda"); s_q = torch.zeros((rows, 12), device="cuda", dtype=torch.float64)
        def ctl_step(i):
            pb.step_device(d_raw.data_ptr(), s_vel.data_ptr(), s_obs.data_ptr(), s_act.data_ptr(), s_q.data_ptr(), rows, prec, stream)
        for i in range(3):
            ctl_step(i)
        torch.cuda.synchronize()
        n_ctl = max(3, min(args.steps, 10))
        ctl_ms = timed_loop(ctl_step, n_ctl) / n_ctl
        step_bytes = 156 + 392 + 48 + 12 + 392 + 48 + 96 + 12     # raw, history in, prev action, cmd in | history out, action, q_des, cmd out
        line["batched_step"] = {"robots": rows, "ms_per_step": ctl_ms, "robot_steps_per_sec": rows / (ctl_ms * 1e-3),
                                "launches_per_step": pb.last_launches(), "algorithmic_bytes_per_robot_step": step_bytes,
                                "hbm_frac": step_bytes * rows / (ctl_ms * 1e-3) / 1e9 / hbm_peak,
                                "note": "go2p_step_batch on device buffers: A1-A6 + A7 + A9 + A11 in one launch (assembly fused "
                                        "into the policy kernel's conversion job), per-robot state in HBM"}
        del d_raw, s_obs, s_vel, s_act, s_q
    if rank == 0 and world == 1 and not args.no_b1 and not args.no_extras:
        # BASELINE.json configs[1]: batch-1 closed loop, fused pre/post, resident kernel
        raws = list(synthetic_raw_states(capi, 512, seed=2))
        ctl = pkg.Go2Controller(pkg.DEFAULT_MODEL, device=local_rank)
        ctl.closed_loop(raws, 10_000)
        host_ns, dev_ns, _ = ctl.closed_loop(raws, args.b1_steps)
        ctl.close()
        line["b1_latency_us"] = {"steps": int(args.b1_steps), "p50": float(np.percentile(host_ns, 50)) / 1e3,
                                 "p99": float(np.percentile(host_ns, 99)) / 1e3, "max": float(host_ns.max()) / 1e3,
                                 "device_p50": float(np.percentile(dev_ns, 50)) / 1e3, "device_p99": float(np.percentile(dev_ns, 99)) / 1e3,
                                 "mode": "resident kernel, host-mapped mailbox, fused A1-A6+A7+A9+A11"}
    if rank == 0 and world == 1 and not args.no_cpu:
        r0, _, thr, _ = cpu_reference_rate(32768, 1, 1)
        passes = int(max(1, min(64, round(r0 * 12 / total))))          # ~12 s of CPU work over the same rows
        rate, dtc, thr, _ = cpu_reference_rate(total, passes, 0)
        # the "generous" CPU arms of SURVEY 8d: row-blocked C forward and torch-CPU (MKL/oneDNN) batched GEMMs, all cores
        rate_b, dtb, _, _ = cpu_reference_rate(total, max(1, passes // 4), 0, blocked=True)
        rate_t, thr_t, n_t, dtt = torch_cpu_rate(65536)
        # SURVEY 8d config 1: the control-loop step on one host core (C restatement of publish(), fp32 forward)
        from oracle import coracle
        cm1 = coracle.CModel(pkg.DEFAULT_MODEL)
        raws1 = [coracle.RawState.from_buffer_copy(bytes(r)) for r in synthetic_raw_states(capi, 512, seed=2)]
        coracle.closed_loop_latency_ns(cm1, raws1, 10_000)
        ns1 = coracle.closed_loop_latency_ns(cm1, raws1, 100_000)
        line["b1_cpu_port_us"] = {"steps": 100_000, "p50": float(np.percentile(ns1, 50)) / 1e3, "p99": float(np.percentile(ns1, 99)) / 1e3,
                                  "cores": 1, "kind": "port",
                                  "note": "C restatement of publish() (A1-A11, fp32 forward) on one host thread; ONNX Runtime itself is not installable here"}
        line["cpu_baseline_blocked"] = {"value": rate_b, "unit": UNIT, "cores": thr, "kind": "port",
                                        "sample": f"{max(1, passes // 4)} passes over {total} rows in {dtb:.1f} s; row-blocked C forward "
                                                  "(oracle_mlp.c: orc_forward_blocked_f32), a batched CPU implementation the reference does not have"}
        line["cpu_baseline_torch"] = {"value": rate_t, "unit": UNIT, "cores": thr_t, "kind": "port",
                                      "sample": f"{n_t} passes over 65,536 rows in {dtt:.1f} s; torch-CPU F.linear/F.elu (MKL/oneDNN GEMMs) "
                                                "over all host cores: the generous batched arm of SURVEY 8d, not ONNX Runtime"}
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": thr, "kind": "port",
                                "sample": f"{passes} passes over {total} rows of the same N(0,1) workload in {dtc:.1f} s; C restatement "
                                          "(oracle/oracle_mlp.c), batch-1 semantics per row, OpenMP over all host cores; "
                                          "ORT CPU EP itself is not installable here"}
    if last_action is not None:
        dump_outputs(args.dump_outputs, "action", last_action.cpu().numpy(), rank, world)
    pb.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
