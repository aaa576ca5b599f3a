"""Cost of replaying T steps of per-field sensor streams: 1,048,576 robots, fp16, device buffers, T = 8 and 32.

Times, with CUDA events, in one process, four variants alternately over several rounds (after a warm-up of each):
  steps     T calls of go2p_step_batch_fields on the step-t slices (with q_des, which the single step requires)
  seq       one go2p_step_batch_fields_seq call (published actions only)
  seq+qdes  the same with d_qdes_seq
  seq+obs   the same with d_obs_seq (every step's observation)
and prints the card's name, power limit and maximum SM clock next to the fastest round and the median per robot-step,
with the algorithmic HBM bytes per robot-step and the fraction of 7.7 TB/s they reach at the median.  The streams
(T x 150 B per robot) and the state are far larger than L2, so every step reads from HBM.  Before timing, the seq call
is checked to leave the bytes of the T single steps.

    python scripts/fields_seq_time.py [--rounds 7] [--steps 8 32]
"""
import argparse
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import go2_onnx_controller_b200 as pkg  # noqa: E402
from go2_onnx_controller_b200 import actor, capi  # noqa: E402
from reset_step_time import ROWS, card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12                        # HGX B200 data sheet, one GPU
FIELD_BYTES = 16 + 12 + 48 + 48 + 16 + 8 + 1 + 1
STATE_BYTES = 98 * 4 + 3 * 4 + 12 * 4           # history, joystick command, previous action: read and written once


def algorithmic_bytes(variant, T):
    """HBM bytes per robot-step the variant has to move at least."""
    if variant == "steps":                      # every step: fields, state in and out, q_des out
        return FIELD_BYTES + 2 * STATE_BYTES + 12 * 8
    b = FIELD_BYTES + 12 * 4 + 2 * STATE_BYTES / T
    return b + (12 * 8 if variant == "seq+qdes" else 0) + (98 * 4 if variant == "seq+obs" else 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, nargs="+", default=[8, 32])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (the library has no CPU path)")

    pb = pkg.PolicyBatch(pkg.DEFAULT_MODEL)
    lib, h = pb._hd.lib, pb._hd.h
    stream = torch.cuda.current_stream().cuda_stream
    P, B = capi.PREC_FP16, ROWS
    print(f"card: {card()}")
    print(f"{B:,} robots, fp16, {args.rounds} alternating rounds; ms per step of all robots (a call's time / T): "
          f"fastest round / median; bytes = algorithmic HBM bytes per robot-step")
    for T in args.steps:
        g = torch.Generator(device="cuda").manual_seed(T)
        dev = dict(device="cuda", generator=g)
        quat = torch.randn((T, B, 4), **dev)
        quat /= quat.norm(dim=-1, keepdim=True)
        fields = dict(quat=quat, gyro=torch.randn((T, B, 3), **dev), q=0.3 * torch.randn((T, B, 12), **dev),
                      dq=torch.randn((T, B, 12), **dev), axes=2.0 * torch.rand((T, B, 4), **dev) - 1.0,
                      foot_force=torch.randint(0, 60, (T, B, 4), dtype=torch.int16, **dev),
                      joy_valid=torch.rand((T, B), **dev) < 0.6, button0=(torch.rand((T, B), **dev) < 0.1).to(torch.uint8))
        f_all = capi.RawFields(*[fields[n].data_ptr() for n, _ in actor.RAW_FIELDS])
        f_t = [capi.RawFields(*[fields[n][t].data_ptr() for n, _ in actor.RAW_FIELDS]) for t in range(T)]
        obs = torch.zeros((B, 98), device="cuda"); vel = torch.zeros((B, 3), device="cuda")
        act = torch.zeros((B, 12), device="cuda"); q = torch.zeros((B, 12), device="cuda", dtype=torch.float64)
        act_seq = torch.zeros((T, B, 12), device="cuda")
        q_seq = torch.zeros((T, B, 12), device="cuda", dtype=torch.float64)
        obs_seq = torch.zeros((T, B, 98), device="cuda")

        def steps():
            for t in range(T):
                capi.check(lib.go2p_step_batch_fields(h, C.byref(f_t[t]), None, vel.data_ptr(), obs.data_ptr(),
                                                      act.data_ptr(), q.data_ptr(), None, B, P, stream))

        def seq(qs=None, os_=None):
            capi.check(lib.go2p_step_batch_fields_seq(h, C.byref(f_all), T, None, vel.data_ptr(), obs.data_ptr(),
                                                      act.data_ptr(), act_seq.data_ptr(),
                                                      None if qs is None else qs.data_ptr(), None,
                                                      None if os_ is None else os_.data_ptr(), B, P, stream))

        variants = {"steps": steps, "seq": seq, "seq+qdes": lambda: seq(qs=q_seq), "seq+obs": lambda: seq(os_=obs_seq)}

        outs = {}
        for k in ("steps", "seq"):                   # from the same (zero) state: the same final state
            for t in (obs, vel, act):
                t.zero_()
            variants[k]()
            torch.cuda.synchronize()
            outs[k] = [t.cpu().numpy().view(np.uint8) for t in (obs, vel, act)]
            if k == "seq":
                assert pb.last_launches() == 1
        assert all(np.array_equal(a, b) for a, b in zip(outs["steps"], outs["seq"]))

        for fn in variants.values():                   # warm-up: module load, smem opt-in, clocks
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = {k: [] for k in variants}
        for r in range(args.rounds):
            order = list(variants) if r % 2 == 0 else list(reversed(variants))
            for k in order:
                variants[k]()
                e0.record()
                variants[k]()
                e1.record()
                e1.synchronize()
                ms[k].append(e0.elapsed_time(e1) / T)      # per step of B robots
        print(f"T = {T}")
        base = float(np.median(ms["steps"]))
        for k, v in ms.items():
            med = float(np.median(v))
            nbytes = algorithmic_bytes(k, T)
            frac = nbytes * B / (med * 1e-3) / HBM_BYTES_PER_S
            print(f"  {k:<9} {min(v):.4f} / {med:.4f} ms per step  {med / base:.3f} x steps (median)  "
                  f"{nbytes:7.1f} B/robot-step  {frac:.2f} of HBM")
        del fields, act_seq, q_seq, obs_seq
        torch.cuda.empty_cache()
    pb.close()


if __name__ == "__main__":
    main()
