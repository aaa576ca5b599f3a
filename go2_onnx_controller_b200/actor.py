"""Host-side mirror of the reference's operator interface for the hot path.

  ONNXActor      same surface as the reference class (reference: onnx_inference/include/onnx_actor.hpp:14-53,
                 usage as in onnx_inference/src/python/main.py:5-28): bind an observation and an action buffer,
                 act() fills the action in place.
  Go2Controller  the arithmetic of ONNXController::publish() (reference: onnx_controller/src/controller.cpp:173-251)
                 as one fused device step.
  PolicyBatch    many robots / rollouts through the same policy (device or host buffers).

Everything computes on the GPU through include/go2policy.h; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import capi

DEFAULT_MODEL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "model.onnx")


def default_config(**overrides) -> capi.Config:
    cfg = capi.Config()
    capi.load().go2p_config_default(C.byref(cfg))
    for k, v in overrides.items():
        if k == "q0":
            cfg.q0[:] = [float(x) for x in v]
        else:
            setattr(cfg, k, v)
    return cfg


class _Handle:
    def __init__(self, model_path: str, cfg: capi.Config | None = None):
        self.lib = capi.load()
        self.h = C.c_void_p()
        cfg = cfg if cfg is not None else default_config()
        capi.check(self.lib.go2p_create(os.fspath(model_path).encode(), C.byref(cfg), C.byref(self.h)))
        self.cfg = cfg
        info = capi.ModelInfo()
        capi.check(self.lib.go2p_model_info(self.h, C.byref(info)))
        self.info = info
        self.in_dim, self.out_dim = info.in_dim, info.out_dim
        self.input_name = info.input_name.decode()
        self.output_name = info.output_name.decode()
        self.dims = [info.dims[i] for i in range(info.n_layers + 1)]

    def set_weights(self, weights, biases, obs_mean, obs_std, stream: int, host_only: bool) -> None:
        kind = weight_arrays(self.dims, weights, biases, obs_mean, obs_std, device=self.cfg.device)
        if host_only and kind != "host":
            raise TypeError("this form takes numpy arrays (host memory)")
        w, b = _ptr_array(weights), (_ptr_array(biases) if biases is not None else None)
        if kind == "host":
            capi.check(self.lib.go2p_set_weights_host(self.h, w, b, len(weights), _ptr(obs_mean), _ptr(obs_std)))
        else:
            capi.check(self.lib.go2p_set_weights(self.h, w, b, len(weights), _ptr(obs_mean), _ptr(obs_std), stream or None))

    def close(self):
        if self.h:
            self.lib.go2p_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def host_reset_mask(reset, B: int) -> np.ndarray:
    """Validates a per-robot reset mask for the host-buffer steps: a numpy bool / uint8 array of shape (B,), C-contiguous
    (one byte per robot, as go2p_step_batch_host_ex reads it).  Returns it unchanged; raises TypeError / ValueError."""
    if not isinstance(reset, np.ndarray) or reset.dtype not in (np.bool_, np.uint8):
        raise TypeError(f"reset must be a numpy bool or uint8 array, got {type(reset).__name__}"
                        + (f" of {reset.dtype}" if isinstance(reset, np.ndarray) else ""))
    if reset.shape != (B,):
        raise ValueError(f"reset must have shape ({B},), got {reset.shape}")
    if not reset.flags.c_contiguous:
        raise ValueError("reset must be C-contiguous")
    return reset


def _is_device_tensor(a) -> bool:
    """A torch-like tensor (duck-typed: this package does not import torch)."""
    return all(hasattr(a, x) for x in ("data_ptr", "is_contiguous", "device"))


def weight_arrays(dims, weights, biases=None, obs_mean=None, obs_std=None, device: int | None = None) -> str:
    """Validates a set_weights() argument list against a policy's layer widths ``dims`` ([in, h1, ..., out]) before any
    native call.  weights[l]: float32 [dims[l+1], dims[l]] (torch nn.Linear.weight layout), biases: None or a list with
    float32 [dims[l+1]] or None per layer, obs_mean / obs_std: float32 [dims[0]], both or neither.  Every array is a
    C-contiguous numpy array (host form) or every one a contiguous CUDA tensor on device ``device`` (device form);
    the two are not mixed.  Returns "host" or "device"; raises TypeError / ValueError."""
    n = len(dims) - 1
    if not isinstance(weights, (list, tuple)):
        raise TypeError(f"weights must be a list of {n} arrays, got {type(weights).__name__}")
    if len(weights) != n:
        raise ValueError(f"weights has {len(weights)} layers, the policy has {n}")
    if biases is not None:
        if not isinstance(biases, (list, tuple)):
            raise TypeError(f"biases must be None or a list of {n} arrays, got {type(biases).__name__}")
        if len(biases) != n:
            raise ValueError(f"biases has {len(biases)} layers, the policy has {n}")
    if (obs_mean is None) != (obs_std is None):
        raise ValueError("obs_mean and obs_std go together")
    named = [(f"weights[{l}]", w, (dims[l + 1], dims[l])) for l, w in enumerate(weights)]
    named += [(f"biases[{l}]", b, (dims[l + 1],)) for l, b in enumerate(biases or []) if b is not None]
    if obs_mean is not None:
        named += [("obs_mean", obs_mean, (dims[0],)), ("obs_std", obs_std, (dims[0],))]
    kinds = set()
    for name, a, shape in named:
        if isinstance(a, np.ndarray):
            kinds.add("host")
            if a.dtype != np.float32:
                raise TypeError(f"{name} must be float32, got {a.dtype}")
            contiguous = a.flags.c_contiguous
        elif _is_device_tensor(a):
            kinds.add("device")
            if str(a.dtype) != "torch.float32":
                raise TypeError(f"{name} must be float32, got {a.dtype}")
            if getattr(a.device, "type", None) != "cuda":
                raise TypeError(f"{name} is a tensor on {a.device}: pass a CUDA tensor or a numpy array")
            if device is not None and a.device.index != device:
                raise ValueError(f"{name} is on cuda:{a.device.index}, the handle on cuda:{device}")
            contiguous = a.is_contiguous()
        else:
            raise TypeError(f"{name} must be a numpy array or a CUDA tensor, got {type(a).__name__}")
        if tuple(a.shape) != shape:
            raise ValueError(f"{name} must have shape {shape}, got {tuple(a.shape)}")
        if not contiguous:
            raise ValueError(f"{name} must be C-contiguous")
    if len(kinds) > 1:
        raise TypeError("host (numpy) and device (CUDA tensor) arrays cannot be mixed in one update")
    return kinds.pop()


RAW_FIELDS = (("quat", 4), ("gyro", 3), ("q", 12), ("dq", 12), ("axes", 4), ("foot_force", 4), ("joy_valid", None),
              ("button0", None))
_FLAG_DTYPES = ("torch.bool", "torch.uint8")


def step_field_tensors(in_dim: int, device: int, fields: dict, vel_cmd, obs, action, qdes=None, cmd=None, reset=None,
                       action_seq=None, obs_seq=None, seq: bool = False):
    """Validates the arguments of PolicyBatch.step_fields before any native call.  fields: the eight raw-state tensors by
    name (RAW_FIELDS): float32 [B,w], foot_force int16 [B,4], joy_valid / button0 bool or uint8 [B].  vel_cmd float32
    [B,3], obs float32 [B,in_dim], action float32 [B,12], qdes float64 [B,12] or None, cmd uint8 [B,112] or None (not
    both None), reset bool / uint8 [B] or None.  Every tensor is a contiguous CUDA tensor on device ``device`` (duck-typed:
    this package does not import torch).  Returns B; raises TypeError / ValueError.
    seq=True validates PolicyBatch.step_fields_seq instead: the fields, reset, qdes and cmd carry a leading step dimension
    T ([T,B,w]), action_seq float32 [T,B,12] is required, obs_seq float32 [T,B,in_dim] or None, qdes and cmd may both be
    None; vel_cmd, obs and action keep their [B,w] shapes.  Returns (T, B)."""
    if seq:
        if action_seq is None:
            raise ValueError("action_seq is required: it receives every step's published action")
    elif qdes is None and cmd is None:
        raise ValueError("qdes and cmd are both None: the step needs at least one output")
    quat = fields["quat"]
    if not _is_device_tensor(quat):
        raise TypeError(f"quat must be a CUDA tensor, got {type(quat).__name__}")
    if len(quat.shape) != (3 if seq else 2):
        raise ValueError(f"quat must have shape ({'T, ' if seq else ''}B, 4), got {tuple(quat.shape)}")
    T = int(quat.shape[0]) if seq else None
    B = int(quat.shape[-2])
    lead = (T,) if seq else ()                 # the per-step tensors' leading dimension
    named = [(name, fields[name], lead + ((B, w) if w else (B,)), "torch.int16" if name == "foot_force" else
              _FLAG_DTYPES if w is None else "torch.float32") for name, w in RAW_FIELDS]
    named += [("vel_cmd", vel_cmd, (B, 3), "torch.float32"), ("obs", obs, (B, in_dim), "torch.float32"),
              ("action", action, (B, 12), "torch.float32")]
    if seq:
        named.append(("action_seq", action_seq, (T, B, 12), "torch.float32"))
        if obs_seq is not None:
            named.append(("obs_seq", obs_seq, (T, B, in_dim), "torch.float32"))
    if qdes is not None:
        named.append(("qdes", qdes, lead + (B, 12), "torch.float64"))
    if cmd is not None:
        named.append(("cmd", cmd, lead + (B, C.sizeof(capi.MotorCmd)), "torch.uint8"))
    if reset is not None:
        named.append(("reset", reset, lead + (B,), _FLAG_DTYPES))
    for name, a, shape, dtypes in named:
        if not _is_device_tensor(a):
            raise TypeError(f"{name} must be a CUDA tensor, got {type(a).__name__}")
        if str(a.dtype) not in ((dtypes,) if isinstance(dtypes, str) else dtypes):
            raise TypeError(f"{name} must be {' or '.join((dtypes,) if isinstance(dtypes, str) else dtypes)}, got {a.dtype}")
        if getattr(a.device, "type", None) != "cuda":
            raise TypeError(f"{name} is a tensor on {a.device}: pass a CUDA tensor")
        if a.device.index != device:
            raise ValueError(f"{name} is on cuda:{a.device.index}, the handle on cuda:{device}")
        if tuple(a.shape) != shape:
            raise ValueError(f"{name} must have shape {shape}, got {tuple(a.shape)}")
        if not a.is_contiguous():
            raise ValueError(f"{name} must be contiguous")
    return (T, B) if seq else B


def _ptr(a):
    return None if a is None else (a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())


def _ptr_array(arrays):
    """Host array of pointers (NULL for None), as go2p_set_weights* read them."""
    return (C.c_void_p * len(arrays))(*[_ptr(a) for a in arrays])


class ONNXActor:
    """Python face of the reference's ONNXActor: observation/action numpy buffers are bound at construction
    (they must be C-contiguous float32 and outlive the actor) and act() overwrites ``action`` in place."""

    def __init__(self, model_path: str, observation: np.ndarray, action: np.ndarray, log_level: int = 2,
                 b1_mode: int | None = None, device: int = 0):
        for name, a in (("observation", observation), ("action", action)):
            if not (isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags.c_contiguous and a.flags.writeable):
                raise TypeError(f"{name} must be a writable C-contiguous float32 numpy array")
        kw = {"log_level": log_level, "device": device}
        if b1_mode is not None:
            kw["b1_mode"] = b1_mode
        self._hd = _Handle(model_path, default_config(**kw))
        self.observation, self.action = observation, action
        fp = C.POINTER(C.c_float)
        capi.check(self._hd.lib.go2p_bind(self._hd.h, observation.ctypes.data_as(fp), observation.size,
                                          action.ctypes.data_as(fp), action.size))

    def act(self) -> None:
        capi.check(self._hd.lib.go2p_act(self._hd.h))

    def check_dims(self) -> bool:
        return self.observation.size == self._hd.in_dim and self.action.size == self._hd.out_dim

    def print_model_info(self) -> None:
        print(f"Input dimension: {self._hd.in_dim}")
        print(f"Output dimension: {self._hd.out_dim}")
        print(f"Input name: {self._hd.input_name}")
        print(f"Output name: {self._hd.output_name}")

    def stats(self, reset: bool = False) -> capi.B1Stats:
        s = capi.B1Stats()
        capi.check(self._hd.lib.go2p_b1_stats_get(self._hd.h, C.byref(s), int(reset)))
        return s

    def close(self) -> None:
        self._hd.close()


class Go2Controller:
    """publish()'s arithmetic as one device step: raw robot state in, ObservationAction + joint targets out."""

    def __init__(self, model_path: str = DEFAULT_MODEL, **cfg):
        self._hd = _Handle(model_path, default_config(**cfg))

    def step(self, raw: capi.RawState) -> capi.StepOut:
        out = capi.StepOut()
        capi.check(self._hd.lib.go2p_step_fused(self._hd.h, C.byref(raw), C.byref(out)))
        return out

    def step_cmd(self, raw: capi.RawState):
        """step() plus the same step's send_command arguments in Unitree motor order (controller.cpp:235-251)."""
        out, cmd = capi.StepOut(), capi.MotorCmd()
        capi.check(self._hd.lib.go2p_step_fused_cmd(self._hd.h, C.byref(raw), C.byref(out), C.byref(cmd)))
        return out, cmd

    def log_enable(self, capacity: int) -> None:
        """ObservationAction ring on the device (ObservationAction.msg:1-2); 0 turns it off."""
        capi.check(self._hd.lib.go2p_log_enable(self._hd.h, int(capacity)))

    def log_drain(self, max_records: int = 4096):
        """Records written since the last drain, oldest first: ([n, in_dim] observations, [n, 12] actions, dropped)."""
        rec = self._hd.in_dim + 12
        buf = np.zeros((max_records, rec), np.float32)
        n, dropped = C.c_int(), C.c_uint64()
        capi.check(self._hd.lib.go2p_log_drain(self._hd.h, buf.ctypes.data, max_records, C.byref(n), C.byref(dropped)))
        buf = buf[: n.value]
        return buf[:, : self._hd.in_dim].copy(), buf[:, self._hd.in_dim:].copy(), int(dropped.value)

    def closed_loop(self, raws, steps: int):
        """`steps` fused steps over the raw states (cycled), timed in native code.
        Returns (host_ns[steps], device_ns[steps], last StepOut)."""
        arr = (capi.RawState * len(raws))(*raws)
        host = np.zeros(steps, np.uint64)
        dev = np.zeros(steps, np.uint64)
        last = capi.StepOut()
        u64 = C.POINTER(C.c_uint64)
        capi.check(self._hd.lib.go2p_b1_closed_loop(self._hd.h, arr, len(raws), steps, host.ctypes.data_as(u64),
                                                    dev.ctypes.data_as(u64), C.byref(last)))
        return host, dev, last

    def selfdriven(self, raws, steps: int):
        """Profiling twin of the resident kernel: one bounded launch of `steps` closed-loop steps.
        Returns (last published action[12], elapsed ms)."""
        arr = (capi.RawState * len(raws))(*raws)
        act = np.zeros(12, np.float32)
        ms = C.c_float()
        capi.check(self._hd.lib.go2p_b1_selfdriven(self._hd.h, arr, len(raws), steps,
                                                   act.ctypes.data_as(C.POINTER(C.c_float)), C.byref(ms)))
        return act, float(ms.value)

    def reset(self) -> None:
        capi.check(self._hd.lib.go2p_reset_history(self._hd.h))

    def set_gains(self, kp: float, kd: float) -> None:
        capi.check(self._hd.lib.go2p_set_gains(self._hd.h, kp, kd))

    def set_weights(self, weights, biases=None, obs_mean=None, obs_std=None) -> None:
        """Replace the policy's weights (numpy float32 arrays; see PolicyBatch.set_weights).  The controller's history,
        previous action, joystick command and gains carry over to the next step."""
        self._hd.set_weights(weights, biases, obs_mean, obs_std, 0, host_only=True)

    def stop(self) -> None:
        capi.check(self._hd.lib.go2p_persistent_stop(self._hd.h))

    def stats(self, reset: bool = False) -> capi.B1Stats:
        s = capi.B1Stats()
        capi.check(self._hd.lib.go2p_b1_stats_get(self._hd.h, C.byref(s), int(reset)))
        return s

    def close(self) -> None:
        self._hd.close()


class PolicyBatch:
    """Batched inference.  Device tensors are passed as raw pointers (torch ``.data_ptr()`` or go2p_dev_alloc).

    ``precision`` of every method: capi.PREC_FP32 (the default: CUDA cores, the reference's 1e-5 contract),
    capi.PREC_FP32_TC (the same 1e-5 contract on the tensor cores, each operand split into three bf16 pieces; not
    bit-identical to PREC_FP32), capi.PREC_FP16 or capi.PREC_BF16 (16-bit operands, looser tolerances)."""

    def __init__(self, model_path: str = DEFAULT_MODEL, device: int = 0, **cfg):
        self._hd = _Handle(model_path, default_config(device=device, **cfg))
        self.in_dim, self.out_dim = self._hd.in_dim, self._hd.out_dim

    @property
    def info(self) -> capi.ModelInfo:
        return self._hd.info

    def infer_device(self, d_obs: int, d_act: int, B: int, precision: int = capi.PREC_FP32, stream: int = 0,
                     d_button0: int | None = None, d_qdes: int | None = None, flags: int = 0, d_cmd: int | None = None) -> None:
        """precision defaults to the reference's (fp32, 1e-5 contract); the tensor-core precisions are opt-in, and
        PREC_FP32_TC keeps the 1e-5 contract."""
        capi.check(self._hd.lib.go2p_infer_batch_cmd(self._hd.h, d_obs, d_button0, d_act, d_qdes, d_cmd, B, precision, flags,
                                                     stream or None))

    def time_device(self, d_obs: int, d_act: int, B: int, precision: int, iters: int, stream: int = 0,
                    d_button0: int | None = None, d_qdes: int | None = None, flags: int = 0) -> float:
        ms = C.c_float()
        capi.check(self._hd.lib.go2p_time_batch(self._hd.h, d_obs, d_button0, d_act, d_qdes, B, precision, flags,
                                                stream or None, iters, C.byref(ms)))
        return float(ms.value)

    def infer_host(self, obs: np.ndarray, act: np.ndarray | None = None, precision: int = capi.PREC_FP32) -> np.ndarray:
        obs = np.ascontiguousarray(obs, np.float32).reshape(-1, self.in_dim)
        if act is None:
            act = np.empty((obs.shape[0], self.out_dim), np.float32)
        capi.check(self._hd.lib.go2p_infer_batch_host(self._hd.h, obs.ctypes.data, act.ctypes.data, obs.shape[0], precision))
        return act

    def saturation_count(self, reset: bool = True, stream: int = 0) -> int:
        """(row, operand block) pairs clipped at +-65504 by fp16 launches made with F_SAT_COUNT since the last reset."""
        n = C.c_uint64()
        capi.check(self._hd.lib.go2p_saturation_count(self._hd.h, C.byref(n), int(reset), stream or None))
        return int(n.value)

    def last_launches(self) -> int:
        return int(self._hd.lib.go2p_last_launch_count(self._hd.h))

    def pinned(self, shape, dtype=np.float32) -> np.ndarray:
        """numpy view over cudaHostAlloc'ed memory (freed with the handle's process)."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        capi.check(self._hd.lib.go2p_host_alloc(self._hd.h, n, C.byref(p)))
        buf = (C.c_char * n).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def assemble_device(self, d_raw: int, d_prev_action: int | None, d_vel_cmd: int, d_obs: int, B: int, stream: int = 0):
        capi.check(self._hd.lib.go2p_assemble_batch(self._hd.h, d_raw, d_prev_action, d_vel_cmd, d_obs, B, stream or None))

    def step_device(self, d_raw: int, d_vel_cmd: int, d_obs: int, d_action: int, d_qdes: int, B: int,
                    precision: int = capi.PREC_FP32, stream: int = 0, d_reset: int | None = None) -> None:
        """Batched publish() (reference: controller.cpp:173-251 per robot): raw states -> observation history ->
        policy -> clamp/mask -> q_des, all on device buffers; d_action is the previous published action on entry.
        d_reset: device pointer to [B] bytes (e.g. a torch.bool tensor); robots with a non-zero byte start from the
        controller's initial state this step (go2p_step_batch_ex)."""
        if d_reset is None:
            capi.check(self._hd.lib.go2p_step_batch(self._hd.h, d_raw, d_vel_cmd, d_obs, d_action, d_qdes, B, precision,
                                                    stream or None))
        else:
            capi.check(self._hd.lib.go2p_step_batch_ex(self._hd.h, d_raw, d_reset, d_vel_cmd, d_obs, d_action, d_qdes, None,
                                                       B, precision, stream or None))

    def step_device_cmd(self, d_raw: int, d_vel_cmd: int, d_obs: int, d_action: int, d_qdes: int | None, d_cmd: int | None,
                        B: int, precision: int = capi.PREC_FP32, stream: int = 0, d_reset: int | None = None) -> None:
        """step_device ending in motor commands: d_cmd [B] go2p_motor_cmd (Unitree motor order), d_qdes may be None."""
        if d_reset is None:
            capi.check(self._hd.lib.go2p_step_batch_cmd(self._hd.h, d_raw, d_vel_cmd, d_obs, d_action, d_qdes, d_cmd, B,
                                                        precision, stream or None))
        else:
            capi.check(self._hd.lib.go2p_step_batch_ex(self._hd.h, d_raw, d_reset, d_vel_cmd, d_obs, d_action, d_qdes, d_cmd,
                                                       B, precision, stream or None))

    def step_fields(self, quat, gyro, q, dq, axes, foot_force, joy_valid, button0, vel_cmd, obs, action, qdes=None,
                    cmd=None, precision: int = capi.PREC_FP32, stream: int = 0, reset=None) -> None:
        """step_device_cmd with the raw states as one CUDA tensor per field, the way a GPU simulator keeps them
        (go2p_step_batch_fields): quat [B,4], gyro [B,3], q [B,12], dq [B,12], axes [B,4] float32, foot_force [B,4]
        int16 (Unitree order), joy_valid / button0 [B] bool or uint8.  vel_cmd [B,3], obs [B,in_dim] and action [B,12]
        (previous published action on entry) are the robots' state, updated in place; qdes float64 [B,12] and / or cmd
        uint8 [B,112] receive the outputs; reset: bool / uint8 [B] or None.  Every tensor contiguous and on the handle's
        device; a slice of a wider tensor must be made contiguous first.  B = 0 does nothing."""
        fields = dict(quat=quat, gyro=gyro, q=q, dq=dq, axes=axes, foot_force=foot_force, joy_valid=joy_valid,
                      button0=button0)
        B = step_field_tensors(self.in_dim, self._hd.cfg.device, fields, vel_cmd, obs, action, qdes, cmd, reset)
        if B == 0:
            return
        f = capi.RawFields(*[fields[name].data_ptr() for name, _ in RAW_FIELDS])
        capi.check(self._hd.lib.go2p_step_batch_fields(self._hd.h, C.byref(f), _ptr(reset), vel_cmd.data_ptr(),
                                                       obs.data_ptr(), action.data_ptr(), _ptr(qdes), _ptr(cmd), B,
                                                       precision, stream or None))

    def step_fields_seq(self, quat, gyro, q, dq, axes, foot_force, joy_valid, button0, vel_cmd, obs, action, action_seq,
                        qdes_seq=None, cmd_seq=None, obs_seq=None, reset=None, precision: int = capi.PREC_FP32,
                        stream: int = 0) -> None:
        """T consecutive step_fields steps in one call (go2p_step_batch_fields_seq), e.g. to replay recorded sensor
        streams closed-loop: every field and reset as in step_fields with a leading step dimension, [T,B,w].  vel_cmd,
        obs and action are the robots' state before step 0 on entry and after step T-1 on return.  action_seq float32
        [T,B,12] receives every step's published action; qdes_seq float64 [T,B,12], cmd_seq uint8 [T,B,112] and obs_seq
        float32 [T,B,in_dim] (every step's observation) are optional.  T or B = 0 does nothing."""
        fields = dict(quat=quat, gyro=gyro, q=q, dq=dq, axes=axes, foot_force=foot_force, joy_valid=joy_valid,
                      button0=button0)
        T, B = step_field_tensors(self.in_dim, self._hd.cfg.device, fields, vel_cmd, obs, action, qdes_seq, cmd_seq, reset,
                                  action_seq=action_seq, obs_seq=obs_seq, seq=True)
        if T == 0 or B == 0:
            return
        f = capi.RawFields(*[fields[name].data_ptr() for name, _ in RAW_FIELDS])
        capi.check(self._hd.lib.go2p_step_batch_fields_seq(self._hd.h, C.byref(f), T, _ptr(reset), vel_cmd.data_ptr(),
                                                           obs.data_ptr(), action.data_ptr(), action_seq.data_ptr(),
                                                           _ptr(qdes_seq), _ptr(cmd_seq), _ptr(obs_seq), B, precision,
                                                           stream or None))

    def step_host(self, raw: np.ndarray, action: np.ndarray, cmd: np.ndarray | None = None,
                  precision: int = capi.PREC_FP32, reset: np.ndarray | None = None) -> None:
        """Closed-loop step for len(raw) robots from host buffers; per-robot history stays on the device.
        raw: uint8 [B, 156] (go2p_raw_state records), action: float32 [B, 12] out, cmd: uint8 [B, 112] out or None,
        reset: bool / uint8 [B] or None -- robots to start from the controller's initial state this step."""
        B = raw.shape[0]
        cmd_p = cmd.ctypes.data if cmd is not None else None
        if reset is None:
            capi.check(self._hd.lib.go2p_step_batch_host(self._hd.h, raw.ctypes.data, action.ctypes.data, cmd_p, B, precision))
        else:
            reset = host_reset_mask(reset, B)
            capi.check(self._hd.lib.go2p_step_batch_host_ex(self._hd.h, raw.ctypes.data, reset.ctypes.data, action.ctypes.data,
                                                            cmd_p, B, precision))

    def step_host_reset(self) -> None:
        capi.check(self._hd.lib.go2p_step_batch_host_reset(self._hd.h))

    def set_weights(self, weights, biases=None, obs_mean=None, obs_std=None, stream: int = 0) -> None:
        """Replace the weights of every layer; the topology stays.  weights[l]: float32 [dims[l+1], dims[l]] (the layout
        of torch nn.Linear.weight), biases: None or float32 [dims[l+1]] (None) per layer, obs_mean / obs_std: float32
        [in_dim], both or neither, an observation normaliser (x - mean) / std folded into the first layer.
        numpy arrays: synchronous (go2p_set_weights_host).  CUDA tensors on the handle's device: packed on the device,
        ordered on ``stream`` (go2p_set_weights); keep them alive until the stream has passed the update.  Robot state
        kept by the handle (step_host, the batch-1 controller) carries over."""
        self._hd.set_weights(weights, biases, obs_mean, obs_std, stream, host_only=False)

    def close(self) -> None:
        self._hd.close()


class Fleet:
    """One process, several GPUs: rows are split into contiguous shards, one handle + host thread per device
    (include/go2policy.h: go2p_fleet_*).  No data crosses between devices.  ``precision`` as in PolicyBatch: PREC_FP32
    by default, PREC_FP32_TC for the same accuracy on the tensor cores, PREC_FP16 / PREC_BF16."""

    def __init__(self, model_path: str = DEFAULT_MODEL, devices=(0,), **cfg):
        self.lib = capi.load()
        self.f = C.c_void_p()
        c = default_config(**cfg)
        dev = (C.c_int32 * len(devices))(*devices)
        capi.check(self.lib.go2p_fleet_create(os.fspath(model_path).encode(), C.byref(c), dev, len(devices), C.byref(self.f)))
        self.n_devices = len(devices)
        self.model_path = os.fspath(model_path)

    def infer_host(self, obs: np.ndarray, act: np.ndarray, precision: int = capi.PREC_FP32) -> None:
        capi.check(self.lib.go2p_fleet_infer_host(self.f, obs.ctypes.data, act.ctypes.data, obs.shape[0], precision))

    def step_host(self, raw: np.ndarray, action: np.ndarray, cmd: np.ndarray | None = None, precision: int = capi.PREC_FP32,
                  reset: np.ndarray | None = None) -> None:
        """PolicyBatch.step_host over the devices' shards; reset: bool / uint8 [B] or None."""
        cmd_p = cmd.ctypes.data if cmd is not None else None
        if reset is None:
            capi.check(self.lib.go2p_fleet_step_host(self.f, raw.ctypes.data, action.ctypes.data, cmd_p, raw.shape[0], precision))
        else:
            reset = host_reset_mask(reset, raw.shape[0])
            capi.check(self.lib.go2p_fleet_step_host_ex(self.f, raw.ctypes.data, reset.ctypes.data, action.ctypes.data, cmd_p,
                                                        raw.shape[0], precision))

    def set_weights(self, weights, biases=None, obs_mean=None, obs_std=None) -> None:
        """PolicyBatch.set_weights with numpy arrays, on every device of the fleet (go2p_fleet_set_weights_host)."""
        info = capi.ModelInfo()
        capi.check(self.lib.go2p_inspect_model(self.model_path.encode(), C.byref(info), None))
        if weight_arrays([info.dims[i] for i in range(info.n_layers + 1)], weights, biases, obs_mean, obs_std) != "host":
            raise TypeError("Fleet.set_weights takes numpy arrays (host memory)")
        capi.check(self.lib.go2p_fleet_set_weights_host(self.f, _ptr_array(weights),
                                                        _ptr_array(biases) if biases is not None else None, len(weights),
                                                        _ptr(obs_mean), _ptr(obs_std)))

    def close(self) -> None:
        if self.f:
            self.lib.go2p_fleet_destroy(self.f)
            self.f = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def shard_rows(total_rows: int, n: int, i: int):
    """(begin, end) of shard i of n as the C ABI splits them (go2p_shard_rows)."""
    b, e = C.c_int64(), C.c_int64()
    capi.check(capi.load().go2p_shard_rows(total_rows, n, i, C.byref(b), C.byref(e)))
    return b.value, e.value
