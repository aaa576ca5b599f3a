"""ctypes binding of include/go2policy.h (the C ABI the reference's FFI would bind)."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

GO2P_DOF = 12
GO2P_FRAME = 49
GO2P_MAX_HISTORY = 8
GO2P_MAX_LAYERS = 8

OK, ERR_INVALID, ERR_IO, ERR_MODEL, ERR_CUDA, ERR_NO_DEVICE, ERR_UNSUPPORTED, ERR_STATE, ERR_TIMEOUT = range(9)
PREC_FP32, PREC_BF16, PREC_FP16 = 0, 1, 2
PREC_FP32_TC = 4               # fp32 accuracy on the tensor cores (three bf16 pieces per operand); 3 is rejected
B1_PERSISTENT, B1_GRAPH, B1_LAUNCH = 0, 1, 2
F_CLAMP_MASK, F_QDES, F_MOTOR_CMD, F_SAT_COUNT = 1, 2, 4, 8

PREC_NAMES = {"fp32": PREC_FP32, "bf16": PREC_BF16, "fp16": PREC_FP16}


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("b1_mode", C.c_int32), ("history", C.c_int32),
        ("action_limit", C.c_float), ("action_scale", C.c_double), ("q0", C.c_double * GO2P_DOF),
        ("foot_threshold", C.c_int32), ("kp", C.c_float), ("kd", C.c_float), ("kp_deadman", C.c_float),
        ("log_level", C.c_int32), ("timeout_ms", C.c_int32), ("idle_exit_ms", C.c_int32),
    ]


class RawState(C.Structure):
    _fields_ = [
        ("quat", C.c_float * 4), ("gyro", C.c_float * 3), ("q", C.c_float * 12), ("dq", C.c_float * 12),
        ("axes", C.c_float * 4), ("foot_force", C.c_int16 * 4), ("joy_valid", C.c_int32), ("button0", C.c_int32),
    ]


class RawFields(C.Structure):
    """Device pointers to the per-field raw states of B robots (include/go2policy.h: go2p_raw_fields)."""
    _fields_ = [(name, C.c_void_p) for name in ("quat", "gyro", "q", "dq", "axes", "foot_force", "joy_valid", "button0")]


class StepOut(C.Structure):
    _fields_ = [
        ("observation", C.c_float * (GO2P_FRAME * GO2P_MAX_HISTORY)), ("action_raw", C.c_float * 12),
        ("action", C.c_float * 12), ("q_des", C.c_double * 12), ("kp", C.c_double), ("kd", C.c_double),
        ("device_ns", C.c_uint64),
    ]


class MotorCmd(C.Structure):
    """send_command arguments in Unitree motor order (include/go2policy.h: go2p_motor_cmd)."""
    _fields_ = [("q_des", C.c_double * GO2P_DOF), ("kp", C.c_double), ("kd", C.c_double)]


class ModelInfo(C.Structure):
    _fields_ = [
        ("in_dim", C.c_int32), ("out_dim", C.c_int32), ("n_layers", C.c_int32),
        ("dims", C.c_int32 * (GO2P_MAX_LAYERS + 1)), ("has_elu", C.c_int32 * GO2P_MAX_LAYERS),
        ("elu_alpha", C.c_float * GO2P_MAX_LAYERS), ("input_name", C.c_char_p), ("output_name", C.c_char_p),
        ("n_params", C.c_int64), ("sm_count", C.c_int32), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
        ("tensor_core_path", C.c_int32),
    ]


class B1Stats(C.Structure):
    _fields_ = [("steps", C.c_uint64), ("device_ns_min", C.c_uint64), ("device_ns_max", C.c_uint64),
                ("device_ns_sum", C.c_uint64)]


# every symbol include/go2policy.h declares: name -> (restype, argtypes)
_H = C.c_void_p
_fp = C.POINTER(C.c_float)
SIGNATURES = {
    "go2p_config_default": (None, [C.POINTER(Config)]),
    "go2p_create": (C.c_int, [C.c_char_p, C.POINTER(Config), C.POINTER(_H)]),
    "go2p_inspect_model": (C.c_int, [C.c_char_p, C.POINTER(ModelInfo), C.POINTER(C.c_double)]),
    "go2p_destroy": (C.c_int, [_H]),
    "go2p_model_info": (C.c_int, [_H, C.POINTER(ModelInfo)]),
    "go2p_last_error": (C.c_char_p, []),
    "go2p_abi_version": (C.c_int, []),
    "go2p_bind": (C.c_int, [_H, _fp, C.c_size_t, _fp, C.c_size_t]),
    "go2p_act": (C.c_int, [_H]),
    "go2p_step_fused": (C.c_int, [_H, C.POINTER(RawState), C.POINTER(StepOut)]),
    "go2p_b1_closed_loop": (C.c_int, [_H, C.POINTER(RawState), C.c_int, C.c_int, C.POINTER(C.c_uint64),
                                       C.POINTER(C.c_uint64), C.POINTER(StepOut)]),
    "go2p_b1_selfdriven": (C.c_int, [_H, C.POINTER(RawState), C.c_int, C.c_int, _fp, _fp]),
    "go2p_reset_history": (C.c_int, [_H]),
    "go2p_set_gains": (C.c_int, [_H, C.c_float, C.c_float]),
    "go2p_b1_stats_get": (C.c_int, [_H, C.POINTER(B1Stats), C.c_int]),
    "go2p_persistent_start": (C.c_int, [_H]),
    "go2p_persistent_stop": (C.c_int, [_H]),
    "go2p_infer_batch": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "go2p_infer_batch_ex": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                       C.c_uint32, C.c_void_p]),
    "go2p_infer_batch_host": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "go2p_assemble_batch": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "go2p_step_batch": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                  C.c_void_p]),
    "go2p_last_launch_count": (C.c_int, [_H]),
    "go2p_saturation_count": (C.c_int, [_H, C.POINTER(C.c_uint64), C.c_int, C.c_void_p]),
    "go2p_infer_batch_cmd": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                        C.c_uint32, C.c_void_p]),
    "go2p_step_batch_cmd": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_int, C.c_void_p]),
    "go2p_step_batch_ex": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int64, C.c_int, C.c_void_p]),
    "go2p_step_batch_fields": (C.c_int, [_H, C.POINTER(RawFields), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "go2p_step_batch_fields_seq": (C.c_int, [_H, C.POINTER(RawFields), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                              C.c_int, C.c_void_p]),
    "go2p_step_fused_cmd": (C.c_int, [_H, C.POINTER(RawState), C.POINTER(StepOut), C.POINTER(MotorCmd)]),
    "go2p_motor_order": (C.c_int, [C.POINTER(C.c_int32)]),
    "go2p_step_batch_host": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "go2p_step_batch_host_reset": (C.c_int, [_H]),
    "go2p_step_batch_host_ex": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "go2p_log_enable": (C.c_int, [_H, C.c_int]),
    "go2p_log_drain": (C.c_int, [_H, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "go2p_fleet_create": (C.c_int, [C.c_char_p, C.POINTER(Config), C.POINTER(C.c_int32), C.c_int, C.POINTER(C.c_void_p)]),
    "go2p_fleet_destroy": (C.c_int, [C.c_void_p]),
    "go2p_fleet_device_count": (C.c_int, [C.c_void_p]),
    "go2p_shard_rows": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "go2p_fleet_infer_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "go2p_fleet_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "go2p_fleet_step_host_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "go2p_set_weights": (C.c_int, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "go2p_set_weights_host": (C.c_int, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_void_p,
                                        C.c_void_p]),
    "go2p_fleet_set_weights_host": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                              C.c_void_p, C.c_void_p]),
    "go2p_dev_alloc": (C.c_int, [_H, C.c_size_t, C.POINTER(C.c_void_p)]),
    "go2p_dev_free": (C.c_int, [_H, C.c_void_p]),
    "go2p_host_alloc": (C.c_int, [_H, C.c_size_t, C.POINTER(C.c_void_p)]),
    "go2p_host_free": (C.c_int, [_H, C.c_void_p]),
    "go2p_memcpy_h2d": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "go2p_memcpy_d2h": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "go2p_stream_sync": (C.c_int, [_H, C.c_void_p]),
    "go2p_time_batch": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_uint32,
                                   C.c_void_p, C.c_int, C.POINTER(C.c_float)]),
}

_lib = None


class Go2PolicyError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"go2policy error {code}: {msg}")
        self.code = code


def load(build_if_missing: bool = True):
    """dlopen the in-tree libgo2policy.so.  There is no Python/CPU fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB):
        if not build_if_missing:
            raise OSError(f"{_build.LIB} is missing (run python -m go2_onnx_controller_b200.build)")
        _build.build()
    lib = C.CDLL(_build.LIB)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # raises AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != OK:
        raise Go2PolicyError(rc, load().go2p_last_error().decode(errors="replace"))
