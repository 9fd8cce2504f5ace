"""quadrupedal_loco_b200 -- B200-native batched Go1 gait-planning MPC (host-side Python binding).

The product is libgo1mpc.so (CUDA, sm_100a) behind the C ABI in include/go1mpc.h; this
package is the thin ctypes binding tests and bench.py use.  PyTorch is only used by
callers for device memory and streams.  There is no CPU fallback: if the library is
missing or no CUDA device is usable, calls raise.
"""
from .binding import (  # noqa: F401
    Go1Mpc, Go1MpcError, load_library, library_path, body_in_stride, body_out_stride,
    body_diag_stride, pack_body_inputs, EXPORTED_SYMBOLS, QP_ITERS, BODY_DIAG_ACTIVE,
    STEP_STATE, STEP_IN, STEP_OUT, STEP_DIAG, BODY_TICK_OUT, body_tick_in_stride, split_body_record,
    ControlTick, COMPACT_DOUBLES, lpf_coefficients, GaitStackTick, STACK_SENSOR_ROWS, STACK_SLOTS_MAX, STACK_ROW_NLP,
    STACK_ROW_GAIT, STACK_ROW_RT2NRT, STACK_ROW_WALKDTIME, STACK_ROW_TRAJ, STACK_ROW_RT,
    ServoStackTick, SERVO_TICKS_MAX, SERVO_STATE_ROWS, SERVO_ROW_Q, SERVO_ROW_HOMING, SERVO_ROW_LPF, SERVO_LPF_SLOTS,
    GaitStackClockedTick, GaitStackReset, ServoTorqueTick, SERVO_FORCE_ROWS, FarmColumns, FarmCopy,
    HEALTH_ROWS, HEALTH_PLAN_OK, HEALTH_PLAN_INFEASIBLE, HEALTH_PLAN_FAILED, HEALTH_BODY_OK, HEALTH_BODY_INFEASIBLE,
    HEALTH_BODY_FAILED, HEALTH_GRF_OK, HEALTH_GRF_FAILED, HEALTH_GRF_FALLBACK, HEALTH_IK_CAP, HEALTH_NONFINITE, HEALTH_EVENTS,
)
from ._build import build  # noqa: F401

__all__ = [
    "Go1Mpc", "Go1MpcError", "load_library", "library_path", "build", "body_in_stride",
    "body_out_stride", "body_diag_stride", "pack_body_inputs", "EXPORTED_SYMBOLS", "QP_ITERS",
    "BODY_DIAG_ACTIVE", "STEP_STATE", "STEP_IN", "STEP_OUT", "STEP_DIAG", "BODY_TICK_OUT", "body_tick_in_stride",
    "split_body_record", "ControlTick", "COMPACT_DOUBLES", "lpf_coefficients",
    "GaitStackTick", "STACK_SENSOR_ROWS", "STACK_SLOTS_MAX", "STACK_ROW_NLP", "STACK_ROW_GAIT", "STACK_ROW_RT2NRT",
    "STACK_ROW_WALKDTIME", "STACK_ROW_TRAJ", "STACK_ROW_RT",
    "ServoStackTick", "SERVO_TICKS_MAX", "SERVO_STATE_ROWS", "SERVO_ROW_Q", "SERVO_ROW_HOMING", "SERVO_ROW_LPF", "SERVO_LPF_SLOTS",
    "GaitStackClockedTick", "GaitStackReset", "ServoTorqueTick", "SERVO_FORCE_ROWS", "FarmColumns", "FarmCopy",
    "HEALTH_ROWS", "HEALTH_PLAN_OK", "HEALTH_PLAN_INFEASIBLE", "HEALTH_PLAN_FAILED", "HEALTH_BODY_OK", "HEALTH_BODY_INFEASIBLE",
    "HEALTH_BODY_FAILED", "HEALTH_GRF_OK", "HEALTH_GRF_FAILED", "HEALTH_GRF_FALLBACK", "HEALTH_IK_CAP", "HEALTH_NONFINITE",
    "HEALTH_EVENTS",
]
