"""ctypes binding of include/go1mpc.h.  Mirrors the C ABI one to one."""
import ctypes
import os

import numpy as np

from . import _build

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)

# every symbol include/go1mpc.h declares (tests check the .so exports all of them)
EXPORTED_SYMBOLS = [
    "go1mpc_version", "go1mpc_config_default", "go1mpc_create", "go1mpc_destroy",
    "go1mpc_last_error", "go1mpc_device", "go1mpc_launch_count", "go1mpc_synchronize",
    "go1mpc_stream", "go1mpc_sm_count", "go1mpc_copy_device_async",
    "go1mpc_qp_solve_batch", "go1mpc_qp_solve_batch_host",
    "go1mpc_body_in_stride", "go1mpc_body_out_stride", "go1mpc_body_diag_stride",
    "go1mpc_body_mpc_step_batch", "go1mpc_body_mpc_step_batch_host", "go1mpc_body_handover_total", "go1mpc_body_guard_trips",
    "go1mpc_body_model", "go1mpc_body_default_tx", "go1mpc_measure_dfma_peak",
    "go1mpc_step_timing_step_batch", "go1mpc_step_timing_step_batch_host", "go1mpc_step_default_state",
    "go1mpc_body_mpc_step_batch_host_async", "go1mpc_step_timing_step_batch_host_async",
    "go1mpc_body_tick_in_stride", "go1mpc_body_mpc_step_batch_resident_host_async",
    "go1mpc_foot_trajectory_batch", "go1mpc_foot_trajectory_batch_host", "go1mpc_foot_default_state",
    "go1mpc_leg_fk_batch", "go1mpc_leg_ik_batch", "go1mpc_servo_kin_tick_batch", "go1mpc_fused_tick_batch",
    "go1mpc_grf_force_opt_batch", "go1mpc_grf_force_distribution_batch", "go1mpc_grf_joint_torques_batch", "go1mpc_ref_interp_batch", "go1mpc_ref_interp_model",
    "go1mpc_control_tick_host_async", "go1mpc_pack_compact_batch", "go1mpc_stream_wait", "go1mpc_graph_capture_begin",
    "go1mpc_graph_capture_end", "go1mpc_graph_launch", "go1mpc_graph_destroy",
    "go1mpc_rt_node_state_doubles", "go1mpc_rt_node_default_state", "go1mpc_rt_node_tick_batch", "go1mpc_rt_node_tick_msgs_batch",
    "go1mpc_gather_create", "go1mpc_gather_destroy", "go1mpc_gather_export", "go1mpc_gather_import", "go1mpc_gather_dest",
    "go1mpc_gather_block", "go1mpc_gather_acquire", "go1mpc_gather_publish", "go1mpc_gather_wait_all", "go1mpc_gather_release",
    "go1mpc_gather_status", "go1mpc_body_phase_timing", "go1mpc_body_phase_ms", "go1mpc_forget_buffer", "go1mpc_lpf_coefficients", "go1mpc_lpf_batch", "go1mpc_force_filter_batch",
    "go1mpc_nlp_node_state_doubles", "go1mpc_nlp_node_default_state", "go1mpc_nlp_walkdtime_max", "go1mpc_nlp_t_end_footstep",
    "go1mpc_nlp_node_tick_batch", "go1mpc_foot_trajectory_stop_batch", "go1mpc_nlp_node_tick_batch_host", "go1mpc_rt_node_tick_batch_host", "go1mpc_foot_trajectory_stop_batch_host",
    "go1mpc_grf_force_opt_batch_host", "go1mpc_grf_force_distribution_batch_host", "go1mpc_grf_joint_torques_batch_host", "go1mpc_leg_fk_batch_host", "go1mpc_leg_ik_batch_host",
    "go1mpc_gait_stack_state_doubles", "go1mpc_gait_stack_default_state", "go1mpc_gait_stack_tick_host_async",
    "go1mpc_servo_stack_tick_async", "go1mpc_gait_stack_tick_clocked_async", "go1mpc_gait_stack_reset_async",
    "go1mpc_servo_torque_tick_async", "go1mpc_farm_copy_async",
    "go1mpc_gait_stack_tick_clocked_health_async", "go1mpc_servo_torque_tick_health_async",
]


QP_ITERS = 6           # GO1MPC_ITERS
BODY_DIAG_ACTIVE = 10  # first int of the final active set in a body-MPC diag record


class Go1MpcError(RuntimeError):
    pass


class BodyCfg(ctypes.Structure):
    _fields_ = [
        ("dt_mpc", ctypes.c_double), ("dt_slow", ctypes.c_double), ("tstep", ctypes.c_double),
        ("height_offset_time", ctypes.c_double), ("g", ctypes.c_double), ("mass", ctypes.c_double),
        ("j_ini", ctypes.c_double), ("foot_length", ctypes.c_double), ("foot_width", ctypes.c_double),
        ("theta_lim", ctypes.c_double), ("torque_lim", ctypes.c_double), ("Rtheta", ctypes.c_double),
        ("alphatheta", ctypes.c_double), ("beltatheta", ctypes.c_double), ("gama_zmp", ctypes.c_double),
        ("lamda", ctypes.c_double * 4),
    ]


class StepCfg(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in (
        "dt Wn ggg t_min t_max footx_max footx_min footx_vmax footx_vmin footy_vmax footy_vmin comax_max comax_min "
        "comay_max comay_min aax aay aaxv aayv bbx bby rr1 rr2 half_hip_width foot_width").split()] + [
        ("lamda", ctypes.c_double * 4), ("hcom", ctypes.c_double), ("ext_height", ctypes.c_int), ("reserved", ctypes.c_int),
        ("stepwidth0", ctypes.c_double), ("lift_height", ctypes.c_double)]


class Cfg(ctypes.Structure):
    _fields_ = [("body", BodyCfg), ("step", StepCfg), ("qp_iter_cap_scale", ctypes.c_int), ("reserved", ctypes.c_int * 7)]


STEP_STATE, STEP_IN, STEP_OUT, STEP_DIAG = 202, 20, 38, 60


_LIB = None


def library_path():
    """In-tree libgo1mpc.so; GO1MPC_LIB overrides it (A/B runs of differently tuned builds)."""
    return os.environ.get("GO1MPC_LIB") or _build.LIB


def load_library():
    """Load libgo1mpc.so (never builds implicitly on a GPU box: the .so ships in-tree)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise Go1MpcError(
            f"{path} is missing: build it with `python -m quadrupedal_loco_b200._build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    lib.go1mpc_version.restype = ctypes.c_char_p
    lib.go1mpc_last_error.restype = ctypes.c_char_p
    lib.go1mpc_last_error.argtypes = [ctypes.c_void_p]
    lib.go1mpc_launch_count.restype = ctypes.c_longlong
    lib.go1mpc_launch_count.argtypes = [ctypes.c_void_p]
    lib.go1mpc_create.argtypes = [ctypes.POINTER(Cfg), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
    lib.go1mpc_destroy.argtypes = [ctypes.c_void_p]
    lib.go1mpc_destroy.restype = None
    lib.go1mpc_device.argtypes = [ctypes.c_void_p]
    lib.go1mpc_synchronize.argtypes = [ctypes.c_void_p]
    lib.go1mpc_stream.argtypes = [ctypes.c_void_p]
    lib.go1mpc_stream.restype = ctypes.c_void_p
    lib.go1mpc_sm_count.argtypes = [ctypes.c_void_p]
    lib.go1mpc_copy_device_async.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    vp = ctypes.c_void_p
    lib.go1mpc_qp_solve_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [vp] * 12 + [vp]
    lib.go1mpc_qp_solve_batch_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [vp] * 12
    lib.go1mpc_body_mpc_step_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
    lib.go1mpc_body_mpc_step_batch_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    lib.go1mpc_body_model.argtypes = [vp, ctypes.c_int] + [vp] * 6
    lib.go1mpc_body_handover_total.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong)]
    lib.go1mpc_body_guard_trips.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong)]
    lib.go1mpc_body_default_tx.argtypes = [vp, vp]
    lib.go1mpc_measure_dfma_peak.argtypes = [vp, ctypes.c_int, c_double_p]
    lib.go1mpc_step_timing_step_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp]
    lib.go1mpc_step_timing_step_batch_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp]
    lib.go1mpc_step_default_state.argtypes = [vp] + [ctypes.c_double] * 4 + [vp]
    lib.go1mpc_body_mpc_step_batch_host_async.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    lib.go1mpc_step_timing_step_batch_host_async.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp]
    lib.go1mpc_body_tick_in_stride.argtypes = [ctypes.c_int]
    lib.go1mpc_body_mpc_step_batch_resident_host_async.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp]
    lib.go1mpc_foot_trajectory_batch.argtypes = [vp, ctypes.c_int] + [vp] * 7
    lib.go1mpc_foot_trajectory_batch_host.argtypes = [vp, ctypes.c_int] + [vp] * 6
    lib.go1mpc_foot_default_state.argtypes = [vp, vp]
    lib.go1mpc_leg_fk_batch.argtypes = [vp, ctypes.c_int] + [vp] * 7
    lib.go1mpc_grf_force_opt_batch.argtypes = [vp, ctypes.c_int, vp, vp, vp, vp]
    lib.go1mpc_grf_force_distribution_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_double] + [vp] * 7
    lib.go1mpc_ref_interp_model.argtypes = [vp, vp, vp]
    lib.go1mpc_ref_interp_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_double, vp, vp, vp]
    lib.go1mpc_grf_force_opt_batch_host.argtypes = [vp, ctypes.c_int, vp, vp, vp]
    lib.go1mpc_grf_force_distribution_batch_host.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_double] + [vp] * 6
    lib.go1mpc_grf_joint_torques_batch_host.argtypes = [vp, ctypes.c_int] + [vp] * 7 + [ctypes.c_longlong, ctypes.c_longlong, vp]
    lib.go1mpc_grf_joint_torques_batch.argtypes = [vp, ctypes.c_int] + [vp] * 7 + [ctypes.c_longlong, ctypes.c_longlong, vp, vp]
    lib.go1mpc_servo_kin_tick_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_double] + [vp] * 10
    lib.go1mpc_fused_tick_batch.argtypes = [vp, ctypes.c_int, ctypes.POINTER(FusedTick), vp]
    lib.go1mpc_leg_ik_batch.argtypes = [vp, ctypes.c_int] + [vp] * 9
    lib.go1mpc_control_tick_host_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(ControlTick), vp]
    lib.go1mpc_pack_compact_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int] + [vp] * 6
    lib.go1mpc_rt_node_state_doubles.argtypes = [ctypes.c_int]
    lib.go1mpc_rt_node_default_state.argtypes = [vp, ctypes.c_int, vp]
    lib.go1mpc_rt_node_tick_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int] + [vp] * 10
    lib.go1mpc_rt_node_tick_msgs_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int] + [vp] * 9
    lib.go1mpc_body_phase_timing.argtypes = [vp, ctypes.c_int]
    lib.go1mpc_body_phase_ms.argtypes = [vp, vp]
    lib.go1mpc_forget_buffer.argtypes = [vp, vp]
    lib.go1mpc_lpf_coefficients.argtypes = [ctypes.c_double, ctypes.c_double, vp]
    lib.go1mpc_lpf_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int] + [vp] * 6
    lib.go1mpc_force_filter_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int] + [vp] * 4
    lib.go1mpc_nlp_node_state_doubles.argtypes = []
    lib.go1mpc_nlp_node_default_state.argtypes = [vp, vp]
    lib.go1mpc_nlp_walkdtime_max.argtypes = [vp]
    lib.go1mpc_nlp_t_end_footstep.argtypes = [vp]
    lib.go1mpc_nlp_node_tick_batch.argtypes = [vp, ctypes.c_int] + [vp] * 8
    lib.go1mpc_foot_trajectory_stop_batch.argtypes = [vp, ctypes.c_int] + [vp] * 9
    lib.go1mpc_foot_trajectory_stop_batch_host.argtypes = [vp, ctypes.c_int] + [vp] * 9
    lib.go1mpc_nlp_node_tick_batch_host.argtypes = [vp, ctypes.c_int] + [vp] * 7
    lib.go1mpc_rt_node_tick_batch_host.argtypes = [vp, ctypes.c_int, ctypes.c_int] + [vp] * 6
    lib.go1mpc_stream_wait.argtypes = [vp, vp, vp]
    lib.go1mpc_graph_capture_begin.argtypes = [vp, vp]
    lib.go1mpc_graph_capture_end.argtypes = [vp, vp, ctypes.POINTER(ctypes.c_void_p)]
    lib.go1mpc_graph_launch.argtypes = [vp, vp, vp]
    lib.go1mpc_graph_destroy.argtypes = [vp, vp]
    lib.go1mpc_leg_fk_batch_host.argtypes = [vp, ctypes.c_int] + [vp] * 6
    lib.go1mpc_leg_ik_batch_host.argtypes = [vp, ctypes.c_int] + [vp] * 8
    lib.go1mpc_gait_stack_state_doubles.argtypes = [ctypes.c_int]
    lib.go1mpc_gait_stack_default_state.argtypes = [vp, ctypes.c_int, vp]
    lib.go1mpc_gait_stack_tick_host_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(GaitStackTick), vp]
    lib.go1mpc_servo_stack_tick_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(ServoStackTick), vp]
    lib.go1mpc_gait_stack_tick_clocked_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(GaitStackClockedTick), vp]
    lib.go1mpc_gait_stack_reset_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(GaitStackReset), vp]
    lib.go1mpc_servo_torque_tick_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(ServoTorqueTick), vp]
    lib.go1mpc_farm_copy_async.argtypes = [vp, ctypes.POINTER(FarmCopy), vp]
    lib.go1mpc_gait_stack_tick_clocked_health_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(GaitStackClockedTick), vp, vp]
    lib.go1mpc_servo_torque_tick_health_async.argtypes = [vp, ctypes.c_int, ctypes.POINTER(ServoTorqueTick), vp, vp]
    _LIB = lib
    return lib


def lpf_coefficients(fsampling, fcutoff):
    """butterworthLPF::init (host, no GPU needed): b0 b1 b2 a1 a2 a."""
    c = np.zeros(6)
    rc = load_library().go1mpc_lpf_coefficients(float(fsampling), float(fcutoff), _ptr(c))
    if rc != 0:
        raise Go1MpcError(f"lpf_coefficients: code {rc}")
    return c


def body_in_stride(nh):
    s = 36 + 11 * nh
    return (s + 1) & ~1


def body_out_stride(nh):
    s = 18 + 2 * nh + 1
    return (s + 1) & ~1


def body_diag_stride(nh):
    return BODY_DIAG_ACTIVE + 2 * nh


BODY_TICK_OUT = 20     # GO1MPC_BODY_TICK_OUT: out14 | theta(4) | cost | 0


def body_tick_in_stride(nh):
    return (9 + 9 * nh + 1) & ~1


def split_body_record(nh, rec):
    """Full input records -> (tx [B,28], x_warm [B,2nh], tick records [B, body_tick_in_stride]) of the
    device-resident entry go1mpc_body_mpc_step_batch_resident_host_async."""
    B = rec.shape[0]
    tx = np.zeros((B, 28)); tx[:, :27] = rec[:, :27]
    tick = np.zeros((B, body_tick_in_stride(nh)))
    tick[:, :9] = rec[:, 27:36]
    tick[:, 9:9 + 9 * nh] = rec[:, 36 + 2 * nh:36 + 11 * nh]
    return tx, rec[:, 36:36 + 2 * nh].copy(), tick


def pack_body_inputs(nh, tick, tx, theta, bodyangle_state, x_warm, refs):
    """Pack per-instance arrays into the in-record layout of go1mpc_body_mpc_step_batch.

    tick [B] int, tx [B,27], theta [B,4], bodyangle_state [B,4], x_warm [B,2nh],
    refs [B,9,nh] (zmp x,y | bodyangle x,y | rfoot x,y | lfoot x,y | comacc_z).
    """
    B = len(tick)
    rec = np.zeros((B, body_in_stride(nh)), dtype=np.float64)
    rec[:, 0:27] = tx
    rec[:, 27] = np.asarray(tick, dtype=np.float64)
    rec[:, 28:32] = theta
    rec[:, 32:36] = bodyangle_state
    rec[:, 36:36 + 2 * nh] = x_warm
    rec[:, 36 + 2 * nh:36 + 11 * nh] = np.asarray(refs).reshape(B, 9 * nh)
    return rec


class FusedTick(ctypes.Structure):
    """Go1FusedTick of include/go1mpc.h (device pointers)."""
    _fields_ = [("n_sqp", ctypes.c_int), ("tick_d", ctypes.c_void_p), ("step_state_d", ctypes.c_void_p),
                ("step_in_d", ctypes.c_void_p), ("out38_d", ctypes.c_void_p), ("step_diag_d", ctypes.c_void_p),
                ("foot_d", ctypes.c_void_p), ("out18_d", ctypes.c_void_p), ("right_support_d", ctypes.c_void_p),
                ("nh", ctypes.c_int), ("body_in_d", ctypes.c_void_p), ("body_out_d", ctypes.c_void_p),
                ("body_diag_d", ctypes.c_void_p), ("gait_mode", ctypes.c_int), ("y_offset", ctypes.c_double),
                ("homing_d", ctypes.c_void_p), ("q_d", ctypes.c_void_p), ("jac_d", ctypes.c_void_p),
                ("foot_des_d", ctypes.c_void_p), ("ik_iters_d", ctypes.c_void_p), ("servo_theta_d", ctypes.c_void_p),
                ("grf_in_d", ctypes.c_void_p), ("grf_out_d", ctypes.c_void_p), ("grf_diag_d", ctypes.c_void_p),
                ("swing_d", ctypes.c_void_p), ("p_des_d", ctypes.c_void_p), ("p_est_d", ctypes.c_void_p),
                ("pv_des_d", ctypes.c_void_p), ("pv_est_d", ctypes.c_void_p), ("tau_d", ctypes.c_void_p)]


COMPACT_DOUBLES = 12   # GO1MPC_COMPACT_DOUBLES


class ControlTick(ctypes.Structure):
    """Go1ControlTick of include/go1mpc.h."""
    _fields_ = [("n_sqp", ctypes.c_int), ("nh", ctypes.c_int), ("tick", ctypes.c_void_p), ("step_in", ctypes.c_void_p),
                ("body_tick_in", ctypes.c_void_p), ("step_state_src_d", ctypes.c_void_p), ("step_state_d", ctypes.c_void_p),
                ("tx_d", ctypes.c_void_p), ("body_out_d", ctypes.c_void_p), ("compact_d", ctypes.c_void_p),
                ("compact", ctypes.c_void_p), ("out38", ctypes.c_void_p), ("step_diag", ctypes.c_void_p),
                ("body_diag", ctypes.c_void_p), ("step_in_rows", ctypes.c_int)]


STACK_SENSOR_ROWS = 11   # GO1MPC_STACK_SENSOR_ROWS: /control2rtmpc/state slots 0 | 10 11 13 14 | 19 20 21 | 22 23 24
STACK_SLOTS_MAX = 64     # GO1MPC_STACK_SLOTS_MAX
# GO1MPC_STACK_ROW_*: first row of each block of the gait stack state
STACK_ROW_NLP, STACK_ROW_GAIT, STACK_ROW_RT2NRT, STACK_ROW_WALKDTIME, STACK_ROW_TRAJ, STACK_ROW_RT = 0, 480, 580, 605, 606, 706


class GaitStackTick(ctypes.Structure):
    """Go1GaitStackTick of include/go1mpc.h."""
    _fields_ = [("nh", ctypes.c_int), ("planner", ctypes.c_int), ("sensor", ctypes.c_void_p), ("cmd", ctypes.c_void_p),
                ("start", ctypes.c_void_p), ("state_d", ctypes.c_void_p), ("body_out_d", ctypes.c_void_p),
                ("n_slots", ctypes.c_int), ("slots", ctypes.c_int * STACK_SLOTS_MAX), ("rows_d", ctypes.c_void_p),
                ("rows", ctypes.c_void_p), ("sensor_d", ctypes.c_void_p), ("cmd_d", ctypes.c_void_p), ("start_d", ctypes.c_void_p)]


class GaitStackClockedTick(ctypes.Structure):
    """Go1GaitStackClockedTick of include/go1mpc.h."""
    _fields_ = [("nh", ctypes.c_int), ("sensor", ctypes.c_void_p), ("cmd", ctypes.c_void_p), ("start", ctypes.c_void_p),
                ("state_d", ctypes.c_void_p), ("body_out_d", ctypes.c_void_p), ("n_slots", ctypes.c_int),
                ("slots", ctypes.c_int * STACK_SLOTS_MAX), ("rows_d", ctypes.c_void_p), ("rows", ctypes.c_void_p),
                ("clock_d", ctypes.c_void_p), ("sensor_d", ctypes.c_void_p), ("cmd_d", ctypes.c_void_p), ("start_d", ctypes.c_void_p)]


class GaitStackReset(ctypes.Structure):
    """Go1GaitStackReset of include/go1mpc.h."""
    _fields_ = [("nh", ctypes.c_int), ("reset", ctypes.c_void_p), ("clock_d", ctypes.c_void_p), ("state_d", ctypes.c_void_p),
                ("body_out_d", ctypes.c_void_p), ("servo_state_d", ctypes.c_void_p), ("servo_q0", ctypes.c_double * 12),
                ("reset_d", ctypes.c_void_p)]


SERVO_TICKS_MAX = 10      # GO1MPC_SERVO_TICKS_MAX
SERVO_STATE_ROWS = 69     # GO1MPC_SERVO_STATE_ROWS
# GO1MPC_SERVO_ROW_*: joint angles [0,12) | homing foot positions [12,24) | the 9 filters' state [5][9] from row 24
SERVO_ROW_Q, SERVO_ROW_HOMING, SERVO_ROW_LPF = 0, 12, 24
SERVO_LPF_SLOTS = [0, 1, 2, 6, 7, 8, 9, 10, 11]   # /MPC/Gait slot of filter channel 0..8: CoM | left foot | right foot


class ServoStackTick(ctypes.Structure):
    """Go1ServoStackTick of include/go1mpc.h."""
    _fields_ = [("K", ctypes.c_int), ("gait_mode", ctypes.c_int), ("y_offset", ctypes.c_double),
                ("stack_state_d", ctypes.c_void_p), ("servo_state_d", ctypes.c_void_p), ("q_d", ctypes.c_void_p),
                ("q", ctypes.c_void_p), ("jac_d", ctypes.c_void_p), ("foot_des_d", ctypes.c_void_p), ("iters_d", ctypes.c_void_p)]


SERVO_FORCE_ROWS = 24     # GO1MPC_SERVO_FORCE_ROWS: previous grf_opt [0,12) | F_leg_ref [12,24)


class ServoTorqueTick(ctypes.Structure):
    """Go1ServoTorqueTick of include/go1mpc.h."""
    _fields_ = ServoStackTick._fields_ + [
        ("y_coefficient", ctypes.c_double), ("force_state_d", ctypes.c_void_p), ("meas_d", ctypes.c_void_p),
        ("reset", ctypes.c_void_p), ("tau_d", ctypes.c_void_p), ("tau", ctypes.c_void_p), ("grf_d", ctypes.c_void_p),
        ("grf_diag_d", ctypes.c_void_p), ("reset_d", ctypes.c_void_p)]


# GO1MPC_HEALTH_*: rows of a farm's health counters, int32 [HEALTH_ROWS][B] (see include/go1mpc.h)
HEALTH_ROWS = 12
(HEALTH_PLAN_OK, HEALTH_PLAN_INFEASIBLE, HEALTH_PLAN_FAILED, HEALTH_BODY_OK, HEALTH_BODY_INFEASIBLE, HEALTH_BODY_FAILED,
 HEALTH_GRF_OK, HEALTH_GRF_FAILED, HEALTH_GRF_FALLBACK, HEALTH_IK_CAP, HEALTH_NONFINITE, HEALTH_EVENTS) = range(HEALTH_ROWS)


class FarmColumns(ctypes.Structure):
    """Go1FarmColumns of include/go1mpc.h: one farm-shaped buffer set (device)."""
    _fields_ = [("B", ctypes.c_int), ("state_d", ctypes.c_void_p), ("body_out_d", ctypes.c_void_p), ("clock_d", ctypes.c_void_p),
                ("servo_state_d", ctypes.c_void_p), ("force_state_d", ctypes.c_void_p), ("health_d", ctypes.c_void_p)]


class FarmCopy(ctypes.Structure):
    """Go1FarmCopy of include/go1mpc.h."""
    _fields_ = [("nh", ctypes.c_int), ("dst", FarmColumns), ("src", FarmColumns), ("index_d", ctypes.c_void_p),
                ("bad_d", ctypes.c_void_p)]


def _ptr(a):
    """Raw address of a numpy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise Go1MpcError("array must be C-contiguous")
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        if not a.is_contiguous():
            raise Go1MpcError("tensor must be contiguous")
        return a.data_ptr()
    raise Go1MpcError(f"cannot take the address of {type(a)}")


class Go1Mpc:
    """Handle wrapper: one per host thread / GPU."""

    def __init__(self, device=-1, cfg=None):
        self.lib = load_library()
        self.cfg = Cfg()
        self.lib.go1mpc_config_default(ctypes.byref(self.cfg))
        if cfg:
            for k, v in cfg.items():
                if k == "lamda":
                    for i in range(4):
                        self.cfg.body.lamda[i] = v[i]
                elif k == "qp_iter_cap_scale":
                    self.cfg.qp_iter_cap_scale = v
                elif k == "step":
                    for sk, sv in v.items():
                        if sk == "lamda":
                            for i in range(4):
                                self.cfg.step.lamda[i] = sv[i]
                        else:
                            setattr(self.cfg.step, sk, sv)
                else:
                    setattr(self.cfg.body, k, v)
        self.h = ctypes.c_void_p()
        rc = self.lib.go1mpc_create(ctypes.byref(self.cfg), device, ctypes.byref(self.h))
        if rc != 0:
            raise Go1MpcError(f"go1mpc_create failed with {rc} (no usable CUDA device? there is no CPU fallback)")

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.go1mpc_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise Go1MpcError(f"{what} failed ({rc}): {self.lib.go1mpc_last_error(self.h).decode()}")

    @property
    def launch_count(self):
        return int(self.lib.go1mpc_launch_count(self.h))

    @property
    def stream(self):
        """Raw cudaStream_t of the handle (int), usable with torch.cuda.ExternalStream."""
        return int(self.lib.go1mpc_stream(self.h) or 0)

    @property
    def sm_count(self):
        return int(self.lib.go1mpc_sm_count(self.h))

    def synchronize(self):
        self._check(self.lib.go1mpc_synchronize(self.h), "synchronize")

    # --- body-inclination MPC ---
    def body_mpc_step(self, nh, B, in_d, out_d, diag_d=None, stream=None):
        """Device-pointer entry (torch CUDA tensors or raw addresses)."""
        self._check(self.lib.go1mpc_body_mpc_step_batch(self.h, nh, B, _ptr(in_d), _ptr(out_d), _ptr(diag_d), stream),
                    "body_mpc_step_batch")

    def body_mpc_step_host(self, nh, B, in_h, out_h, diag_h=None):
        """Host-buffer entry: H2D, launch, D2H and a stream sync inside the call."""
        self._check(self.lib.go1mpc_body_mpc_step_batch_host(self.h, nh, B, _ptr(in_h), _ptr(out_h), _ptr(diag_h)),
                    "body_mpc_step_batch_host")

    def body_handover_total(self):
        """Instances the roll/pitch-split kernel handed to the combined-solve kernel so far (synchronises)."""
        t = ctypes.c_longlong(0)
        self._check(self.lib.go1mpc_body_handover_total(self.h, ctypes.byref(t)), "body_handover_total")
        return int(t.value)

    def body_guard_trips(self):
        t = ctypes.c_longlong(0)
        self._check(self.lib.go1mpc_body_guard_trips(self.h, ctypes.byref(t)), "body_guard_trips")
        return int(t.value)

    def body_mpc_step_host_async(self, nh, B, in_h, out_h, diag_h=None):
        """Pipelined: returns after enqueueing H2D + kernel + D2H; call synchronize() before reading out_h."""
        self._check(self.lib.go1mpc_body_mpc_step_batch_host_async(self.h, nh, B, _ptr(in_h), _ptr(out_h), _ptr(diag_h)),
                    "body_mpc_step_batch_host_async")

    def body_mpc_step_resident_host_async(self, nh, B, tx_d, out_d, tick_in_h, tick_out_h, diag_h=None):
        """Pipelined, tx [B][28] and the output records [B][out_stride] resident on the device; only the
        per-tick record (body_tick_in_stride doubles) goes up and BODY_TICK_OUT doubles (+ diag) come down."""
        self._check(self.lib.go1mpc_body_mpc_step_batch_resident_host_async(self.h, nh, B, _ptr(tx_d), _ptr(out_d), _ptr(tick_in_h),
                                                                            _ptr(tick_out_h), _ptr(diag_h)),
                    "body_mpc_step_batch_resident_host_async")

    def step_timing_step_host_async(self, n_sqp, B, tick_h, state_d, in_h, out_h, diag_h=None, state_out_d=None):
        """Pipelined; the planner state stays on the device (state_d: device buffer, updated in place
        unless state_out_d is given)."""
        so = state_d if state_out_d is None else state_out_d
        self._check(self.lib.go1mpc_step_timing_step_batch_host_async(self.h, n_sqp, B, _ptr(tick_h), _ptr(state_d), _ptr(so),
                                                                      _ptr(in_h), _ptr(out_h), _ptr(diag_h)),
                    "step_timing_step_batch_host_async")

    def body_model(self, nh):
        out = {k: np.zeros((2, nh) if k in ("pps", "pvs") else (nh, nh)) for k in ("pps", "pvs", "ppu", "pvu", "ppu_2", "pvu_2")}
        self._check(self.lib.go1mpc_body_model(self.h, nh, *[_ptr(out[k]) for k in ("pps", "pvs", "ppu", "pvu", "ppu_2", "pvu_2")]),
                    "body_model")
        return {k: v.T.copy() for k, v in out.items()}   # column-major -> [row, col]

    def body_default_tx(self):
        tx = np.zeros(27)
        self._check(self.lib.go1mpc_body_default_tx(self.h, _ptr(tx)), "body_default_tx")
        return tx

    # --- generic dense QP ---
    def qp_solve(self, n, p, m, B, G, g0, CE, ce0, CI, ci0, x, cost=None, active=None, nactive=None, iters=None,
                 status=None, stream=None):
        self._check(self.lib.go1mpc_qp_solve_batch(self.h, n, p, m, B, _ptr(G), _ptr(g0), _ptr(CE), _ptr(ce0), _ptr(CI),
                                                   _ptr(ci0), _ptr(x), _ptr(cost), _ptr(active), _ptr(nactive),
                                                   _ptr(iters), _ptr(status), stream), "qp_solve_batch")

    def qp_solve_host(self, n, p, m, B, G, g0, CE, ce0, CI, ci0, x, cost=None, active=None, nactive=None, iters=None,
                      status=None):
        self._check(self.lib.go1mpc_qp_solve_batch_host(self.h, n, p, m, B, _ptr(G), _ptr(g0), _ptr(CE), _ptr(ce0),
                                                        _ptr(CI), _ptr(ci0), _ptr(x), _ptr(cost), _ptr(active),
                                                        _ptr(nactive), _ptr(iters), _ptr(status)), "qp_solve_batch_host")

    # --- step-location / step-timing SQP (SoA buffers: [field][B]) ---
    def step_timing_step(self, n_sqp, B, tick_d, state_d, in_d, out_d, diag_d=None, stream=None, state_out_d=None):
        """state_out_d=None updates state_d in place."""
        so = state_d if state_out_d is None else state_out_d
        self._check(self.lib.go1mpc_step_timing_step_batch(self.h, n_sqp, B, _ptr(tick_d), _ptr(state_d), _ptr(so), _ptr(in_d),
                                                           _ptr(out_d), _ptr(diag_d), stream), "step_timing_step_batch")

    def step_timing_step_host(self, n_sqp, B, tick, state, inp, out, diag=None):
        self._check(self.lib.go1mpc_step_timing_step_batch_host(self.h, n_sqp, B, _ptr(tick), _ptr(state), _ptr(inp),
                                                                _ptr(out), _ptr(diag)), "step_timing_step_batch_host")

    def step_default_state(self, steplength=0.075, stepwidth=0.2535, stepheight=0.0, tstep=0.7):
        s = np.zeros(STEP_STATE)
        self._check(self.lib.go1mpc_step_default_state(self.h, steplength, stepwidth, stepheight, tstep, _ptr(s)),
                    "step_default_state")
        return s

    # --- swing-foot trajectory of the step planner (SoA) ---
    def foot_trajectory(self, B, tick_d, state_d, out38_d, foot_d, out18_d, right_support_d=None, stream=None):
        self._check(self.lib.go1mpc_foot_trajectory_batch(self.h, B, _ptr(tick_d), _ptr(state_d), _ptr(out38_d), _ptr(foot_d),
                                                          _ptr(out18_d), _ptr(right_support_d), stream), "foot_trajectory_batch")

    def foot_trajectory_host(self, B, tick, state, out38, foot, out18, right_support=None):
        self._check(self.lib.go1mpc_foot_trajectory_batch_host(self.h, B, _ptr(tick), _ptr(state), _ptr(out38), _ptr(foot),
                                                               _ptr(out18), _ptr(right_support)), "foot_trajectory_batch_host")

    def foot_default_state(self):
        f = np.zeros(32)
        self._check(self.lib.go1mpc_foot_default_state(self.h, _ptr(f)), "foot_default_state")
        return f

    # --- leg kinematics (SoA buffers: [3][B], [9][B]) ---
    def leg_fk(self, B, q, leg, body_p, body_r, pos, jac=None, stream=None):
        self._check(self.lib.go1mpc_leg_fk_batch(self.h, B, _ptr(q), _ptr(leg), _ptr(body_p), _ptr(body_r), _ptr(pos),
                                                 _ptr(jac), stream), "leg_fk_batch")

    def leg_ik(self, B, pdes, qini, leg, body_p, body_r, q, jac=None, iters=None, stream=None):
        self._check(self.lib.go1mpc_leg_ik_batch(self.h, B, _ptr(pdes), _ptr(qini), _ptr(leg), _ptr(body_p), _ptr(body_r),
                                                 _ptr(q), _ptr(jac), _ptr(iters), stream), "leg_ik_batch")

    def servo_kin_tick(self, B, gait_mode, y_offset, com, theta, rfoot, lfoot, homing, q, jac=None, foot_des=None, iters=None,
                       stream=None):
        """Device buffers (SoA).  q [12][B] is updated in place."""
        self._check(self.lib.go1mpc_servo_kin_tick_batch(self.h, B, gait_mode, y_offset, _ptr(com), _ptr(theta), _ptr(rfoot),
                                                         _ptr(lfoot), _ptr(homing), _ptr(q), _ptr(jac), _ptr(foot_des),
                                                         _ptr(iters), stream), "servo_kin_tick_batch")

    def fused_tick(self, B, n_sqp, tick, step_state, step_in, out38, foot, out18, nh, body_in, body_out, gait_mode, y_offset,
                   homing, q, servo_theta, step_diag=None, right_support=None, body_diag=None, jac=None, foot_des=None,
                   ik_iters=None, stream=None, grf_in=None, grf_out=None, grf_diag=None, swing=None, p_des=None, p_est=None,
                   pv_des=None, pv_est=None, tau=None):
        """go1mpc_fused_tick_batch: planner tick -> swing foot -> body MPC -> servo IK (-> GRF QP -> joint torques when
        grf_in / tau are given) in one call (device buffers)."""
        def a(x):
            v = _ptr(x)
            return v if isinstance(v, int) or v is None else ctypes.cast(v, ctypes.c_void_p).value
        t = FusedTick(n_sqp, a(tick), a(step_state), a(step_in), a(out38), a(step_diag), a(foot), a(out18), a(right_support),
                      nh, a(body_in), a(body_out), a(body_diag), gait_mode, y_offset, a(homing), a(q), a(jac), a(foot_des),
                      a(ik_iters), a(servo_theta), a(grf_in), a(grf_out), a(grf_diag), a(swing), a(p_des), a(p_est), a(pv_des),
                      a(pv_est), a(tau))
        self._check(self.lib.go1mpc_fused_tick_batch(self.h, B, ctypes.byref(t), stream), "fused_tick_batch")

    def grf_force_opt(self, B, in_d, out_d, diag_d=None, stream=None):
        """Device records: in [B,48], out [B,16], diag [B,32] ints."""
        self._check(self.lib.go1mpc_grf_force_opt_batch(self.h, B, _ptr(in_d), _ptr(out_d), _ptr(diag_d), stream), "grf_force_opt_batch")

    def grf_joint_torques(self, B, jac, swing, p_des, p_est, pv_des, pv_est, F_leg_ref, tau, F_strides=None, stream=None):
        """Dynamiccclass::compute_joint_torques for the four legs; F_strides = (element, robot) strides of F_leg_ref in
        doubles, default SoA (B, 1); (1, 16) reads the out records of grf_force_opt."""
        ks, bs = F_strides if F_strides is not None else (B, 1)
        self._check(self.lib.go1mpc_grf_joint_torques_batch(self.h, B, _ptr(jac), _ptr(swing), _ptr(p_des), _ptr(p_est), _ptr(pv_des),
                                                            _ptr(pv_est), _ptr(F_leg_ref), ks, bs, _ptr(tau), stream),
                    "grf_joint_torques_batch")

    def ref_interp(self, B, nh, walktime, dt_sample, samples, out, stream=None):
        """PRMPCClass::XGetSolution_position_mod3 for B items: walktime [B] ints, samples [12,B], out [9+3(nh-1),B] (device)."""
        self._check(self.lib.go1mpc_ref_interp_batch(self.h, B, nh, _ptr(walktime), dt_sample, _ptr(samples), _ptr(out), stream),
                    "ref_interp_batch")

    def grf_force_distribution(self, B, gait_mode, y_coefficient, com, leg, F, rfoot, lfoot, F_leg_ref, stream=None):
        self._check(self.lib.go1mpc_grf_force_distribution_batch(self.h, B, gait_mode, y_coefficient, _ptr(com), _ptr(leg), _ptr(F),
                                                                 _ptr(rfoot), _ptr(lfoot), _ptr(F_leg_ref), stream),
                    "grf_force_distribution_batch")

    def leg_fk_host(self, B, q, leg, body_p, body_r, pos, jac=None):
        self._check(self.lib.go1mpc_leg_fk_batch_host(self.h, B, _ptr(q), _ptr(leg), _ptr(body_p), _ptr(body_r), _ptr(pos),
                                                      _ptr(jac)), "leg_fk_batch_host")

    def leg_ik_host(self, B, pdes, qini, leg, body_p, body_r, q, jac=None, iters=None):
        self._check(self.lib.go1mpc_leg_ik_batch_host(self.h, B, _ptr(pdes), _ptr(qini), _ptr(leg), _ptr(body_p),
                                                      _ptr(body_r), _ptr(q), _ptr(jac), _ptr(iters)), "leg_ik_batch_host")

    # --- the 100 Hz node (message in, message out) ---
    def rt_node_state_doubles(self, nh):
        return int(self.lib.go1mpc_rt_node_state_doubles(nh))

    def rt_node_default_state(self, nh):
        s = np.zeros(self.rt_node_state_doubles(nh))
        self._check(self.lib.go1mpc_rt_node_default_state(self.h, nh, _ptr(s)), "rt_node_default_state")
        return s

    def rt_node_tick(self, nh, B, state_d, msg_d, body_in_d, body_out_d, out100_d, ctrl_d=None, bodyangle_state_d=None,
                     body_diag_d=None, active_d=None, stream=None):
        self._check(self.lib.go1mpc_rt_node_tick_batch(self.h, nh, B, _ptr(state_d), _ptr(msg_d), _ptr(ctrl_d), _ptr(bodyangle_state_d),
                                                       _ptr(body_in_d), _ptr(body_out_d), _ptr(body_diag_d), _ptr(out100_d),
                                                       _ptr(active_d), stream), "rt_node_tick_batch")

    def body_phase_timing(self, enable):
        self._check(self.lib.go1mpc_body_phase_timing(self.h, 1 if enable else 0), "body_phase_timing")

    def body_phase_ms(self):
        ms = (ctypes.c_float * 3)()
        self._check(self.lib.go1mpc_body_phase_ms(self.h, ms), "body_phase_ms")
        return [float(v) for v in ms]

    def forget_buffer(self, buf_d):
        self._check(self.lib.go1mpc_forget_buffer(self.h, _ptr(buf_d)), "forget_buffer")

    # --- signal filters of the servo loop ---
    def lpf_batch(self, B, C, coef, in_d, state_d, out_d, in_rows_d=None, stream=None):
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        self._check(self.lib.go1mpc_lpf_batch(self.h, B, C, _ptr(coef), _ptr(in_d), _ptr(in_rows_d), _ptr(state_d), _ptr(out_d), stream), "lpf_batch")

    def force_filter_batch(self, B, C, in_d, state_d, out_d, stream=None):
        self._check(self.lib.go1mpc_force_filter_batch(self.h, B, C, _ptr(in_d), _ptr(state_d), _ptr(out_d), stream), "force_filter_batch")

    # --- the 40 Hz planner node (message out) ---
    def nlp_node_state_doubles(self):
        return int(self.lib.go1mpc_nlp_node_state_doubles())

    def nlp_node_default_state(self):
        s = np.zeros(self.nlp_node_state_doubles())
        self._check(self.lib.go1mpc_nlp_node_default_state(self.h, _ptr(s)), "nlp_node_default_state")
        return s

    def nlp_walkdtime_max(self):
        return int(self.lib.go1mpc_nlp_walkdtime_max(self.h))

    def nlp_node_tick(self, B, state_d, walkdtime_d, msg_d, start_d=None, cmd_d=None, rfoot_fb_d=None, lfoot_fb_d=None, stream=None):
        self._check(self.lib.go1mpc_nlp_node_tick_batch(self.h, B, _ptr(state_d), _ptr(walkdtime_d), _ptr(start_d), _ptr(cmd_d),
                                                        _ptr(rfoot_fb_d), _ptr(lfoot_fb_d), _ptr(msg_d), stream), "nlp_node_tick_batch")

    def rt_node_tick_msgs(self, nh, B, state_d, gait_msg_d, ctl_msg_d, body_in_d, body_out_d, traj_msg_d, rt2nrt_msg_d=None,
                          body_diag_d=None, stream=None):
        self._check(self.lib.go1mpc_rt_node_tick_msgs_batch(self.h, nh, B, _ptr(state_d), _ptr(gait_msg_d), _ptr(ctl_msg_d), _ptr(body_in_d),
                                                            _ptr(body_out_d), _ptr(body_diag_d), _ptr(traj_msg_d), _ptr(rt2nrt_msg_d),
                                                            stream), "rt_node_tick_msgs_batch")

    # --- gait stack tick: both nodes behind one host call ---
    def gait_stack_state_doubles(self, nh):
        return int(self.lib.go1mpc_gait_stack_state_doubles(nh))

    def gait_stack_default_state(self, nh):
        s = np.zeros(self.gait_stack_state_doubles(nh))
        self._check(self.lib.go1mpc_gait_stack_default_state(self.h, nh, _ptr(s)), "gait_stack_default_state")
        return s

    def gait_stack_tick_struct(self, nh, planner, sensor, state_d, body_out_d, slots, rows_d, rows=None, cmd=None, start=None,
                               sensor_d=None, cmd_d=None, start_d=None):
        """Go1GaitStackTick for the given buffers (host: sensor [11][B], cmd / start [B] int32, rows [B][len(slots)]).  sensor_d /
        cmd_d / start_d: the same inputs as device buffers, read in place (sensor = None with sensor_d)."""
        t = GaitStackTick(nh, 1 if planner else 0, _ptr(sensor), _ptr(cmd), _ptr(start), _ptr(state_d), _ptr(body_out_d), len(slots))
        for k, v in enumerate(slots[:STACK_SLOTS_MAX]):
            t.slots[k] = int(v)
        t.rows_d = _ptr(rows_d)
        t.rows = _ptr(rows)
        t.sensor_d, t.cmd_d, t.start_d = _ptr(sensor_d), _ptr(cmd_d), _ptr(start_d)
        return t

    def gait_stack_tick_host_async(self, B, t, stream=None):
        """go1mpc_gait_stack_tick_host_async with a GaitStackTick (gait_stack_tick_struct); returns after enqueueing on `stream`
        (None = the handle's)."""
        self._check(self.lib.go1mpc_gait_stack_tick_host_async(self.h, B, ctypes.byref(t), stream), "gait_stack_tick_host_async")

    def gait_stack_tick_clocked_struct(self, nh, sensor, clock_d, state_d, body_out_d, slots, rows_d, rows=None, cmd=None, start=None,
                                       sensor_d=None, cmd_d=None, start_d=None):
        """Go1GaitStackClockedTick for the given buffers (device clock_d [B] int32: periods since each robot's reset); sensor_d /
        cmd_d / start_d as gait_stack_tick_struct."""
        t = GaitStackClockedTick(nh, _ptr(sensor), _ptr(cmd), _ptr(start), _ptr(state_d), _ptr(body_out_d), len(slots))
        for k, v in enumerate(slots[:STACK_SLOTS_MAX]):
            t.slots[k] = int(v)
        t.rows_d = _ptr(rows_d)
        t.rows = _ptr(rows)
        t.clock_d = _ptr(clock_d)
        t.sensor_d, t.cmd_d, t.start_d = _ptr(sensor_d), _ptr(cmd_d), _ptr(start_d)
        return t

    def gait_stack_tick_clocked_async(self, B, t, stream=None, health_d=None):
        """go1mpc_gait_stack_tick_clocked_async with a GaitStackClockedTick: each robot plans on its own clock; returns after
        enqueueing on `stream` (None = the handle's).  health_d (device int32 [HEALTH_ROWS][B]) calls
        go1mpc_gait_stack_tick_clocked_health_async instead, which also updates the farm's health counters."""
        if health_d is None:
            self._check(self.lib.go1mpc_gait_stack_tick_clocked_async(self.h, B, ctypes.byref(t), stream), "gait_stack_tick_clocked_async")
        else:
            self._check(self.lib.go1mpc_gait_stack_tick_clocked_health_async(self.h, B, ctypes.byref(t), _ptr(health_d), stream),
                        "gait_stack_tick_clocked_health_async")

    def gait_stack_reset_struct(self, nh, reset, clock_d, state_d, body_out_d, servo_state_d=None, servo_q0=None, reset_d=None):
        """Go1GaitStackReset for the given buffers (host reset [B] int32, pinned for graph capture, or reset = None and device
        reset_d [B] int32; servo_q0: 12 joint angles)."""
        r = GaitStackReset(nh, _ptr(reset), _ptr(clock_d), _ptr(state_d), _ptr(body_out_d), _ptr(servo_state_d))
        r.reset_d = _ptr(reset_d)
        if servo_q0 is not None:
            q0 = np.asarray(servo_q0, dtype=np.float64).reshape(12)
            for k in range(12):
                r.servo_q0[k] = float(q0[k])
        return r

    def gait_stack_reset_async(self, B, r, stream=None):
        """go1mpc_gait_stack_reset_async with a GaitStackReset: the flagged robots restart from the default state on the device."""
        self._check(self.lib.go1mpc_gait_stack_reset_async(self.h, B, ctypes.byref(r), stream), "gait_stack_reset_async")

    # --- servo stack tick: K 1 kHz servo ticks from the gait stack's resident messages ---
    def servo_stack_tick_struct(self, K, gait_mode, y_offset, stack_state_d, servo_state_d, q_d, q=None, jac_d=None, foot_des_d=None,
                                iters_d=None):
        """Go1ServoStackTick for the given buffers (device: stack state, servo state [69][B], q_d [B][12 K]; host q or None)."""
        return ServoStackTick(int(K), int(gait_mode), float(y_offset), _ptr(stack_state_d), _ptr(servo_state_d), _ptr(q_d), _ptr(q),
                              _ptr(jac_d), _ptr(foot_des_d), _ptr(iters_d))

    def servo_stack_tick(self, B, K, gait_mode, y_offset, stack_state_d, servo_state_d, q_d, q=None, jac_d=None, foot_des_d=None,
                         iters_d=None, stream=None):
        """go1mpc_servo_stack_tick_async: K consecutive 1 kHz servo ticks (filters + leg IK) on the gait stack state; joint
        targets into q_d [B][12 K] (and the host q when given).  Returns after enqueueing on `stream` (None = the handle's)."""
        t = self.servo_stack_tick_struct(K, gait_mode, y_offset, stack_state_d, servo_state_d, q_d, q, jac_d, foot_des_d, iters_d)
        self._check(self.lib.go1mpc_servo_stack_tick_async(self.h, B, ctypes.byref(t), stream), "servo_stack_tick_async")

    # --- servo torque tick: the servo stack, then force distribution, force QP and torque map per tick ---
    def servo_torque_tick_struct(self, K, gait_mode, y_offset, y_coefficient, stack_state_d, servo_state_d, force_state_d, meas_d,
                                 q_d, tau_d, q=None, tau=None, reset=None, grf_d=None, grf_diag_d=None, jac_d=None, foot_des_d=None,
                                 iters_d=None, reset_d=None):
        """Go1ServoTorqueTick for the given buffers (device: stack state, servo state [69][B], force state [24][B], meas [24][B],
        q_d / tau_d [B][12 K], reset_d [B] int32 or None; host q / tau / reset (pinned) or None)."""
        return ServoTorqueTick(int(K), int(gait_mode), float(y_offset), _ptr(stack_state_d), _ptr(servo_state_d), _ptr(q_d), _ptr(q),
                               _ptr(jac_d), _ptr(foot_des_d), _ptr(iters_d), float(y_coefficient), _ptr(force_state_d), _ptr(meas_d),
                               _ptr(reset), _ptr(tau_d), _ptr(tau), _ptr(grf_d), _ptr(grf_diag_d), _ptr(reset_d))

    def servo_torque_tick(self, B, K, gait_mode, y_offset, y_coefficient, stack_state_d, servo_state_d, force_state_d, meas_d, q_d,
                          tau_d, stream=None, health_d=None, **kw):
        """go1mpc_servo_torque_tick_async: K 1 kHz servo ticks (filters, leg IK, force distribution, force QP, joint torques) on
        the gait stack state; joint targets into q_d and torques into tau_d, both [B][12 K].  Keyword arguments: q, tau, reset,
        reset_d, grf_d, grf_diag_d, jac_d, foot_des_d, iters_d.  health_d (device int32 [HEALTH_ROWS][B]) calls
        go1mpc_servo_torque_tick_health_async instead.  Returns after enqueueing on `stream` (None = the handle's)."""
        t = self.servo_torque_tick_struct(K, gait_mode, y_offset, y_coefficient, stack_state_d, servo_state_d, force_state_d, meas_d,
                                          q_d, tau_d, **kw)
        if health_d is None:
            self._check(self.lib.go1mpc_servo_torque_tick_async(self.h, B, ctypes.byref(t), stream), "servo_torque_tick_async")
        else:
            self._check(self.lib.go1mpc_servo_torque_tick_health_async(self.h, B, ctypes.byref(t), _ptr(health_d), stream),
                        "servo_torque_tick_health_async")

    # --- farm column copy: whole robots between two farm-shaped buffer sets, picked by a device index ---
    @staticmethod
    def farm_columns(B, state_d, body_out_d, clock_d=None, servo_state_d=None, force_state_d=None, health_d=None):
        """FarmColumns for one buffer set (torch CUDA tensors or raw addresses)."""
        return FarmColumns(int(B), _ptr(state_d), _ptr(body_out_d), _ptr(clock_d), _ptr(servo_state_d), _ptr(force_state_d),
                           _ptr(health_d))

    def farm_copy(self, nh, dst, src, index_d, bad_d=None, stream=None):
        """go1mpc_farm_copy_async: destination column i of every given block <- source column index_d[i] (device int32 [dst.B];
        -1 keeps column i).  dst / src are FarmColumns (farm_columns) or dicts of its fields.  bad_d (device int32) counts the
        entries outside -1..src.B-1, whose columns are kept.  Returns after enqueueing on `stream` (None = the handle's)."""
        d = dst if isinstance(dst, FarmColumns) else self.farm_columns(**dst)
        s = src if isinstance(src, FarmColumns) else self.farm_columns(**src)
        c = FarmCopy(int(nh), d, s, _ptr(index_d), _ptr(bad_d))
        self._check(self.lib.go1mpc_farm_copy_async(self.h, ctypes.byref(c), stream), "farm_copy_async")

    def measure_dfma_peak(self, ms=200):
        g = ctypes.c_double(0.0)
        self._check(self.lib.go1mpc_measure_dfma_peak(self.h, ms, ctypes.byref(g)), "measure_dfma_peak")
        return g.value
