"""ctypes view of include/robotick.h -- the C-ABI of librobotick_b200.so.

The library is the product: hand-written CUDA for sm_100a behind plain-C entry points.
There is no Python/CPU fallback; `load()` raises when the library has not been built.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ROBOTICK_LIB") or os.path.join(_HERE, "librobotick_b200.so")  # env: tuning builds only

RK_OK = 0

# ---- enums of robotick.h -------------------------------------------------------------
RK_SENSOR_HOLD, RK_SENSOR_PLANT, RK_SENSOR_STREAM = 0, 1, 2
RK_CMD_NONE, RK_CMD_MOVE, RK_CMD_STOP = 0, 1, 2
RK_CMD_MSG_MOVE_DIR, RK_CMD_MSG_MOVE_CONT_DIR, RK_CMD_MSG_UNKNOWN = 3, 4, 5
(RK_DIR_MOVE_STOP, RK_DIR_GO_FORWARD, RK_DIR_GO_BACK, RK_DIR_GO_RIGHT, RK_DIR_GO_LEFT, RK_DIR_GO_RIGHT_FORWARD,
 RK_DIR_GO_LEFT_FORWARD, RK_DIR_GO_RIGHT_BACK, RK_DIR_GO_LEFT_BACK, RK_DIR_ROT_RIGHT, RK_DIR_ROT_LEFT) = range(11)
RK_VDT_TRACE_WORDS = 16
RK_OPT_FORCE_TRANSCRIPTION = 1
RK_OPT_FAST_OCCUPANCY = 2
RK_OPT_FAST_PACKED = 3
RK_OPT_TICK_SIDE_CTAS = 4
RK_OPT_FAST_FFSAT = 5
RK_OPT_STREAM_CTAS = 6


class VdtParams(C.Structure):
    """rk_vdt_params_t"""

    _fields_ = [
        ("wheel_radius_mm", C.c_float),
        ("wheel_l_mm", C.c_float),
        ("sqrtf2", C.c_float),
        ("ts", C.c_float),
        ("ctrl_freq", C.c_float),
        ("kff", C.c_float),
        ("kp", C.c_float),
        ("ki", C.c_float),
        ("kd", C.c_float),
        ("i_limit", C.c_float),
        ("lpf_freq", C.c_float),
        ("ff_limit", C.c_float),
        ("accel_move", C.c_float * 3),
        ("jerk_move", C.c_float * 3),
        ("accel_stop", C.c_float * 3),
        ("jerk_stop", C.c_float * 3),
        ("motor_dir", C.c_int32 * 4),
        ("raw_curr_lim", C.c_int32),
        ("default_speed_mmps", C.c_float),
        ("limit_speed_mmps", C.c_float),
        ("default_rot_radps", C.c_float),
        ("limit_rot_radps", C.c_float),
        ("task_freq_hz", C.c_uint32),
    ]


class RmtParams(C.Structure):
    """rk_rmt_params_t"""

    _fields_ = [("no_cmd_stop_thre", C.c_uint32), ("wall_leave_time_ms", C.c_uint32), ("wall_leave_speed_mmps", C.c_uint32)]


RK_ADH_MODE_INIT, RK_ADH_MODE_INIT_POS_MOVE = 1, 2
RK_ROS_NONE, RK_ROS_MECANUM_CMD, RK_ROS_MECANUM_CONT, RK_ROS_CMD_VEL, RK_ROS_COMMAND = range(5)


class VdtCmd(C.Structure):
    """rk_vdt_cmd_t"""

    _fields_ = [("vx", C.c_float), ("vy", C.c_float), ("vth", C.c_float), ("kind", C.c_int32)]


class VdtRollout(C.Structure):
    """rk_vdt_rollout_t (pointers are device pointers for the library, host for the oracle)"""

    _fields_ = [
        ("steps", C.c_int32),
        ("sensor_mode", C.c_int32),
        ("d_cmd", C.c_void_p),
        ("n_seg", C.c_int32),
        ("seg_len", C.c_int32),
        ("d_yaw", C.c_void_p),
        ("n_yaw", C.c_int32),
        ("yaw_period", C.c_int32),
        ("d_frames", C.c_void_p),
        ("d_trace", C.c_void_p),
        ("d_goal", C.c_void_p),
        ("d_cost", C.c_void_p),
        ("task_period", C.c_int32),
        ("d_yaw_reg", C.c_void_p),
        ("d_imu_regs", C.c_void_p),
        ("d_imu_have_quat", C.c_void_p),
        ("d_imu_yaw0_deg", C.c_void_p),
        ("reset_state", C.c_int32),
    ]


class AdtParams(C.Structure):
    """rk_adt_params_t"""

    _fields_ = [
        ("ctrl_time_s", C.c_float * 7),
        ("gear_ratio", C.c_float * 7),
        ("motor_dir", C.c_float * 7),
        ("curlim_default_A", C.c_float * 7),
        ("cycle_time_s", C.c_float),
        ("mechend_pos_deg", C.c_float * 7),
        ("vel_init_degps", C.c_float * 7),
        ("curlim_init_A", C.c_float * 7),
        ("initpos_deg", C.c_float * 7),
    ]


class AdtPosCmd(C.Structure):
    """rk_adt_poscmd_t == ADTModePositioningSeq::PosCmd (AD_mode_positioning_seq.hpp:15-18)"""

    _fields_ = [("dt_ms", C.c_uint32), ("tgt_deg", C.c_float * 5)]


class AdtPosCmdSeq(C.Structure):
    """rk_adt_poscmdseq_t == ADTModePositioningSeq::PosCmdSeq (:20-24), 776 bytes"""

    _fields_ = [("id", C.c_uint32), ("len", C.c_uint8), ("cmd", AdtPosCmd * 32)]


class StreamDesc(C.Structure):
    """rk_stream_desc_t"""

    _fields_ = [
        ("first", C.c_int64),
        ("seed", C.c_uint32),
        ("first_update", C.c_uint32),
        ("stop_every", C.c_uint32),
        ("drop_every", C.c_uint32),
        ("arm_min_len", C.c_uint32),
        ("arm_max_len", C.c_uint32),
        ("arm_seq_id", C.c_uint32),
        ("arm_dt_zero_every", C.c_uint32),
        ("rsv", C.c_uint32 * 2),
    ]


class TickRollout(C.Structure):
    """rk_tick_rollout_t"""

    _fields_ = [
        ("steps", C.c_int32),
        ("slow_period", C.c_int32),
        ("d_cmd", C.c_void_p),
        ("n_seg", C.c_int32),
        ("seg_len", C.c_int32),
        ("d_regs", C.c_void_p),
        ("d_have_quat", C.c_void_p),
        ("d_yaw", C.c_void_p),
        ("d_goal", C.c_void_p),
        ("d_cost", C.c_void_p),
        ("d_vdt_trace", C.c_void_p),
        ("d_adt_trace", C.c_void_p),
        ("reset_vehicle", C.c_int32),
        ("d_yaw_reg", C.c_void_p),
        ("d_imu_desc", C.c_void_p),
    ]


class PlanSample(C.Structure):
    """rk_plan_sample_t"""

    _fields_ = [("first", C.c_int64), ("seed", C.c_uint32), ("rsv", C.c_uint32), ("sigma", C.c_float * 3), ("rsv2", C.c_float)]


class PlanCost(C.Structure):
    """rk_plan_cost_t"""

    _fields_ = [("d_ref", C.c_void_p), ("w_pos", C.c_float), ("w_goal", C.c_float), ("w_cur", C.c_float), ("rsv", C.c_float)]


class PlanObstacles(C.Structure):
    """rk_plan_obstacles_t"""

    _fields_ = [("d_obs", C.c_void_p), ("m", C.c_int32), ("check_period", C.c_int32), ("w_obst", C.c_float), ("rsv", C.c_float)]


class PlanMap(C.Structure):
    """rk_plan_map_t"""

    _fields_ = [("d_cells", C.c_void_p), ("d_map_of", C.c_void_p), ("n_maps", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
                ("x0", C.c_float), ("y0", C.c_float), ("inv_res", C.c_float), ("outside", C.c_float), ("w_map", C.c_float)]


class PlanCtg(C.Structure):
    """rk_plan_ctg_t"""

    _fields_ = [("step_axial", C.c_float), ("step_diag", C.c_float), ("k_cost", C.c_float), ("lethal", C.c_float)]


class PlanField(C.Structure):
    """rk_plan_field_t"""

    _fields_ = [("d_field", C.c_void_p), ("d_field_of", C.c_void_p), ("d_offset", C.c_void_p), ("n_fields", C.c_int32), ("fw", C.c_int32),
                ("fh", C.c_int32), ("x0", C.c_float), ("y0", C.c_float), ("inv_res", C.c_float), ("outside", C.c_float), ("w_field", C.c_float)]


class PlanInflate(C.Structure):
    """rk_plan_inflate_t"""

    _fields_ = [("d_table", C.c_void_p), ("n_table", C.c_int32), ("lethal", C.c_float)]


class PlanRefit(C.Structure):
    """rk_plan_refit_t"""

    _fields_ = [("elite", C.c_int32), ("alpha", C.c_float), ("sigma_min", C.c_float * 3), ("rsv", C.c_float)]


_lib = None


class RobotickError(RuntimeError):
    pass


def _proto(lib):
    vp = C.c_void_p
    lib.rk_version.restype = C.c_int
    lib.rk_last_error.restype = C.c_char_p
    lib.rk_device_info.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]
    lib.rk_set_device.argtypes = [C.c_int]
    lib.rk_set_option.argtypes = [C.c_int, C.c_int]
    lib.rk_vdt_fast_path_proven.argtypes = [C.POINTER(VdtParams)]
    lib.rk_vdt_prepare.argtypes = [C.POINTER(VdtParams)]
    lib.rk_probe_fp32.argtypes = [C.c_int, C.c_int, C.c_int, vp, C.POINTER(C.c_double), vp]
    lib.rk_vdt_default_params.argtypes = [C.POINTER(VdtParams)]
    lib.rk_vdt_default_params.restype = None
    lib.rk_vdt_state_words.restype = C.c_size_t
    lib.rk_vdt_state_bytes.argtypes = [C.c_int64]
    lib.rk_vdt_state_bytes.restype = C.c_size_t
    lib.rk_vdt_rollout.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.POINTER(VdtRollout), vp]
    lib.rk_vdt_set_power.argtypes = [vp, C.c_int64, vp, vp]
    lib.rk_vdt_set_target_vel.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, vp, vp, vp, vp]
    lib.rk_vdt_tx_frames.argtypes = [vp, C.c_int64, vp, vp]
    lib.rk_vdt_motor_rx.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.c_int, vp, vp, vp]
    lib.rk_imt_state_words.restype = C.c_size_t
    lib.rk_imt_state_bytes.argtypes = [C.c_int64]
    lib.rk_imt_state_bytes.restype = C.c_size_t
    lib.rk_imt_update.argtypes = [vp, C.c_int64, C.c_int32, vp, vp, vp, C.c_int, vp]
    lib.rk_imt_update_yaw.argtypes = [vp, C.c_int64, C.c_int32, vp, vp, vp, vp, C.c_int, vp]
    lib.rk_imt_parser_words.restype = C.c_size_t
    lib.rk_imt_parser_bytes.argtypes = [C.c_int64]
    lib.rk_imt_parser_bytes.restype = C.c_size_t
    lib.rk_imt_feed_bytes.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_int, vp]
    lib.rk_tick_rollout.argtypes = [C.POINTER(VdtParams), C.POINTER(AdtParams), vp, vp, vp, vp, C.c_int64,
                                    C.POINTER(TickRollout), vp]
    lib.rk_stream_default_desc.argtypes = [C.POINTER(StreamDesc)]
    lib.rk_stream_default_desc.restype = None
    lib.rk_stream_vehicle_commands.argtypes = [vp, C.c_int64, C.c_int32, vp, vp]
    lib.rk_stream_vehicle_yaw_reg.argtypes = [vp, C.c_int64, C.c_int32, vp, vp]
    lib.rk_stream_imu_samples.argtypes = [vp, C.c_int64, C.c_int32, vp, vp, vp]
    lib.rk_stream_imu_samples_yaw.argtypes = [vp, C.c_int64, C.c_int32, vp, vp, vp, vp]
    lib.rk_stream_arm_sequences.argtypes = [vp, C.c_int64, vp, vp]
    lib.rk_plan_sample_commands.argtypes = [C.POINTER(VdtParams), C.POINTER(PlanSample), vp, C.c_int64, C.c_int32, C.c_int32, vp, vp]
    lib.rk_plan_rollout.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.c_int32, vp, C.c_int32, C.c_int32, C.POINTER(PlanCost), vp,
                                    vp]
    lib.rk_plan_rollout_obstacles.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.c_int32, vp, C.c_int32, C.c_int32, C.POINTER(PlanCost),
                                              C.POINTER(PlanObstacles), vp, vp]
    lib.rk_plan_rollout_moving.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.c_int32, vp, C.c_int32, C.c_int32, C.POINTER(PlanCost),
                                           C.POINTER(PlanObstacles), vp, vp, vp]
    lib.rk_plan_rollout_map.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.c_int32, vp, C.c_int32, C.c_int32, C.POINTER(PlanCost),
                                        C.POINTER(PlanObstacles), C.POINTER(PlanMap), vp, vp, vp]
    lib.rk_plan_rollout_field.argtypes = [C.POINTER(VdtParams), vp, C.c_int64, C.c_int32, vp, C.c_int32, C.c_int32, C.POINTER(PlanCost),
                                          C.POINTER(PlanObstacles), C.POINTER(PlanMap), C.POINTER(PlanField), vp, vp, vp]
    lib.rk_plan_cost_to_go.argtypes = [C.POINTER(PlanMap), C.POINTER(PlanCtg), vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp,
                                       C.POINTER(C.c_int32), vp]
    lib.rk_plan_cost_to_go_work_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.rk_plan_cost_to_go_work_bytes.restype = C.c_size_t
    lib.rk_plan_inflate.argtypes = [C.POINTER(PlanMap), C.POINTER(PlanInflate), vp, vp, vp]
    lib.rk_plan_inflate_work_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.rk_plan_inflate_work_bytes.restype = C.c_size_t
    lib.rk_plan_peer_discs.argtypes = [vp, C.c_int64, C.c_int32, vp, C.c_int32, C.c_float, vp, C.c_int32, C.c_int32, vp]
    lib.rk_plan_select.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_int32, vp, vp, vp, vp]
    lib.rk_plan_sample_commands_sigma.argtypes = [C.POINTER(VdtParams), C.POINTER(PlanSample), vp, vp, C.c_int64, C.c_int32, C.c_int32, vp,
                                                  vp]
    lib.rk_plan_refit.argtypes = [vp, vp, vp, C.c_int64, C.c_int32, C.c_int32, C.POINTER(PlanRefit), C.c_int32, vp, vp, vp, vp, vp]
    lib.rk_adt_bldc_rx.argtypes = [C.POINTER(AdtParams), vp, C.c_int64, C.c_int, vp, vp, vp, vp]
    lib.rk_adt_mg_rx.argtypes = [C.POINTER(AdtParams), vp, C.c_int64, vp, vp, vp]
    lib.rk_selftest_div_rcp64.argtypes = [C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32)]
    lib.rk_tick_debug_timeline.argtypes = [C.c_int, C.POINTER(C.c_float)]
    lib.rk_rmt_default_params.argtypes = [C.POINTER(RmtParams)]
    lib.rk_rmt_default_params.restype = None
    lib.rk_rmt_state_words.restype = C.c_size_t
    lib.rk_rmt_state_bytes.argtypes = [C.c_int64]
    lib.rk_rmt_state_bytes.restype = C.c_size_t
    lib.rk_rmt_guard.argtypes = [C.POINTER(RmtParams), vp, C.c_int64, C.c_int32, vp, vp, vp, vp]
    lib.rk_mymath_atan2f.argtypes = [vp, vp, vp, C.c_int64, vp]
    lib.rk_rmt_create.argtypes = [C.POINTER(vp), C.POINTER(RmtParams)]
    lib.rk_rmt_destroy.argtypes = [vp]
    lib.rk_rmt_destroy.restype = None
    lib.rk_rmt_cycle.argtypes = [vp, C.POINTER(C.c_uint32), C.POINTER(VdtCmd), C.POINTER(C.c_uint32)]
    lib.rk_rmt_get_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.rk_adt_rx.argtypes = [vp, C.c_int, C.c_uint32, C.POINTER(C.c_uint8), C.POINTER(C.c_float)]
    lib.rk_adt_home_init.argtypes = [vp, C.c_int]
    lib.rk_adt_home_tick.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    lib.rk_imt_create.argtypes = [C.POINTER(vp)]
    lib.rk_imt_destroy.argtypes = [vp]
    lib.rk_imt_destroy.restype = None
    lib.rk_imt_init.argtypes = [vp, C.POINTER(C.c_int16)]
    lib.rk_imt_update1.argtypes = [vp, C.POINTER(C.c_int16), C.c_int]
    lib.rk_imt_get.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    lib.rk_imt_get_yaw.argtypes = [vp, C.POINTER(C.c_float)]
    lib.rk_imt_get_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.rk_imt_set_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.rk_adt_default_params.argtypes = [C.POINTER(AdtParams)]
    lib.rk_adt_default_params.restype = None
    for nm in ("rk_adt_state_bytes", "rk_adt_cmdtab_bytes"):
        getattr(lib, nm).argtypes = [C.c_int64]
        getattr(lib, nm).restype = C.c_size_t
    lib.rk_adt_state_words.restype = C.c_size_t
    lib.rk_adt_mode_init.argtypes = [C.POINTER(AdtParams), vp, C.c_int64, vp]
    lib.rk_adt_push_cmdseq.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
    lib.rk_adt_update.argtypes = [C.POINTER(AdtParams), vp, vp, C.c_int64, C.c_int32, vp, vp]
    lib.rk_adt_cmdseq_status.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
    lib.rk_adp_state_words.restype = C.c_size_t
    lib.rk_adp_state_bytes.argtypes = [C.c_int64]
    lib.rk_adp_state_bytes.restype = C.c_size_t
    lib.rk_adh_state_words.restype = C.c_size_t
    lib.rk_adh_state_bytes.argtypes = [C.c_int64]
    lib.rk_adh_state_bytes.restype = C.c_size_t
    lib.rk_adh_mode_init.argtypes = [vp, C.c_int64, C.c_int, vp]
    lib.rk_adh_update.argtypes = [C.POINTER(AdtParams), vp, vp, C.c_int64, C.c_int32, vp, vp, vp]
    lib.rk_adp_mode_init.argtypes = [vp, C.c_int64, vp]
    lib.rk_adp_push_cmd.argtypes = [vp, C.c_int64, vp, vp, vp]
    lib.rk_adp_update.argtypes = [C.POINTER(AdtParams), vp, vp, C.c_int64, C.c_int32, vp, vp]
    lib.rk_adp_cmd_status.argtypes = [vp, C.c_int64, vp, vp, vp]
    lib.rk_adt_create.argtypes = [C.POINTER(vp), C.POINTER(AdtParams)]
    lib.rk_adt_destroy.argtypes = [vp]
    lib.rk_adt_destroy.restype = None
    lib.rk_adt_init.argtypes = [vp]
    lib.rk_adt_push.argtypes = [vp, C.POINTER(AdtPosCmdSeq)]
    lib.rk_adt_tick.argtypes = [vp]
    lib.rk_adt_status.argtypes = [vp, C.c_uint32, C.POINTER(C.c_int32)]
    lib.rk_adt_get_targets_deg.argtypes = [vp, C.POINTER(C.c_float)]
    lib.rk_adt_get_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.rk_adt_set_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.rk_vdt_create.argtypes = [C.POINTER(vp), C.POINTER(VdtParams)]
    lib.rk_vdt_destroy.argtypes = [vp]
    lib.rk_vdt_destroy.restype = None
    for name in ("rk_vdt_update", "rk_vdt_start", "rk_vdt_stop"):
        getattr(lib, name).argtypes = [vp]
    f3 = C.POINTER(C.c_float)
    lib.rk_vdt_set_target.argtypes = [vp, f3, f3, f3]
    lib.rk_vdt_set_yaw.argtypes = [vp, C.c_float]
    lib.rk_vdt_rx.argtypes = [vp, C.c_int, C.c_char_p, C.c_int16]
    for name in ("rk_vdt_get_pos", "rk_vdt_get_vel", "rk_vdt_get_vel_tgt"):
        getattr(lib, name).argtypes = [vp, f3]
    lib.rk_vdt_get_raw_current.argtypes = [vp, C.POINTER(C.c_int16)]
    lib.rk_vdt_get_angle_sum.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.rk_vdt_get_tx_frame.argtypes = [vp, C.POINTER(C.c_uint8)]
    lib.rk_vdt_get_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.rk_vdt_set_state.argtypes = [vp, C.POINTER(C.c_uint32)]
    return lib


def load():
    """dlopen librobotick_b200.so (built by `python -m ...build` / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RobotickError(
                f"{LIB_PATH} is not built: run __graft_entry__.build() (nvcc, sm_100a). "
                "There is no CPU fallback."
            )
        _lib = _proto(C.CDLL(LIB_PATH))
    return _lib


def check(rc):
    if rc != RK_OK:
        msg = load().rk_last_error()
        raise RobotickError(f"robotick call failed rc={rc}: {msg.decode() if msg else ''}")


def default_params():
    """The firmware constants (VD_task_main.cpp:22-48,75-108,157-160); must equal
    rk_vdt_default_params() -- tests/test_cabi_cpu.py checks that."""
    p = VdtParams()
    p.wheel_radius_mm = 37.5
    p.wheel_l_mm = 13.08148
    p.sqrtf2 = 1.41421356
    p.ts = 0.001  # float(1.0f/1000.0f) == float(0.001)
    p.ctrl_freq = 100.0
    p.kff, p.kp, p.ki, p.kd = 0.0075, 0.02, 0.01, 0.0
    p.i_limit = 0.5
    p.lpf_freq = 10.0
    p.ff_limit = 1.0
    p.accel_move[:] = [1000.0, 1000.0, 30.0]
    p.jerk_move[:] = [10000.0, 10000.0, 300.0]
    p.accel_stop[:] = [2000.0, 2000.0, 70.0]
    p.jerk_stop[:] = [30000.0, 30000.0, 1000.0]
    p.motor_dir[:] = [1, 1, -1, -1]
    p.raw_curr_lim = 3000
    import math

    p.default_speed_mmps, p.limit_speed_mmps = 200.0, 400.0
    p.default_rot_radps, p.limit_rot_radps = 2.0 * math.pi, 6.0 * math.pi  # double expressions stored as float (:25,:27)
    p.task_freq_hz = 100
    return p


def default_arm_params():
    """JointBase::ConstParams of AD_task_main.cpp:38-107 in RK_AJ_* order + FL_CYCLE_TIME_S (:149);
    must equal rk_adt_default_params()."""
    f = C.c_float
    p = AdtParams()
    p.ctrl_time_s[:] = [0.01] * 7
    p.gear_ratio[:] = [1.0, 1.0, 1.0, 1.0, f(f(24.0).value / f(7.0).value).value, f(f(48.0).value / f(7.0).value).value,
                       f(f(48.0).value / f(19.0).value).value]
    p.motor_dir[:] = [-1.0, 1.0, 1.0, 1.0, 1.0, 1.0, -1.0]
    p.curlim_default_A[:] = [3.0, 0.7, 0.5, 0.5, 1.0, 1.0, 0.8]
    p.cycle_time_s = 0.01
    p.mechend_pos_deg[:] = [-45.0, 150.0, 0.0, 0.0, 0.0, 0.0, -90.0]
    p.vel_init_degps[:] = [15.0, 30.0, 10.0, 10.0, 30.0, 30.0, -60.0]
    p.curlim_init_A[:] = [1.0, 0.15, 0.5, 0.5, 1.0, 1.0, 0.5]
    p.initpos_deg[:] = [0.0, 145.0, 0.0, 0.0, -90.0, 0.0, 0.0]
    return p
