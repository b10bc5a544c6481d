/* robotick.h -- C-ABI of the B200-native batched control-tick engine.
 *
 * Drop-in boundary for the numeric control tick of Moryu-Io/Roboken-FMSKF-robot-controller
 * (SURVEY.md section 8b).  The reference has no FFI layer: its boundary is ordinary C++ member
 * functions on static objects.  Every entry point below names the reference member it
 * replaces (file:line relative to the reference tree).  Plain pointers and sizes only; no
 * torch / C++ types.  The single-instance "handle" calls are batches of one over the same
 * CUDA kernels, so there is exactly one implementation of the arithmetic and it lives on
 * the GPU (sm_100a).  There is NO CPU fallback: every call fails with RK_ERR_CUDA when no
 * device is usable.
 *
 * Threading: a handle / state block is single-owner (not thread-safe); distinct blocks are
 * independent.  All batch calls are asynchronous on the given CUDA stream (a cudaStream_t
 * passed as void*; NULL = legacy default stream).
 *
 * ---------------------------------------------------------------------------------------
 * Data layout in HBM ("SoA of 128-bit planes")
 * ---------------------------------------------------------------------------------------
 * A state block for n instances is P planes; plane p is n contiguous 16-byte cells, cell i
 * belonging to instance i:   word w of instance i lives at
 *        ((uint32_t*)block)[ ((w / 4) * n + i) * 4 + (w % 4) ]
 * so that one warp moves 32 x 16 B = 512 contiguous bytes per plane with one 128-bit
 * load/store per thread.  n is the "pitch"; blocks must be 16-byte aligned.  A block that is
 * all-zero is the firmware's power-on state (the reference relies on zero-initialised
 * globals, e.g. VD_task_main.cpp:75-108).
 */
#ifndef ROBOTICK_H_
#define ROBOTICK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RK_VERSION 100 /* 0.1.0 */

/* ---- status codes ------------------------------------------------------------------ */
enum {
  RK_OK           = 0,
  RK_ERR_ARG      = 1, /* bad pointer / size / alignment / unsupported option */
  RK_ERR_CUDA     = 2, /* CUDA runtime error or no sm_100 device              */
  RK_ERR_NOMEM    = 3,
  RK_ERR_UNSUPPORTED = 4
};

int         rk_version(void);
const char *rk_last_error(void); /* thread-local message of the last failing call */
/* device properties the bench needs for its roofline (SM count, SM clock in kHz) */
int rk_device_info(int device, int *sm_count, int *sm_clock_khz, size_t *hbm_bytes);
/* Selects the CUDA device for subsequent calls of the calling thread (the library links its
 * own static CUDA runtime; one process per GPU calls this once with LOCAL_RANK). */
int rk_set_device(int device);
/* Library options (process-wide).  RK_OPT_FORCE_TRANSCRIPTION = 1 makes RK_SENSOR_PLANT
 * rollouts use the direct transcription kernel instead of the issue-optimised one (the two
 * are bit-identical; the tests compare them). */
enum {
  RK_OPT_FORCE_TRANSCRIPTION = 1,
  RK_OPT_FAST_OCCUPANCY = 2, /* 3 or 4 (default) resident CTAs/SM: register budget of the rollout kernel */
  RK_OPT_FAST_PACKED = 3,    /* 1 (default): packed FADD2/FFMA2 tick; 0: scalar tick.  Bit-identical; tests compare. */
  RK_OPT_FAST_FFSAT = 5,     /* 1: the feed-forward clamp to +-1 as two FMUL.SAT (FMA pipe); 0 (default): as FMNMX (ALU pipe).  Bit-identical. */
  RK_OPT_STREAM_CTAS = 6,    /* rk_stream_*: at most this many CTAs per SM (0, the default: full grids).  A planner that expands
                              * the next batch's streams beside a running rollout keeps them out of its way.  Scheduling only. */
  RK_OPT_TICK_SIDE_CTAS = 4  /* rk_tick_rollout: CTAs per SM its IMU / arm kernels may occupy beside the vehicle
                              * rollout (0, the default: full grids).  Scheduling only, results do not depend on it. */
};
int rk_set_option(int option, int value);
/* 1 if the exhaustive on-device proofs that gate the issue-optimised kernel hold for these
 * parameters on the current device (csrc/rk_exact.cu), 0 if not, < 0 on error. */
struct rk_vdt_params;
int rk_vdt_fast_path_proven(const struct rk_vdt_params *p);
/* Runs those proofs now (about 12 ms, once per parameter set and device; results are cached) instead of inside the
 * first rk_vdt_rollout with these parameters.  The proofs allocate and synchronise on a private stream: call this
 * before capturing rollouts into a CUDA graph or from latency-sensitive code. */
int rk_vdt_prepare(const struct rk_vdt_params *p);
/* Roofline probe (bench.py): launches a dense FP32 kernel on `stream` -- FFMA chains when
 * fused != 0, alternating FMUL/FADD otherwise -- and reports its flop count; the caller
 * times it with CUDA events.  d_out: >= 4 bytes of device memory. */
int rk_probe_fp32(int fused, int blocks, int iters, float *d_out, double *flops, void *stream);

/* =====================================================================================
 * Vehicle (src/VehicleDrive + the src/Utility math it calls)
 * ===================================================================================== */

/* Broadcast configuration; mirrors the constants wired in VD_task_main.cpp:22-48,75-108,
 * 157-160, VD_vehicle_controller.hpp:82-86 and VD_motor_if_m2006.hpp:64,76-82. */
typedef struct rk_vdt_params {
  float   wheel_radius_mm;   /* WHEEL_RADIUS_MM  37.5f        VD_vehicle_controller.hpp:82 */
  float   wheel_l_mm;        /* WHEEL_L_MM       13.08148f    :85 */
  float   sqrtf2;            /* SQRTF2           1.41421356f  :86 */
  float   ts;                /* VelInterpConstJerk sample time 1.0f/1000  VD_task_main.cpp:95-97 */
  float   ctrl_freq;         /* FF_PI_D c_freq   100.0f (sic: task rate)  VD_task_main.cpp:86 */
  float   kff, kp, ki, kd;   /* 0.0075f 0.02f 0.01f 0.0f      :86-89 */
  float   i_limit;           /* 0.5f */
  float   lpf_freq;          /* 10.0f */
  float   ff_limit;          /* set_FF_limit(1.0f)            :157-160 */
  float   accel_move[3];     /* C_ACCEL_MAX_MOVE {1000,1000,30}      :29-33 */
  float   jerk_move[3];      /* C_JERK_MAX_MOVE  {10000,10000,300}   :34-38 */
  float   accel_stop[3];     /* C_ACCEL_MAX_STOP {2000,2000,70}      :39-43 */
  float   jerk_stop[3];      /* C_JERK_MAX_STOP  {30000,30000,1000}  :44-48 */
  int32_t motor_dir[4];      /* FL,BL,BR,FR = +1,+1,-1,-1            :75-78 */
  int32_t raw_curr_lim;      /* s16_rawCurr_lim 3000          VD_motor_if_m2006.hpp:64 */
  /* VDT::main limiters  VD_task_main.cpp:24-27 */
  float   default_speed_mmps;  /* FL_VEHICLE_DEFAULT_SPEED_MMPS      200 */
  float   limit_speed_mmps;    /* FL_VEHICLE_LIMIT_SPEED_MMPS        400 */
  float   default_rot_radps;   /* FL_VEHICLE_DEFAULT_ROT_SPEED_RADPS (float)(2.0f * M_PI / 1.0f) */
  float   limit_rot_radps;     /* FL_VEHICLE_LIMIT_ROT_SPEED_RADPS   (float)(6.0f * M_PI / 1.0f) */
  uint32_t task_freq_hz;       /* U32_VD_TASK_CTRL_FREQ_HZ 100: move-time count = time_ms * freq / 1000 + 1  :186 */
} rk_vdt_params_t;

void rk_vdt_default_params(rk_vdt_params_t *p);

/* ---- vehicle state words (per instance) -------------------------------------------- */
enum {
  /* plane 0 : VEHICLE_CTRL::now_vhcl_pos_m_, isPowerOn   (VD_vehicle_controller.hpp:73,79) */
  RK_VS_POS_X = 0, RK_VS_POS_Y, RK_VS_POS_TH, RK_VS_FLAGS,
  /* plane 1-2 : now_vhcl_vel_mmps, now_vhcl_vel_tgt_mmps  (:74-75) */
  RK_VS_VEL_X, RK_VS_VEL_Y, RK_VS_VEL_TH, RK_VS_TGT_X,
  RK_VS_TGT_Y, RK_VS_TGT_TH, RK_VS_MOVE_CNT /* VDT::U32_MOVE_TIME_CNT_ORDER  VD_task_main.cpp:115 */, RK_VS_RSV1,
  /* planes 3..11 : three VelInterpConstJerk (x, y, th), 12 words each: vel_now_/acl_now_ and
   * the ACTIVE StatusBuf page (util_vel_interp.hpp:20-21,27-39).  The inactive page is fully
   * overwritten by set_target_params() before it can be read, so it carries no state. */
  RK_VS_INTERP0 = 12,
  /* planes 12..19 : four FF_PI_D (FL,BL,BR,FR), 8 words each (util_controller.hpp:19-31,140-147) */
  RK_VS_CTRL0 = RK_VS_INTERP0 + 3 * 12,
  /* planes 20..27 : four MOTOR_IF_M2006, 8 words each (VD_motor_if_m2006.hpp:60-72)
   *                 + VEHICLE_CTRL::s64_rawAngleSumPrev + the synthetic plant's state */
  RK_VS_MOTOR0 = RK_VS_CTRL0 + 4 * 8,
  RK_VS_WORDS  = RK_VS_MOTOR0 + 4 * 8 /* = 112 words = 28 planes = 448 B / vehicle */
};
/* word offsets inside one interpolator */
enum {
  RK_VI_VEL_NOW = 0, RK_VI_ACL_NOW, RK_VI_VEL_TGT, RK_VI_ACL_MAX,
  RK_VI_JERK_P, RK_VI_JERK_M, RK_VI_DT1, RK_VI_DT2,
  RK_VI_DT3, RK_VI_VEL_INI, RK_VI_ACL_INI, RK_VI_DT
};
/* word offsets inside one wheel controller.  now_val_ == prev_val_ and now_error_ ==
 * prev_error_ hold after every update()/reset(), so each pair is one word. */
enum {
  RK_VC_PREV_VAL = 0, RK_VC_INTEG, RK_VC_LPF_Y, RK_VC_LPF_X,
  RK_VC_NOW_TGT, RK_VC_NOW_ERR, RK_VC_NOW_CTRL, RK_VC_RSV
};
/* word offsets inside one motor */
enum {
  RK_VM_SUM_LO = 0, RK_VM_SUM_HI,   /* s64_rawAngleSum */
  RK_VM_PREV_LO, RK_VM_PREV_HI,     /* VEHICLE_CTRL::s64_rawAngleSumPrev[w] */
  RK_VM_ANG_RPM,  /* head Status: s16_rawAngle | s16_rawSpeedRpm << 16 */
  RK_VM_CUR_TGT,  /* head Status: s16_rawCurr  | s16_rawCurr_tgt  << 16 */
  RK_VM_USEC,     /* head Status: s16_microsec_id (low 16) | status_head << 16 */
  RK_VM_PLANT     /* synthetic plant (not in the reference): ang | rpm << 16, motor frame */
};
#define RK_VS_FLAG_POWER_ON 1u

size_t rk_vdt_state_words(void);        /* RK_VS_WORDS */
size_t rk_vdt_state_bytes(int64_t n);   /* bytes of an n-instance block */

/* ---- rollout: K fused 1 kHz ticks of N vehicles ------------------------------------- */
enum {
  RK_SENSOR_HOLD   = 0, /* no new CAN frames: tick re-reads the last Status (as the ISR does) */
  RK_SENSOR_PLANT  = 1, /* closed loop through the synthetic integer motor plant (below)     */
  RK_SENSOR_STREAM = 2  /* one recorded 8-byte M2006 frame per wheel per tick from HBM       */
};
/* command kinds, the vocabulary of VDT::main (VD_task_main.cpp:178-322) reduced to targets */
enum {
  RK_CMD_NONE = 0, /* no message this segment                                    */
  RK_CMD_MOVE = 1, /* start(); set_target_vel(v, C_ACCEL_MAX_MOVE, C_JERK_MAX_MOVE)  :294-295 */
  RK_CMD_STOP = 2, /* start(); set_target_vel(v, C_ACCEL_MAX_STOP, C_JERK_MAX_STOP)  :271-281,305-319 */
  /* VDT::main's own message vocabulary (VD_task_main.hpp:8-60, VD_task_main.cpp:178-296): speed limiters,
   * direction table and the move-time countdown included.  kind = id | u32_time_ms << 8 (time_ms < 2^24).
   * Messages are taken at task-period boundaries only (seg_len must be a multiple of task_period). */
  RK_CMD_MSG_MOVE_DIR = 3,      /* REQ_MOVE_DIR: the vx / vy slots carry u32_cmd / u32_speed as raw uint32 */
  RK_CMD_MSG_MOVE_CONT_DIR = 4, /* REQ_MOVE_CONT_DIR: vx, vy, vth = fl_vel_x_mmps, fl_vel_y_mmps, fl_vel_th_radps */
  RK_CMD_MSG_UNKNOWN = 5        /* a MsgId the task ignores */
};
/* REQ_MOVE_DIR_CMD  VD_task_main.hpp:37-49 */
enum {
  RK_DIR_MOVE_STOP = 0, RK_DIR_GO_FORWARD, RK_DIR_GO_BACK, RK_DIR_GO_RIGHT, RK_DIR_GO_LEFT, RK_DIR_GO_RIGHT_FORWARD,
  RK_DIR_GO_LEFT_FORWARD, RK_DIR_GO_RIGHT_BACK, RK_DIR_GO_LEFT_BACK, RK_DIR_ROT_RIGHT, RK_DIR_ROT_LEFT
};
typedef struct rk_vdt_cmd { float vx, vy, vth; int32_t kind; } rk_vdt_cmd_t; /* 16 B */

/* Trace record written per tick when d_trace != NULL (tests / small N only):
 * word 0-2 pos, 3-5 vel, 6-8 vel_tgt, 9-12 s16_rawCurr_tgt (sign-extended), 13 the move-time countdown
 * (task_period > 0, else zero), 14-15 the C610 current frame CAN_CTRL::tx_routine() puts on the bus after the tick
 * (VD_can_controller.hpp:43-55: id 0x200, the four currents as big-endian s16; buf[0] in the low byte of word 14). */
#define RK_VDT_TRACE_WORDS 16

typedef struct rk_vdt_rollout {
  int32_t steps;        /* K >= 0 */
  int32_t sensor_mode;  /* RK_SENSOR_* */
  /* commands: cell [s * n + i] applied to instance i BEFORE tick s*seg_len; NULL = none */
  const rk_vdt_cmd_t *d_cmd;
  int32_t n_seg, seg_len;
  /* IMU yaw in radians (what can_tx_routine_intr() passes to set_now_yaw_world(),
   * VD_task_main.cpp:368): cell [y * n + i] applied BEFORE tick y*yaw_period; NULL = keep */
  const float *d_yaw;
  int32_t n_yaw, yaw_period;
  /* RK_SENSOR_STREAM: 8-byte frames, cell [(t * 4 + w) * n + i] for tick t, wheel w */
  const uint64_t *d_frames;
  /* optional per-tick trace: word j of tick t, instance i at [(t * 16 + j) * n + i] */
  uint32_t *d_trace;
  /* optional rollout cost: (pos.x-gx)^2 + (pos.y-gy)^2 at the end; d_goal = float2[n] */
  const float *d_goal;
  float *d_cost;
  /* > 0: VDT::main runs every task_period ticks (firmware: 10 = 1 kHz / 100 Hz, VD_task_main.cpp:21-22):
   * RK_CMD_MSG_* records are decoded and the move-time countdown (U32_MOVE_TIME_CNT_ORDER, :298-316) issues
   * the automatic stop.  0: no task loop (RK_CMD_MOVE / RK_CMD_STOP records only). */
  int32_t task_period;
  /* the same yaw stream as the sensor reports it (used when d_yaw is NULL): the WT901C's Yaw register, int16,
   * 180/32768 degrees per count, same indexing as d_yaw.  The engine forms the float the ISR would see:
   * angle[2] = reg / 32768.0f * 180.0f (IMU_IF_WT901C::updateData, imu_if_wt901c.cpp:100) -> getYawDate() ->
   * mymath::deg2rad (VD_task_main.cpp:368).  Half the bytes of d_yaw -- the rollout's largest input. */
  const int16_t *d_yaw_reg;
  /* the yaw straight from the IMU's register snapshots (used when d_yaw and d_yaw_reg are NULL): d_imu_regs is
   * the block rk_imt_update() consumes (two 128-bit cells per sample; sample y is taken before tick
   * y*yaw_period), d_imu_have_quat its have_quat flags ([n_yaw][n], NULL = all 1).  The vehicle forms what
   * IMT::get_status_now_yaw() returns after IMU update y -- the Yaw register scaled as updateData() does, held
   * over updates without a quaternion frame (imu_if_wt901c.cpp:83-89,100,160) -- so the rollout does not wait for
   * the IMU kernel.  d_imu_yaw0_deg (float[n], may be NULL = keep the vehicle's yaw word): Data.angle[2] of the
   * IMU block at launch, the value held when update 0 carries no quaternion frame.
   * d_imu_have_quat and d_imu_yaw0_deg are honoured with d_yaw_reg as well (the Yaw column of d_imu_regs in 2 bytes). */
  const int16_t *d_imu_regs;
  const uint8_t *d_imu_have_quat;
  const float *d_imu_yaw0_deg;
  /* != 0: every vehicle starts this rollout from the power-on block (all zeros: the firmware's static initialisation)
   * instead of the contents of d_state -- a planner's "reset and roll out" in one call (the block is cleared on the
   * stream in front of the kernel; the default closed-loop configuration runs an instantiation of the kernel that starts
   * from zeros in registers instead: no clear and no state load at all). */
  int32_t reset_state;
} rk_vdt_rollout_t;

/* VEHICLE_CTRL::update() x steps   (VD_vehicle_controller.cpp:6-99), fused with the callers
 * that feed it each tick: set_now_yaw_world (:57), MOTOR_IF_M2006::rx_callback
 * (VD_motor_if_m2006.cpp:32-72) and set_target_vel (:101-105). */
int rk_vdt_rollout(const rk_vdt_params_t *p, void *d_state, int64_t n,
                   const rk_vdt_rollout_t *args, void *stream);

/* Batched setters for callers that do not use the fused command table. */
/* VEHICLE_CTRL::start()/stop()  VD_vehicle_controller.hpp:54-55 ; d_on NULL = all on */
int rk_vdt_set_power(void *d_state, int64_t n, const uint8_t *d_on, void *stream);
/* VEHICLE_CTRL::set_target_vel  VD_vehicle_controller.cpp:101-105 ; v/a/j = float[3][n] */
int rk_vdt_set_target_vel(const rk_vdt_params_t *p, void *d_state, int64_t n, const float *d_v,
                          const float *d_a, const float *d_j, void *stream);
/* MOTOR_IF_M2006::rx_callback  VD_motor_if_m2006.cpp:32-72 ; frames = uint64[n] for one wheel */
int rk_vdt_motor_rx(const rk_vdt_params_t *p, void *d_state, int64_t n, int wheel,
                    const uint64_t *d_frames, const int16_t *d_usec, void *stream);

/* CAN_CTRL::tx_routine  VD_can_controller.hpp:43-55 for every vehicle: d_frames[i] = the 8-byte C610 frame (id 0x200)
 * holding the four s16_rawCurr_tgt big-endian, FL, BL, BR, FR; buf[0] in the low byte. */
int rk_vdt_tx_frames(const void *d_state, int64_t n, uint64_t *d_frames, void *stream);

/* ---- single-instance handle (drop-in for the static objects of VD_task_main.cpp:75-108) */
typedef struct rk_vdt rk_vdt_t;
int  rk_vdt_create(rk_vdt_t **out, const rk_vdt_params_t *p /* NULL = defaults */);
void rk_vdt_destroy(rk_vdt_t *h);
int  rk_vdt_update(rk_vdt_t *h);                                  /* VEHICLE_CTRL::update()  */
int  rk_vdt_start(rk_vdt_t *h);                                   /* ::start()               */
int  rk_vdt_stop(rk_vdt_t *h);                                    /* ::stop()                */
int  rk_vdt_set_target(rk_vdt_t *h, const float v[3], const float a[3], const float j[3]);
int  rk_vdt_set_yaw(rk_vdt_t *h, float yaw_rad);                  /* ::set_now_yaw_world()   */
int  rk_vdt_rx(rk_vdt_t *h, int wheel, const uint8_t frame[8], int16_t usec_id);
int  rk_vdt_get_pos(rk_vdt_t *h, float out[3]);     /* get_vehicle_pos_m_latest      :59 */
int  rk_vdt_get_vel(rk_vdt_t *h, float out[3]);     /* get_vehicle_vel_mmps_latest   :60 */
int  rk_vdt_get_vel_tgt(rk_vdt_t *h, float out[3]); /* get_vehicle_vel_tgt_mmps_latest :61 */
int  rk_vdt_get_raw_current(rk_vdt_t *h, int16_t out[4]); /* MOTOR_IF_M2006::get_rawCurr_tgt :52 */
int  rk_vdt_get_angle_sum(rk_vdt_t *h, int64_t out[4]);   /* MOTOR_IF_M2006::get_rawAngleSum :42 */
int  rk_vdt_get_tx_frame(rk_vdt_t *h, uint8_t frame[8]);  /* CAN_CTRL::tx_routine's msg.buf  VD_can_controller.hpp:43-55 */
int  rk_vdt_get_state(rk_vdt_t *h, uint32_t words[RK_VS_WORDS]);
int  rk_vdt_set_state(rk_vdt_t *h, const uint32_t words[RK_VS_WORDS]);

/* =====================================================================================
 * IMU (src/Imu): the WT901C "state-estimation update".  The firmware contains no Kalman
 * filter -- the sensor fuses on-chip; IMU_IF_WT901C::updateData() (imu_if_wt901c.cpp:91-129)
 * scales 16 int16 registers, flips the Y/Z signs, re-wraps roll and re-references the
 * quaternion against the boot-time quaternion q_init.
 * ===================================================================================== */
/* register order of one sample (the sReg[] entries updateData() reads; lib/wt901c/REG.h) */
enum {
  RK_IMT_REG_AX = 0, RK_IMT_REG_AY, RK_IMT_REG_AZ, RK_IMT_REG_GX, RK_IMT_REG_GY, RK_IMT_REG_GZ,
  RK_IMT_REG_HX, RK_IMT_REG_HY, RK_IMT_REG_HZ, RK_IMT_REG_ROLL, RK_IMT_REG_PITCH, RK_IMT_REG_YAW,
  RK_IMT_REG_Q0, RK_IMT_REG_Q1, RK_IMT_REG_Q2, RK_IMT_REG_Q3, RK_IMT_REGS
};
/* IMU state words: plane 0 q_init[4] (imu_if_wt901c.hpp:39); planes 1-4 the readable page of
 * d_buf as IMU_IF::Data {accel[3], gyro[3], mag[3], angle[3], qut[4]} in struct order
 * (imu_if_base.hpp:12-18); plane 5 flags. */
enum { RK_IS_QINIT = 0, RK_IS_DATA = 4, RK_IS_FLAGS = 20, RK_IS_WORDS = 24 };
enum { RK_IS_D_ACCEL = 0, RK_IS_D_GYRO = 3, RK_IS_D_MAG = 6, RK_IS_D_ANGLE = 9, RK_IS_D_QUT = 12 };
#define RK_IS_FLAG_ERROR 1u /* IMU_IF_WT901C::is_error */

size_t rk_imt_state_words(void);
size_t rk_imt_state_bytes(int64_t n);

/* K fused IMU_IF_WT901C::update() calls (imu_if_wt901c.cpp:83-89) for n instances.
 *  d_regs      int16, the sReg[] snapshot at the time update() runs, in two 128-bit cells per sample like every
 *              other block: register r (RK_IMT_REG_*) of sample u, instance i at ((u*2 + r/8)*n + i)*8 + r%8
 *              (16-byte aligned; for n = 1 simply 16 consecutive registers per sample)
 *  d_have_quat uint8 [K][n] or NULL (= all 1): whether a quaternion frame arrived since the
 *              last call (isComComp(), :132-143); 0 -> is_error = true, data retained
 *  d_out       optional getDataLatest() after each update, as 128-bit planes like the state:
 *              word w of sample u, instance i at ((u*4 + w/4)*n + i)*4 + w%4 (16-byte aligned)
 *  do_init     != 0: the first sample is consumed by IMU_IF_WT901C::init() (:63-77) instead:
 *              updateData() against the current q_init, then q_init latched from q0..q3 */
int rk_imt_update(void *d_state, int64_t n, int32_t K, const int16_t *d_regs, const uint8_t *d_have_quat,
                  float *d_out, int do_init, void *stream);

/* Same, plus the value the vehicle ISR reads after each update: d_yaw_rad[u * n + i] =
 * mymath::deg2rad(IMT::get_status_now_yaw())  (VD_task_main.cpp:368, imu_task_main.cpp:102-104,
 * util_mymath.hpp:16) -- the 4-byte-per-update stream rk_vdt_rollout() consumes as d_yaw. */
int rk_imt_update_yaw(void *d_state, int64_t n, int32_t K, const int16_t *d_regs, const uint8_t *d_have_quat,
                      float *d_out, float *d_yaw_rad, int do_init, void *stream);

/* ---- WIT serial wire codec (SURVEY 8f-3): the byte stream of the WT901C through the vendor parser's state
 * machine -- WitSerialDataIn (lib/wt901c/wit_c_sdk.c:132-164: 11-byte window, 0x55 header resync, byte-sum
 * check), CopeWitData (:77-130: which registers a frame type writes), the update flags of SensorDataUpdata
 * (imu_if_wt901c.cpp:24-46) -- followed by IMU_IF_WT901C::update() (isComComp :132-143 drains every byte on the
 * wire, then asks for a quaternion frame).  Parser block per IMU (3 planes): */
enum {
  RK_IP_WINDOW = 0, /* s_ucWitDataBuff[0..10] packed little-endian in words 0-2; byte 11 = s_uiWitDataCnt */
  RK_IP_FLAGS  = 3, /* bit 0: QUAT_UPDATE pending; bits 8-15: s_uiReadRegIndex (0, or q0 = 0x51 after init());
                     * bit 16 (RK_IP_FLAG_INIT_PENDING): init() is still waiting for its first quaternion frame */
  RK_IP_SREG   = 4, /* sReg[AX..Yaw], sReg[q0..q3]: 16 x int16 in RK_IMT_REG_* order, two per word */
  RK_IP_WORDS  = 12
};
#define RK_IP_FLAG_INIT_PENDING 0x10000u
size_t rk_imt_parser_words(void);
size_t rk_imt_parser_bytes(int64_t n);
/* K updates, each preceded by the serial bytes that arrived since the last one.  The wire is laid out like every
 * other block, in 128-bit cells: cell c (bytes 16c .. 16c+15 of the update, wire order from the low byte of the
 * first word up) of update u, IMU i at cell index (u*ncells + c)*n + i.  d_nbytes (NULL: every slot is full) gives
 * the number of bytes really on the wire in update u of IMU i, at [u*n + i], clamped to 16*ncells -- an idle line
 * is 0 bytes, not zeros.  do_init: the first update is IMU_IF_WT901C::init() (:63-77; WitInit empties the window,
 * WitReadReg(q0, 4) arms the read index; the firmware then spins in getDataImmediately() until a quaternion frame has
 * arrived: update slots without one are part of that wait -- nothing is published, q_init is not latched, the pending
 * state is carried in the parser block across slots and launches -- and the slot that brings one completes init().
 * (the text below describes the common case of a frame inside update 0: its bytes contain a quaternion frame -- the firmware spins until one
 * arrives).  d_out / d_yaw_rad as rk_imt_update_yaw. */
int rk_imt_feed_bytes(void *d_state, void *d_parser, int64_t n, int32_t K, int32_t ncells, const void *d_cells,
                      const uint16_t *d_nbytes, float *d_out, float *d_yaw_rad, int do_init, void *stream);

/* single-instance handle (drop-in for `static IMU_IF_WT901C imu_if`, imu_task_main.cpp:25) */
typedef struct rk_imt rk_imt_t;
int   rk_imt_create(rk_imt_t **out);
void  rk_imt_destroy(rk_imt_t *h);
int   rk_imt_init(rk_imt_t *h, const int16_t regs[RK_IMT_REGS]);                /* ::init()          */
int   rk_imt_update1(rk_imt_t *h, const int16_t regs[RK_IMT_REGS], int have_quat); /* ::update()     */
int   rk_imt_get(rk_imt_t *h, float data[16], int *is_error); /* ::getDataLatest() / ::isError()      */
int   rk_imt_get_yaw(rk_imt_t *h, float *yaw_deg);            /* ::getYawDate()  :160-162             */
int   rk_imt_get_state(rk_imt_t *h, uint32_t words[RK_IS_WORDS]);
int   rk_imt_set_state(rk_imt_t *h, const uint32_t words[RK_IS_WORDS]);

/* =====================================================================================
 * Arm (src/ArmDrive): 5-axis joint-command interpolation, ADTModePositioningSeq + the joint
 * classes it drives, one 100 Hz tick = ADT::main's loop body (AD_task_main.cpp:208-229):
 *   m_posseq.update(); j_P1.update(); j_DF_Left.update(); j_DF_Right.update(); j_P3.update();
 *   [CAN tx]; j_Y0.update();
 * Joint objects in this order everywhere: Y0 (ICS), P1 (MG), DF_Left, DF_Right (MyBldc),
 * P2 (DfGearPitch), R0 (DfGearRoll), P3 (MyBldc); mode axes J0..J4 = Y0, P1, P2, R0, P3.
 * ===================================================================================== */
enum { RK_AJ_Y0 = 0, RK_AJ_P1, RK_AJ_DFL, RK_AJ_DFR, RK_AJ_P2, RK_AJ_R0, RK_AJ_P3, RK_AJ_NUM };

/* JointBase::ConstParams of the seven joints (AD_task_main.cpp:38-107) + the mode cycle time */
typedef struct rk_adt_params {
  float ctrl_time_s[RK_AJ_NUM];  /* fl_ctrl_time_s  0.01f                       */
  float gear_ratio[RK_AJ_NUM];   /* fl_gear_ratio   1,1,1,1,24/7,48/7,48/19      */
  float motor_dir[RK_AJ_NUM];    /* fl_motor_dir    -1,1,1,1,1,1,-1              */
  float curlim_default_A[RK_AJ_NUM];
  float cycle_time_s;            /* ADTModeBase::FL_CYCLE_TIME_S 0.01f  AD_task_main.cpp:149 */
  /* homing (ADTModeInitialize / ADTModeInitPosMove) */
  float mechend_pos_deg[RK_AJ_NUM]; /* fl_mechend_pos_deg  -45,150,0,0,0,0,-90       */
  float vel_init_degps[RK_AJ_NUM];  /* fl_vel_init_degps   15,30,10,10,30,30,-60     */
  float curlim_init_A[RK_AJ_NUM];   /* fl_curlim_init_A    1,0.15,0.5,0.5,1,1,0.5    */
  float initpos_deg[RK_AJ_NUM];     /* fl_initpos_deg      0,145,0,0,-90,0,0         */
} rk_adt_params_t;
void rk_adt_default_params(rk_adt_params_t *p);

/* arm state words (19 planes = 76 words = 304 B / arm) */
enum {
  /* ADTModePositioningSeq  AD_mode_positioning_seq.hpp:55-70 */
  RK_AS_FSM = 0,        /* nowState | isModeFirstCall << 8 | is_comp << 9 */
  RK_AS_SEQ_IDX,        /* u16_seq_exec_idx_ | u16_seq_write_head_ << 16 */
  RK_AS_CMD_IDX,        /* u8_nowcmd_idx_ */
  RK_AS_MOVE_CNT,       /* s32_move_cnt_ */
  RK_AS_CYCLE,          /* s32_cycle_counter_ */
  RK_AS_TOTAL_MS,       /* u32_total_move_ms_ */
  RK_AS_NOW_DT,         /* now_cmd_.u32_dt_ms */
  RK_AS_RSV0,
  RK_AS_NOW_TGT = 8,    /* now_cmd_.fl_tgt_pos_deg[5] */
  RK_AS_MOVE_DEG = 13,  /* fl_move_deg_[5] */
  RK_AS_DFV_P = 18,     /* JointDfGearVirtual::fl_rawP_tgt_deg_  AD_joint_dfgear.hpp:35 */
  RK_AS_DFV_R,          /* ::fl_rawR_tgt_deg_ */
  /* 7 x JointBase {fl_out_ofs_deg, fl_raw_tgt_deg, fl_curlim_A, fl_raw_now_deg}  AD_joint_base.hpp:62-74 */
  RK_AS_JOINT0 = 20,
  RK_AS_JFLAGS = 48,    /* 4 bits per joint: connected | torque_on << 1 | initialized << 2 | torque_on_prev << 3 */
  RK_AS_MG_PRE_TGT,     /* JointMgServo::fl_pre_raw_tgt_deg */
  RK_AS_ICS_POS,        /* last position word handed to IcsBaseClass::setPos (-1: none) */
  RK_AS_ICS_SERVO,      /* ideal-servo model of the stubbed UART: position the servo reports */
  /* last transmitted servo commands */
  RK_AS_MG_TX = 52,     /* tx1data[8] (2 words), word 2 = bytes valid, word 3 rsv     AD_joint_mg_servo.hpp:93 */
  RK_AS_BLDC_TX0 = 56,  /* 3 x {txmsg[8] (2 words), u32_txcmdid, valid}: DF_Left, DF_Right, P3 */
  RK_AS_MG_CTRL = 68,   /* JointMgServo::pos_ctrl_ (UTIL::PI_D, the torque-control branches AD_joint_mg_servo.cpp:104-134):
                         * prev_val_, Integ_, velLpf_ y, velLpf_ x, now_tgt_, now_error_, now_ctrl_, "InitGain applied" */
  RK_AS_WORDS = 76
};
enum { RK_AJ_OFS = 0, RK_AJ_RAW_TGT, RK_AJ_CURLIM, RK_AJ_RAW_NOW };
enum { RK_ASTATE_STANDBY = 0, RK_ASTATE_MOVE_START, RK_ASTATE_MOVING, RK_ASTATE_COMPLETED };
#define RK_AS_FSM_FIRSTCALL 0x100u
#define RK_AS_FSM_IS_COMP 0x200u
#define RK_AJF_CONNECTED 1u
#define RK_AJF_TORQUE_ON 2u
#define RK_AJF_INITIALIZED 4u
#define RK_AJF_TORQUE_PREV 8u

/* Command-sequence ring, CMD_SEQ_BUF_LEN = 4 slots of PosCmdSeq per arm
 * (AD_mode_positioning_seq.hpp:11,15-24,59), in its own block so the 100 Hz state stays small:
 * slot s = 260 words = 65 planes: word 0 u32_id, word 1 u8_cmd_seq_len, words 2-3 zero, then
 * 32 waypoints of 8 words {u32_dt_ms, fl_tgt_pos_deg[5], 0, 0}.  Same plane indexing. */
#define RK_ACMD_SLOTS 4
#define RK_ACMD_MAX_LEN 32
#define RK_ACMD_SLOT_WORDS 260
#define RK_ACMD_WORDS (RK_ACMD_SLOTS * RK_ACMD_SLOT_WORDS)
typedef struct rk_adt_poscmd { uint32_t dt_ms; float tgt_deg[5]; } rk_adt_poscmd_t;
typedef struct rk_adt_poscmdseq { uint32_t id; uint8_t len; rk_adt_poscmd_t cmd[RK_ACMD_MAX_LEN]; } rk_adt_poscmdseq_t;

size_t rk_adt_state_words(void);
size_t rk_adt_state_bytes(int64_t n);
size_t rk_adt_cmdtab_bytes(int64_t n);

/* ADTModeBase::init() -> ADTModePositioningSeq::doInit()  (AD_mode_base.hpp:19-22,
 * AD_mode_positioning_seq.cpp:5-11) for every arm, and the joint flags/limits a finished
 * INIT mode leaves behind: connected, torque on, initialized, curlim = default
 * (AD_mode_initialize.cpp:133-135).  Offsets / targets are left as they are. */
int rk_adt_mode_init(const rk_adt_params_t *p, void *d_state, int64_t n, void *stream);
/* ADTModePositioningSeq::push_cmdseq (AD_mode_positioning_seq.cpp:124-137): one sequence per
 * arm from d_seq = n blocks of RK_ACMD_SLOT_WORDS words in plane order (pitch n); d_valid
 * (uint8[n] or NULL) selects the arms that push.  A full ring drops the push silently. */
int rk_adt_push_cmdseq(void *d_state, void *d_cmdtab, int64_t n, const void *d_seq, const uint8_t *d_valid, void *stream);
/* K fused arm ticks.  d_trace (optional): per tick 16 words, word j of tick t, arm i at
 * (t*16 + j)*n + i: 0-4 get_tgt_deg() of J0..J4; 5 MG u16_vel_lim; 6 MG s32_ang; 7-9 MyBldc
 * s32_tgt_ang_deg_Q16 of DF_Left, DF_Right, P3; 10 ICS position word; 11 nowState;
 * 12 u8_nowcmd_idx_; 13 MyBldc txcmdids packed (8 bits each, low byte of the id | 0x80 when
 * the id is >= 0x8000); 14-15 zero. */
#define RK_ADT_TRACE_WORDS 16
int rk_adt_update(const rk_adt_params_t *p, void *d_state, const void *d_cmdtab, int64_t n, int32_t K,
                  uint32_t *d_trace, void *stream);
/* ADTModePositioningSeq::get_q_cmdseq_status (AD_mode_positioning_seq.cpp:146-184):
 * d_status[i] in {0 PROCESSING, 1 DONE, 99 NO_DATA} for command id d_id[i]. */
int rk_adt_cmdseq_status(const void *d_state, const void *d_cmdtab, int64_t n, const uint32_t *d_id,
                         int32_t *d_status, void *stream);

/* ---- servo feedback (SURVEY 8f-3, arm side): the CAN rx callbacks of the arm's servos, one 8-byte frame per arm.
 * JointMyBldcServo::rx_callback -> rx_summary_status (AD_joint_mybldc_servo.cpp:45-70) for servo `slot` (0 DF_Left,
 * 1 DF_Right, 2 P3): fl_raw_now_deg = s16_out_ang_deg_Q4 / 16 / gear * dir, fl_out_now_cur = s8_motor_curr_A_Q4 / 16
 * * dir, and fl_raw_tgt_deg follows the measured angle while torque is off.  d_cmdid (uint32[n], the id without the
 * device id; NULL = CMD_ID_RES_STATUS_SUMMARY 0x1000 for all): other ids are ignored as in the firmware.
 * d_cur_A (float[n], optional) receives fl_out_now_cur -- nothing on the tick reads it, so it is not a state word. */
int rk_adt_bldc_rx(const rk_adt_params_t *p, void *d_state, int64_t n, int slot, const uint64_t *d_frames, const uint32_t *d_cmdid,
                   float *d_cur_A, void *stream);
/* JointMgServo::rx_callback (AD_joint_mg_servo.cpp:75-92): command byte 0x9C / 0xA1 -> fl_out_now_cur through the
 * double-precision quadratic conv_raw_to_current (AD_joint_mg_servo.hpp:120-128) into d_cur_A (optional; untouched by
 * other frames); 0x92 -> fl_raw_now_deg from the multi-turn angle (and fl_raw_tgt_deg while torque is off).  The
 * firmware's byte assembly shifts a promoted int by up to 48 bits (undefined in C++): the Cortex-M7 result -- the
 * sign-extended low 32 bits -- is what is computed; the x86 build of the reference agrees for frames whose bytes 5..7
 * are zero.  Other command bytes are ignored. */
int rk_adt_mg_rx(const rk_adt_params_t *p, void *d_state, int64_t n, const uint64_t *d_frames, float *d_cur_A, void *stream);

/* ---- ADTModePositioning (src/ArmDrive/AD_mode_positioning.{hpp,cpp}): the single-command mode behind
 * REQ_MOVE_POS (AD_task_main.cpp:260-272).  Same joints (the RK_AS_* block), its own mode block:
 * a FIFO of at most four commands (std::deque, push drops the OLDEST when full, :118-124), the
 * move measured from get_now_deg() (:42-46), one state handler per update (:9-20). */
enum {
  RK_PS_STATE = 0,     /* nowState (0 STANDBY, 1 MOVING, 2 COMPLETED) | is_comp << 9 */
  RK_PS_MOVE_CNT,      /* u32_move_cnt_ */
  RK_PS_CYCLE,         /* u32_cycle_counter_ */
  RK_PS_QSIZE,         /* cmd_q_.size() */
  RK_PS_PREV_ID0 = 4,  /* u32_prev_cmd_id_[0], [1] */
  RK_PS_PREV_ID1,
  RK_PS_NOW_CMD = 8,   /* now_cmd_: u32_id, u32_dt_ms, fl_tgt_pos_deg[5], 0 */
  RK_PS_MOVE_DEG = 16, /* fl_move_deg_[5], 0, 0, 0 */
  RK_PS_QUEUE = 24,    /* cmd_q_ front first: 4 x {u32_id, u32_dt_ms, fl_tgt_pos_deg[5], 0} */
  RK_PS_WORDS = 56     /* 14 planes = 224 B */
};
typedef struct rk_adp_poscmd { uint32_t id, dt_ms; float tgt_deg[5]; } rk_adp_poscmd_t; /* == ADTModePositioning::PosCmd */
size_t rk_adp_state_words(void);
size_t rk_adp_state_bytes(int64_t n);
/* ADTModeBase::init() -> ADTModePositioning::doInit()  (AD_mode_base.hpp:19-22, AD_mode_positioning.cpp:5-7) */
int rk_adp_mode_init(void *d_pstate, int64_t n, void *stream);
/* ::push_cmd (:118-124).  d_cmd: two planes per arm, {id, dt_ms, tgt0, tgt1} and {tgt2, tgt3, tgt4, 0} (pitch n) */
int rk_adp_push_cmd(void *d_pstate, int64_t n, const void *d_cmd, const uint8_t *d_valid, void *stream);
/* K fused ticks of ADT::main's loop body with this mode active; trace as rk_adt_update (word 11 = nowState,
 * word 12 = queue size) */
int rk_adp_update(const rk_adt_params_t *p, void *d_state, void *d_pstate, int64_t n, int32_t K, uint32_t *d_trace, void *stream);
/* ::get_q_cmd_status (:134-148): 0 PROCESSING (queued), 1 DONE (one of the last two finished), 99 NO_DATA */
int rk_adp_cmd_status(const void *d_pstate, int64_t n, const uint32_t *d_id, int32_t *d_status, void *stream);

/* ---- Homing modes (SURVEY 8f-4): ADTModeInitialize (src/ArmDrive/AD_mode_initialize.{hpp,cpp}: INIT -> TORQUE_ON
 * (100 cycles) -> MOVE_MECH_END (500 cycles, J1 and J4 pushed towards their mechanical end at the init speed and
 * current limit, the target frozen while it leads the measured angle by more than 45 deg) -> RESET_ANGLE
 * (JointBase::mech_reset_pos and the DfGear overrides re-reference the offsets) -> MOVE_INIT_POS (every axis ramps
 * to its init pose) -> COMPLETED) and ADTModeInitPosMove (AD_mode_initpos_move.{hpp,cpp}: the same without touching
 * the offsets).  Same joints (the RK_AS_* block: the modes switch torque / initialised flags, current limits and
 * offsets, so the MG joint passes through its torque-control branches), their own mode block: */
enum {
  RK_HS_STATE = 0,    /* nowState | is_comp << 9 | mode << 16 */
  RK_HS_WAIT_CNT,     /* u16_wait_cnt_ */
  RK_HS_VEL_DIR = 4,  /* ADTModeInitPosMove::fl_move_vel_dir_[5] */
  RK_HS_WORDS = 12    /* 3 planes */
};
enum { RK_ADH_MODE_INIT = 1, RK_ADH_MODE_INIT_POS_MOVE = 2 };
size_t rk_adh_state_words(void);
size_t rk_adh_state_bytes(int64_t n);
/* ADTModeBase::init() -> doInit() of the chosen mode for every arm */
int rk_adh_mode_init(void *d_hstate, int64_t n, int mode, void *stream);
/* K fused ticks of ADT::main's loop body with the homing mode active.  d_now (optional): the angles the servos
 * reported since the last tick, float [K][4][n] = fl_raw_now_deg of P1 (MG), DF_Left, DF_Right, P3 (MyBldc) as their
 * CAN rx callbacks store them, applied before the mode runs; NULL keeps the angles of the state block (Y0 always
 * follows the ideal ICS servo).  Trace as rk_adt_update with word 11 = nowState, word 12 = u16_wait_cnt_. */
int rk_adh_update(const rk_adt_params_t *p, void *d_state, void *d_hstate, int64_t n, int32_t K, const float *d_now,
                  uint32_t *d_trace, void *stream);

/* single-instance handle (drop-in for the statics of AD_task_main.cpp:108-156) */
/* Self-test (tests): the arm tick divides its five per-segment steps by one count through a shared double-precision
 * reciprocal (csrc/rk_arm.cu div_by_rcp64, proven equal to the IEEE division); this compares the two on `pairs`
 * pseudo-random (x, c) pairs on the device and returns the number of mismatches.  Synchronous. */
int rk_selftest_div_rcp64(uint64_t pairs, uint64_t seed, uint32_t *mismatches);

typedef struct rk_adt rk_adt_t;
int  rk_adt_create(rk_adt_t **out, const rk_adt_params_t *p /* NULL = defaults */);
void rk_adt_destroy(rk_adt_t *h);
int  rk_adt_init(rk_adt_t *h);                                    /* mode init, see rk_adt_mode_init */
int  rk_adt_push(rk_adt_t *h, const rk_adt_poscmdseq_t *seq);     /* push_cmdseq                     */
int  rk_adt_tick(rk_adt_t *h);                                    /* one ADT::main loop body         */
int  rk_adt_home_init(rk_adt_t *h, int mode);                     /* set_next_mode(INIT / INIT_POS_MOVE): RK_ADH_MODE_* */
/* one loop body with the homing mode active; servo_now_deg (or NULL): fl_raw_now_deg of P1, DF_Left, DF_Right, P3
 * as received since the last tick; *completed = ADTModeBase::isCompleted() */
int  rk_adt_home_tick(rk_adt_t *h, const float servo_now_deg[4], int *completed);
int  rk_adt_status(rk_adt_t *h, uint32_t id, int32_t *status);    /* get_q_cmdseq_status             */
/* JointMyBldcServo::rx_callback(cmdid, frame) for slot 0 DF_Left / 1 DF_Right / 2 P3, JointMgServo::rx_callback(frame) for
 * slot 3 (cmdid unused); *cur_A (optional) receives fl_out_now_cur when the frame carries a current */
int  rk_adt_rx(rk_adt_t *h, int slot, uint32_t cmdid, const uint8_t frame[8], float *cur_A);
int  rk_adt_get_targets_deg(rk_adt_t *h, float out[5]);           /* JointBase::get_tgt_deg x5       */
int  rk_adt_get_state(rk_adt_t *h, uint32_t words[RK_AS_WORDS]);
int  rk_adt_set_state(rk_adt_t *h, const uint32_t words[RK_AS_WORDS]);

/* =====================================================================================
 * Full controller tick (BASELINE configs[4]): vehicle at 1 kHz, IMU update + arm tick every
 * `slow_period` vehicle ticks (10: the tasks run at 100 Hz, imu_task_main.cpp:17,
 * AD_task_main.cpp loop), coupled exactly as the firmware couples them: the vehicle ISR reads
 * deg2rad(IMU yaw) before every update (VD_task_main.cpp:368).  Slow tick k runs before
 * vehicle tick k * slow_period.  The three sub-systems are independent apart from that yaw:
 * the vehicle rollout forms it from the IMU's register snapshots itself (rk_vdt_rollout_t::
 * d_imu_regs), so no kernel waits for another -- the IMU update and the arm tick run on an
 * internal high-priority side stream inside the vehicle rollout's shadow (csrc/rk_tick.cu).
 * The call is asynchronous on `stream` like every other batch call; concurrent callers on one
 * device are serialised while they enqueue.
 * ===================================================================================== */
struct rk_stream_desc;
typedef struct rk_tick_rollout {
  int32_t steps;             /* K vehicle ticks */
  int32_t slow_period;       /* vehicle ticks per IMU / arm tick (firmware: 10) */
  const rk_vdt_cmd_t *d_cmd; /* vehicle commands, as rk_vdt_rollout_t */
  int32_t n_seg, seg_len;
  const int16_t *d_regs;     /* IMU samples as rk_imt_update takes them (two 128-bit cells each), n_slow = ceil(K / slow_period) */
  const uint8_t *d_have_quat;/* [n_slow][n] or NULL */
  float *d_yaw;              /* scratch, >= n floats (receives Data.angle[2] of every IMU block as it was at launch) */
  const float *d_goal;       /* optional cost epilogue, as rk_vdt_rollout_t */
  float *d_cost;
  uint32_t *d_vdt_trace;     /* optional traces (tests) */
  uint32_t *d_adt_trace;
  int32_t reset_vehicle;     /* != 0: the vehicles start from the power-on block (rk_vdt_rollout_t::reset_state) */
  const int16_t *d_yaw_reg;  /* optional [n_slow][n]: the Yaw register column of d_regs (register RK_IMT_REG_YAW of every sample) in
                                2 bytes per sample.  The vehicle rollout then reads the yaw from here instead of from the 16-byte
                                register cells (16 B of sector traffic per sample): same values, same hold semantics, 1.6 GB less
                                DRAM traffic per 2^20 robots x 1000 ticks.  rk_stream_imu_samples_yaw() writes it as a by-product. */
  const struct rk_stream_desc *d_imu_desc; /* optional (needs d_yaw_reg; d_regs may then be NULL): the IMU samples are those of
                                rk_stream_imu_samples(d_imu_desc, ...) and the IMU update draws them in registers instead of reading
                                a table -- 3.2 KB per robot and launch that are neither written nor read.  d_yaw_reg / d_have_quat
                                are the columns rk_stream_imu_samples_yaw(d_imu_desc, n, n_slow, NULL, d_have_quat, d_yaw_reg) wrote. */
} rk_tick_rollout_t;

int rk_tick_rollout(const rk_vdt_params_t *vp, const rk_adt_params_t *ap, void *d_vdt_state, void *d_imt_state,
                    void *d_adt_state, const void *d_adt_cmdtab, int64_t n, const rk_tick_rollout_t *args, void *stream);
/* Diagnostics (tools/tick_timeline.py): enable != 0 makes later rk_tick_rollout calls record timestamps; with out !=
 * NULL the call synchronises the device and returns, for the last rk_tick_rollout on the current device, milliseconds
 * since its entry: side stream starts, IMU kernel done, arm kernel done, vehicle rollout starts, vehicle rollout done. */
int rk_tick_debug_timeline(int enable, float out[5]);

/* =====================================================================================
 * Synthetic command / sensor streams (SURVEY.md 8d), generated on the device.  A rollout engine fed over PCIe
 * is bound by the host link (the full tick consumes 4.5 KB of tables per robot and launch); a planner ships the
 * distribution, not the samples.  Each call expands a descriptor held in DEVICE memory into the block the
 * corresponding engine entry consumes, for the n robots first .. first + n - 1 of the global index space.  The
 * streams are defined by streams.py (`*_v2`, a 32-bit counter hash of (seed, stream, robot, index)); the kernels
 * reproduce them bit for bit (tests/test_streams_gpu.py).
 * ===================================================================================== */
typedef struct rk_stream_desc {
  int64_t  first;             /* global index of the batch's robot 0 (robots are hashed modulo 2^32) */
  uint32_t seed;
  uint32_t first_update;      /* IMU: update index of sample 0 */
  uint32_t stop_every;        /* vehicle commands: one segment in stop_every is a STOP (0: never) */
  uint32_t drop_every;        /* IMU: one update in drop_every carries no quaternion frame (0: never) */
  uint32_t arm_min_len, arm_max_len, arm_seq_id, arm_dt_zero_every;
  uint32_t rsv[2];
} rk_stream_desc_t; /* 48 bytes */
void rk_stream_default_desc(rk_stream_desc_t *d); /* seed 0x5EED, first 0, 8, 64, 2..32 waypoints, id 1, 4 */
/* [n_seg][n] rk_vdt_cmd_t (RK_CMD_MOVE / RK_CMD_STOP): vx, vy ~ U[-400, 400] mm/s through speed_limit_xy
 * (VD_task_main.cpp:127-137), vth ~ U[-2 pi, 2 pi] through speed_limit_rot (:139-142) */
int rk_stream_vehicle_commands(const rk_stream_desc_t *d_desc, int64_t n, int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream);
/* int16 [n_yaw][n]: the WT901C Yaw register of a vehicle turning at a constant 1..5 x 182 counts per sample */
int rk_stream_vehicle_yaw_reg(const rk_stream_desc_t *d_desc, int64_t n, int32_t n_yaw, int16_t *d_yaw_reg, void *stream);
/* rk_stream_imu_samples() that also writes the Yaw register of every sample as a 2-byte column [n_upd][n]
 * (rk_tick_rollout_t::d_yaw_reg); d_yaw_reg NULL = rk_stream_imu_samples(); d_regs NULL (d_yaw_reg 16-byte aligned): only
 * the columns are written, for a rollout whose IMU update draws the samples itself (rk_tick_rollout_t::d_imu_desc) */
int rk_stream_imu_samples_yaw(const rk_stream_desc_t *d_desc, int64_t n, int32_t n_upd, int16_t *d_regs, uint8_t *d_have_quat,
                              int16_t *d_yaw_reg, void *stream);
/* WT901 register snapshots in the two-cells-per-sample layout of rk_imt_update (+ have_quat [n_upd][n], may be NULL) */
int rk_stream_imu_samples(const rk_stream_desc_t *d_desc, int64_t n, int32_t n_upd, int16_t *d_regs, uint8_t *d_have_quat, void *stream);
/* one PosCmdSeq per arm as the 65-plane slot image rk_adt_push_cmdseq takes */
int rk_stream_arm_sequences(const rk_stream_desc_t *d_desc, int64_t n, void *d_seq, void *stream);

/* =====================================================================================
 * Vehicle sampling planner: one planning step for R robots with S candidates each is three calls on one stream,
 *   rk_plan_sample_commands  nominal [n_seg][R]           -> candidates [n_seg][R*S]
 *   rk_plan_rollout          R source states + candidates -> cost [R*S]       (source states untouched)
 *   rk_plan_select           cost + candidates            -> new nominal [n_seg][R], best index / cost [R]
 * after which the caller runs the first segment of the new nominal on its robots with rk_vdt_rollout.  Candidate j
 * of robot r is instance r*S + j everywhere.  Every float result is defined as single IEEE float32 operations (round
 * to nearest, no contraction) in the order written here; streams.plan_commands_v2 restates the sampler in numpy.
 * Arguments are checked (RK_ERR_ARG): R >= 0, S >= 1, n_seg * S < 2^32, seg_len >= 1, 0 <= shift < n_seg, lambda >= 0
 * and finite, state blocks and command tables 16-byte aligned.  R == 0 is a no-op.
 * ===================================================================================== */
typedef struct rk_plan_sample {
  int64_t  first;     /* global index of robot 0 (sharded planners draw the same noise as one GPU would) */
  uint32_t seed;
  uint32_t rsv;
  float    sigma[3];  /* noise scale of vx, vy (mm/s) and vth (rad/s) */
  float    rsv2;
} rk_plan_sample_t; /* 32 bytes */

typedef struct rk_plan_cost {
  const float *d_ref; /* float2 [n_seg][R]: where robot r should be (m) when segment s ends; s = n_seg-1 is the goal */
  float w_pos;        /* weight of |pos - ref_s|^2 at the end of segments 0 .. n_seg-2 */
  float w_goal;       /* weight of |pos - ref_{n_seg-1}|^2 after the last tick */
  float w_cur;        /* weight of sum_w cur_tgt_w^2 at the end of every segment */
  float rsv;
} rk_plan_cost_t; /* 24 bytes */

/* Candidate j of robot r (global index g = first + r), segment s: j == 0 is the nominal itself; otherwise, with
 * h = streams.h32(seed, 40, g, s*S + j) and u_k = u01_32(lite32(h, 4a + k)), axis a gets
 * xi_a = ((((u_0 + u_1) + u_2) + u_3) - 2) * 1.7320508f (Irwin-Hall, unit variance) and v_a = nom_a + sigma_a * xi_a.
 * Then speed_limit_xy: ln = sqrtf(vx*vx + vy*vy); ln > p->limit_speed_mmps (L) -> vx = (vx*L)/ln, vy = (vy*L)/ln; vth is
 * clamped to +-p->limit_rot_radps; kind = RK_CMD_MOVE (the nominal's kind is ignored).  d_cmd must not overlap d_nominal. */
int rk_plan_sample_commands(const rk_vdt_params_t *p, const rk_plan_sample_t *s, const rk_vdt_cmd_t *d_nominal,
                            int64_t R, int32_t S, int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream);
/* n_seg * seg_len closed-loop ticks (RK_SENSOR_PLANT) of candidate r*S + j from robot r's block of d_src_state (pitch R),
 * command cell [s][r*S + j] applied before tick s*seg_len as rk_vdt_rollout applies d_cmd; no yaw stream and no task
 * loop (the source heading is held).  At the end of segment s, with (x, y) the position words and c_k = (float) the
 * sign-extended s16_rawCurr_tgt of wheel k:
 *   dx = x - ref[s].x;  dy = y - ref[s].y;  e = dx*dx + dy*dy;  q = ((c0*c0 + c1*c1) + c2*c2) + c3*c3
 *   J  = (J + (s < n_seg-1 ? w_pos : w_goal) * e) + w_cur * q          (J starts at 0)
 * d_cost[r*S + j] = J.  No state is written.  The kernel is chosen as for rk_vdt_rollout (RK_OPT_* included); the costs
 * do not depend on it. */
int rk_plan_rollout(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S,
                    const rk_vdt_cmd_t *d_cmd, int32_t n_seg, int32_t seg_len,
                    const rk_plan_cost_t *cost, float *d_cost, void *stream);

typedef struct rk_plan_obstacles {
  const float *d_obs;   /* float4 [m][R]: disc k of robot r at cell k*R + r = {cx, cy, radius, unused}, metres; 16-byte aligned */
  int32_t m;            /* discs per robot, >= 0 */
  int32_t check_period; /* P >= 1 ticks; seg_len % P == 0 */
  float   w_obst;       /* >= 0, may be +INFINITY (a hard constraint); NaN rejected */
  float   rsv;
} rk_plan_obstacles_t;  /* 24 bytes */

/* rk_plan_rollout with keep-out discs.  Checkpoints are the states after ticks c*P - 1, c = 1 .. K/P (K = n_seg *
 * seg_len): every segment end is one, and so is the last tick.  O starts at 0; at each checkpoint, for k = 0 .. m-1 in
 * order, with (x, y) the position words and {cx, cy, radius} disc k of robot r:
 *   dx = x - cx;  dy = y - cy;  d2 = dx*dx + dy*dy;  pen = radius*radius - d2;  if (pen > 0) O = O + w_obst * pen
 * (a NaN radius or centre contributes nothing; with w_obst = +inf one penetration makes O = +inf).
 * d_cost[r*S + j] = J + O, J exactly the rk_plan_rollout cost, accumulated separately.  obst == NULL or m == 0 is
 * rk_plan_rollout (the same kernel, the same bits); for J >= 0 so is w_obst == 0.  Everything else is as rk_plan_rollout:
 * RK_SENSOR_PLANT, source states untouched, no state written, the kernel chosen by the same RK_OPT_* switches, and the
 * cost does not depend on it.  RK_ERR_ARG besides rk_plan_rollout's checks: m < 0; m > 0 with d_obs NULL or not 16-byte
 * aligned; P < 1 or seg_len % P != 0; w_obst < 0 or NaN.  R == 0 is a no-op. */
int rk_plan_rollout_obstacles(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S,
                              const rk_vdt_cmd_t *d_cmd, int32_t n_seg, int32_t seg_len,
                              const rk_plan_cost_t *cost, const rk_plan_obstacles_t *obst,
                              float *d_cost, void *stream);
/* best[r] = argmin_j cost[r*S + j] (NaN counts as +inf, ties to the lowest j; all NaN: 0), best_cost[r] = that cost.
 * nominal_out[s][r] takes segment s + shift of the candidates (the last segment repeated past the end):
 *   lambda == 0: candidate best copied bit for bit;
 *   lambda > 0:  vx, vy, vth = sum_j w_j v_j / sum_j w_j with w_j = expf(-(c_j - c_min) / lambda) (NaN cost: w = 0),
 *                kind = RK_CMD_MOVE, in a fixed reduction order (repeatable bit for bit); a robot without a finite
 *                minimum cost gets candidate best as under lambda == 0.
 * d_best / d_best_cost may be NULL.  d_nominal_out must not overlap d_cmd. */
int rk_plan_select(const float *d_cost, const rk_vdt_cmd_t *d_cmd, int64_t R, int32_t S, int32_t n_seg,
                   float lambda, int32_t shift, rk_vdt_cmd_t *d_nominal_out, int32_t *d_best, float *d_best_cost,
                   void *stream);

/* Cross-entropy planning (CEM): several sample -> rollout -> refit rounds per planning step from the same source states,
 * each drawing the candidates from a per-robot, per-segment distribution (nominal, sigma table) and refitting it to the
 * round's k best candidates:
 *   rk_plan_sample_commands_sigma  nominal + sigma [n_seg][R]  -> candidates [n_seg][R*S]
 *   rk_plan_rollout(_obstacles)    as above                    -> cost [R*S]
 *   rk_plan_refit                  cost + candidates + sigma   -> new nominal + sigma [n_seg][R], best index / cost [R] */

/* rk_plan_sample_commands with the noise scale taken per robot and segment: axis a of candidate j > 0 of robot r,
 * segment s is nom_a + d_sigma[s*R + r][a] * xi_a.  xi, the hash, j == 0, the limiters and kind are exactly those of
 * rk_plan_sample_commands, and s->sigma is ignored.  So a table holding s->sigma in every cell gives the same bits as
 * rk_plan_sample_commands.  d_sigma: float4 [n_seg][R] {sx, sy, sth, unused}, 16-byte aligned, and it must not overlap
 * d_cmd.  Argument checks as rk_plan_sample_commands, plus d_sigma NULL, misaligned or overlapping d_cmd (RK_ERR_ARG). */
int rk_plan_sample_commands_sigma(const rk_vdt_params_t *p, const rk_plan_sample_t *s, const rk_vdt_cmd_t *d_nominal,
                                  const float *d_sigma, int64_t R, int32_t S, int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream);

typedef struct rk_plan_refit {
  int32_t elite;        /* k, 1 <= k <= S */
  float   alpha;        /* smoothing toward the previous distribution, 0 <= alpha <= 1 (0: none) */
  float   sigma_min[3]; /* floor of the refitted sigma, finite and >= 0 */
  float   rsv;
} rk_plan_refit_t;      /* 24 bytes */

/* Refit of robot r's distribution to its elite candidates.  Every float operation is one IEEE float32 operation (round to
 * nearest, no contraction) in the order written.
 *   Order:  candidates are ordered by (cost, j), costs compared as floats (-0 equals +0), ties to the lower j.
 *   Elites: E_r = the first k_eff = min(k, number of finite costs of r) candidates in that order; a NaN or +-inf cost is
 *           never an elite (a candidate priced +inf by w_obst = INFINITY never weighs in the mean).
 *   Best:   d_best / d_best_cost exactly as rk_plan_select writes them (argmin, NaN as +inf, all NaN: 0); either may be NULL.
 *   Output segment s reads source segment ss = min(s + shift, n_seg - 1), as rk_plan_select does.  Per axis a, with v the
 *   axis-a word of the candidate's cell [ss][r*S + j] and the elites taken in ascending j:
 *     m   = (((v_e0 + v_e1) + ...) + v_e(k_eff-1)) / (float)k_eff     (the sum starts from the first elite)
 *     q   = ((0 + (v_e0 - m)*(v_e0 - m)) + ...) + (v_e(k_eff-1) - m)*(v_e(k_eff-1) - m)
 *     sd  = sqrtf(q / (float)k_eff)
 *     alpha > 0:  mean = alpha*c0 + (1 - alpha)*m,  sig = alpha*sigma_in[ss][a] + (1 - alpha)*sd
 *                 (c0: candidate 0 of robot r in segment ss, the centre that segment was drawn around)
 *     alpha == 0: mean = m,  sig = sd
 *   sigma_out[s][r] = {fmaxf(sig_x, sigma_min[0]), fmaxf(sig_y, sigma_min[1]), fmaxf(sig_th, sigma_min[2]), 0} and
 *   nominal_out[s][r] = {mean_x, mean_y, mean_th, RK_CMD_MOVE}.  k_eff == 0 (no finite cost): nominal_out[s][r] is candidate
 *   best of segment ss and sigma_out[s][r] is sigma_in[ss][r], both copied bit for bit.
 * d_sigma_in / d_sigma_out: float4 [n_seg][R], 16-byte aligned.  RK_ERR_ARG: rk_plan_select's checks; rf NULL; elite
 * outside [1, S]; alpha NaN or outside [0, 1]; a sigma_min NaN, negative or inf; a NULL or misaligned sigma table;
 * d_nominal_out overlapping d_cmd; d_sigma_out overlapping d_sigma_in, except the same table with shift == 0 (each robot
 * and segment reads only its own cell then).  R == 0 is a no-op.  No limit on S or k beyond n_seg * S < 2^32. */
int rk_plan_refit(const float *d_cost, const rk_vdt_cmd_t *d_cmd, const float *d_sigma_in, int64_t R, int32_t S,
                  int32_t n_seg, const rk_plan_refit_t *rf, int32_t shift, rk_vdt_cmd_t *d_nominal_out,
                  float *d_sigma_out, int32_t *d_best, float *d_best_cost, void *stream);

/* Moving keep-out discs and predicted paths (fleet planning): every robot of a planner keeps clear of the positions its
 * peers' nominal plans predict, checkpoint by checkpoint.  One fleet step on one stream:
 *   rk_plan_rollout_moving (S = 1, d_cmd = nominal, m = 0, d_path)  R states + nominal   -> path [n_ck][R]
 *   rk_plan_peer_discs                                               path + peer indices -> discs [n_ck][M][R]
 *   rk_plan_sample_commands, rk_plan_rollout_moving (the discs), rk_plan_select as above
 * Positions are checked at checkpoints only, and the peers replan every step, so this is avoidance by cost, not a
 * guarantee (INTEGRATION.md §2). */

/* rk_plan_rollout_obstacles with a disc table per checkpoint, and optionally the candidates' paths.  obst is required;
 * n_ck = n_seg * seg_len / P.  obst->d_obs is float4 [n_ck][m][R]: cell (c*m + k)*R + r is disc k of robot r at
 * checkpoint c + 1, the state after tick (c + 1)*P - 1.  The checkpoints, the per-disc formula, its float32 order, NaN
 * discs and w_obst = +inf are those of rk_plan_rollout_obstacles; checkpoint c reads its own table.  So a table repeating
 * one [m][R] table at every checkpoint gives rk_plan_rollout_obstacles' bits, and m == 0 gives rk_plan_rollout's.
 * d_path (NULL: not written): float2 [n_ck][R*S], 8-byte aligned; cell c*R*S + i = the position words (x, y) of
 * candidate i at checkpoint c + 1, bit for bit the words the cost read.  Writing it never changes d_cost.
 * RK_ERR_ARG: rk_plan_rollout_obstacles' checks, obst NULL, and d_path not 8-byte aligned. */
int rk_plan_rollout_moving(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S,
                           const rk_vdt_cmd_t *d_cmd, int32_t n_seg, int32_t seg_len,
                           const rk_plan_cost_t *cost, const rk_plan_obstacles_t *obst,
                           float *d_path, float *d_cost, void *stream);

/* Peer discs from predicted paths: d_path float2 [n_ck][R] (8-byte aligned), d_peer int32 [m][R], d_obs float4
 * [n_ck][M][R] (16-byte aligned).  For c < n_ck, k < m, r < R with q = d_peer[k*R + r], cell (c*M + k0 + k)*R + r becomes
 *   {path[c][q].x, path[c][q].y, radius, 0}   if 0 <= q < R and q != r,
 *   {0, 0, NaN, 0}                             otherwise (a disc that contributes nothing; nothing out of range is read).
 * Cells of slots outside [k0, k0 + m) are not touched, so static discs or several peer sets can share one table.
 * RK_ERR_ARG: R < 0, n_ck < 0, m < 0, k0 < 0, k0 + m > M, radius NaN, inf or < 0, a NULL or misaligned table (when
 * R, n_ck and m are > 0), d_obs overlapping d_path.  R, n_ck or m == 0 is a no-op. */
int rk_plan_peer_discs(const float *d_path, int64_t R, int32_t n_ck, const int32_t *d_peer, int32_t m, float radius,
                       float *d_obs, int32_t M, int32_t k0, void *stream);

/* Cost maps: a grid of cell costs, stored once per world (not per robot) and looked up at every checkpoint, one cell load
 * whatever the world holds -- walls, corridors, shelving.  It shares the checkpoints and the accumulator O with the discs,
 * so peer discs and a building map compose in one rollout.  The robot is a point read at checkpoints only: inflate walls by
 * the body radius plus the distance covered in P ticks (at most 0.4 mm per tick at 400 mm/s) with rk_plan_inflate, see
 * INTEGRATION.md §2. */
typedef struct rk_plan_map {
  const float   *d_cells;  /* float [n_maps][height][width]: cell (ix, iy) of map k at (k*height + iy)*width + ix; 4-byte aligned */
  const int32_t *d_map_of; /* int32 [R]: the map of robot r; NULL: map 0 for every robot */
  int32_t n_maps, width, height;  /* >= 1 each; n_maps*height*width < 2^31; width, height <= 2^24 */
  float   x0, y0;          /* metres: the outer corner of cell (0, 0); finite */
  float   inv_res;         /* cells per metre; finite, > 0 */
  float   outside;         /* the value of every point off the grid; may be +inf; NaN rejected */
  float   w_map;           /* >= 0, may be +inf; NaN rejected */
} rk_plan_map_t;           /* 48 bytes */

/* rk_plan_rollout_moving plus a map term.  obst is required (it gives check_period; m may be 0), d_path as there.  At each
 * checkpoint: the path cell is stored, discs k = 0 .. m-1 are added to O exactly as rk_plan_rollout_moving does, then the
 * map term is added to the same O.  Each operation is one IEEE float32 operation in the written order, no contraction:
 *   k = d_map_of ? d_map_of[r] : 0;        k < 0 or k >= n_maps: no map term for robot r
 *   u = (x - x0) * inv_res;  v = (y - y0) * inv_res
 *   c = (u >= 0 && u < (float)width && v >= 0 && v < (float)height) ? cells[(k*height + (int)v)*width + (int)u] : outside
 *   if (c > 0) O = O + w_map * c
 * So a NaN position reads `outside`; NaN, zero and negative cells contribute nothing; a +inf cell, or w_map = +inf with a
 * cell above 0, makes O = +inf (a hard wall).  d_cost = J + O.  map == NULL or w_map == 0 is rk_plan_rollout_moving (the
 * same kernel and bits, never 0 * inf).  Cells are read with ordinary loads: no texture filtering.
 * RK_ERR_ARG: rk_plan_rollout_moving's checks; d_cells NULL or not 4-byte aligned; d_map_of not 4-byte aligned; n_maps,
 * width or height < 1, width or height > 2^24, n_maps*height*width >= 2^31; x0, y0 or inv_res not finite, inv_res <= 0;
 * outside NaN; w_map < 0 or NaN.  R == 0 is a no-op. */
int rk_plan_rollout_map(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S,
                        const rk_vdt_cmd_t *d_cmd, int32_t n_seg, int32_t seg_len, const rk_plan_cost_t *cost,
                        const rk_plan_obstacles_t *obst, const rk_plan_map_t *map, float *d_path, float *d_cost,
                        void *stream);

/* Cost-to-go fields (navigation functions): the shortest-path distance from a goal through the free cells of a cost map,
 * built on the device.  Used as a rollout's terminal cost it has no local minimum except at the goal, so robots route
 * around walls and out of dead ends that the straight-line goal term w_goal * |pos - goal|^2 traps them in.
 *   rk_plan_cost_to_go     map + goals [n_fields]                -> fields [n_fields][fh][fw] (synchronises the stream)
 *   rk_plan_rollout_field  rk_plan_rollout_map + the field term  -> cost [R*S]
 * Build fields when goals or the map change, not every planning step (INTEGRATION.md §2). */
typedef struct rk_plan_ctg {
  float step_axial, step_diag; /* metres per axial / diagonal step; finite, > 0 (e.g. float(res), float(res * sqrt(2))) */
  float k_cost;                /* extra traversal cost per unit of cell cost; finite, >= 0 */
  float lethal;                /* a cell with c >= lethal is not traversable; > 0, may be +inf (then only +inf cells block) */
} rk_plan_ctg_t;               /* 16 bytes */

/* Field f is a fw x fh window of map k = d_field_map[f] (NULL: 0) of `map`; window cell (ix, iy) is map cell
 * (ox + ix, oy + iy), (ox, oy) = d_offset[f] (NULL: (0, 0)).  Cell (ix, iy) of field f is d_field[(f*fh + iy)*fw + ix].
 * Every operation is one IEEE float32 operation in the written order, no contraction:
 *   cost     c = map cell (ox + ix, oy + iy) of map k, or map->outside where that cell is off the map
 *   blocked  c >= lethal  (NaN compares false: a NaN cell never blocks)
 *   factor   t = c > 0 ? 1 + k_cost*c : 1
 *   goal     gu = (gx - map->x0)*map->inv_res, gv likewise.  If gu >= (float)ox && gu < (float)(ox + fw) and the same for
 *            gv, the goal cell is ((int)floorf(gu) - ox, (int)floorf(gv) - oy).  Otherwise the field has no goal and is
 *            +inf everywhere: a NaN goal, a goal off the window, k outside [0, n_maps), or a window whose |ox|, |oy|,
 *            |ox + fw| or |oy + fh| exceeds 2^24 (where (float) is no longer exact).
 *   edges    the goal cell gets D = 0, even if blocked.  An edge p -> q runs to each of the 8 neighbours q of p that lies
 *            in the window and is not blocked; a diagonal edge also needs both cells that share a side with p and with q
 *            to be in the window and unblocked (no corner cutting).  Its weight is w = step * t_q (step_axial or
 *            step_diag).
 *   field    D(q) = the minimum over all paths from the goal of the left fold D = D + w; +inf where no path reaches q
 *            (blocked cells other than the goal included).
 * The bits do not depend on the order of relaxation: fl(a + w) is monotone in a and w >= 0, so every relaxation keeps D(q)
 * an upper bound that some path attains, and any order that runs to a fixed point (Bellman-Ford in any order, chaotic
 * in-place updates, or a float32 Dijkstra) stops at the same minimum.  The device relaxes 32 x 32 tiles in rounds, each
 * tile in place in shared memory until it stops changing, and runs the next round over the tiles that changed and their
 * neighbours; the host enqueues rounds in batches and reads the number of changed tiles after each batch, so the call
 * synchronises `stream`.  It ends after the first round that changes nothing; no cap is needed, since values only
 * decrease over finitely many floats.  *rounds_out (may be NULL) = the number of rounds that changed a cell.
 * d_goal: float2 [n_fields] metres, 8-byte aligned; d_field_map: int32 [n_fields] (may be NULL); d_offset: int2
 * [n_fields], 8-byte aligned (may be NULL); d_field: float [n_fields][fh][fw]; d_work: rk_plan_cost_to_go_work_bytes()
 * bytes of device memory, 4-byte aligned, owned by the caller (nothing is allocated).
 * RK_ERR_ARG, checked before any device call: map NULL or failing rk_plan_rollout_map's map checks (w_map is ignored);
 * spec NULL; a step not finite or <= 0; k_cost negative, NaN or inf; lethal NaN or <= 0; n_fields, fw or fh < 1; fw or
 * fh > 2^24; n_fields*fh*fw >= 2^31; d_goal, d_field or d_work NULL; a misaligned table. */
int rk_plan_cost_to_go(const rk_plan_map_t *map, const rk_plan_ctg_t *spec, const float *d_goal, const int32_t *d_field_map,
                       const int32_t *d_offset, int32_t n_fields, int32_t fw, int32_t fh, float *d_field, void *d_work,
                       int32_t *rounds_out, void *stream);
/* Bytes of d_work for rk_plan_cost_to_go; 0 for sizes it rejects. */
size_t rk_plan_cost_to_go_work_bytes(int32_t n_fields, int32_t fw, int32_t fh);

typedef struct rk_plan_field {
  const float   *d_field;    /* float [n_fields][fh][fw] (rk_plan_cost_to_go's, or any caller's grid); 4-byte aligned */
  const int32_t *d_field_of; /* int32 [R]: the field of robot r; NULL: field 0 for every robot */
  const int32_t *d_offset;   /* int2 [n_fields]: the grid cell of window cell (0, 0); NULL: (0, 0); 8-byte aligned */
  int32_t n_fields, fw, fh;  /* >= 1 each; n_fields*fh*fw < 2^31; fw, fh <= 2^24 */
  float   x0, y0, inv_res;   /* the map's grid: the outer corner of grid cell (0, 0), cells per metre; finite, inv_res > 0 */
  float   outside;           /* the value off the window; may be +inf; NaN rejected */
  float   w_field;           /* finite, >= 0 */
} rk_plan_field_t;           /* 56 bytes */

/* rk_plan_rollout_map plus a terminal cost-to-go term, read at the state after the last tick (after the last checkpoint's
 * map term), into the same O.  One IEEE float32 operation each, in the written order:
 *   f = d_field_of ? d_field_of[r] : 0;     f < 0 or f >= n_fields: no term for robot r
 *   u = (x - x0) * inv_res;  v = (y - y0) * inv_res;  (ox, oy) = d_offset ? d_offset[f] : (0, 0)
 *   c = field cell ((int)floorf(u) - ox, (int)floorf(v) - oy) of field f if (u, v) lies in the window by the comparisons
 *       of rk_plan_cost_to_go's goal cell (the same 2^24 rule), else outside
 *   if (c > 0) O = O + w_field * c;         d_cost = J + O
 * With ox, oy >= 0 this is the cell plan_map reads for the same map grid.  A blocked or unreachable cell (+inf) prices
 * the candidate at +inf; a NaN cell adds nothing.  map may be NULL (no map term).  field == NULL or w_field == 0 is
 * rk_plan_rollout_map (the same kernel and bits).
 * RK_ERR_ARG: rk_plan_rollout_map's checks; n_fields, fw or fh < 1, fw or fh > 2^24, n_fields*fh*fw >= 2^31; x0, y0 or
 * inv_res not finite, inv_res <= 0; outside NaN; w_field negative, NaN or inf; d_field NULL, or a misaligned table.
 * R == 0 is a no-op. */
int rk_plan_rollout_field(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S,
                          const rk_vdt_cmd_t *d_cmd, int32_t n_seg, int32_t seg_len, const rk_plan_cost_t *cost,
                          const rk_plan_obstacles_t *obst, const rk_plan_map_t *map, const rk_plan_field_t *field,
                          float *d_path, float *d_cost, void *stream);

/* Cost-map inflation: every cell priced by its Euclidean distance to the nearest obstacle of its map, through a table the
 * caller fills (a ROS-style inflation profile, planner.inflation_table), so that robots keep their body clear of walls.
 * The maps and fields above treat the robot as a point; an inflated map is what they should read.  Meant to run when the
 * map changes, not every step. */
typedef struct rk_plan_inflate {
  const float *d_table;  /* float [n_table]: the cost at squared cell distance d2 = 0 .. n_table-1; 4-byte aligned */
  int32_t      n_table;  /* 1 .. 65536 (so only obstacles within 255 cells matter) */
  float        lethal;   /* a cell c >= lethal is an obstacle; > 0, may be +inf; NaN rejected */
} rk_plan_inflate_t;     /* 16 bytes */

/* d_dst: float [n_maps][height][width], the inflated cells of `map` (d_cells; map_of, x0, y0, inv_res and w_map are not
 * used, but x0, y0, inv_res and outside pass rk_plan_rollout_map's map checks).  Every step is integer, or a comparison of
 * float32 values, so the output has one right answer:
 *   obstacle  a cell of map k with c >= lethal (NaN never); the cells off the grid are obstacles exactly when
 *             map->outside >= lethal (the rule rk_plan_cost_to_go uses off the map)
 *   distance  d2(q) = the least (qx - ox)^2 + (qy - oy)^2 over the obstacles o of the same map, exact in integers (maps do
 *             not see each other's obstacles), "none" without an obstacle.  The nearest off-grid obstacle is always the
 *             axial one: min((x+1)^2, (W-x)^2, (y+1)^2, (H-y)^2).
 *   output    with c the source cell: if d2 < n_table, v = d_table[d2] and out = (v > c || c != c) ? v : c; otherwise
 *             out = c.  So the larger value wins, a NaN source cell takes the table's value, and signed zeros keep the
 *             source's bits.
 * The call is asynchronous on `stream` (no host read, no synchronise).  d_work: rk_plan_inflate_work_bytes() bytes of device
 * memory, 4-byte aligned, owned by the caller.  d_dst and d_work must not overlap each other, the cells or the table.
 * RK_ERR_ARG, checked before any device call: map or spec NULL; the map checks of rk_plan_cost_to_go; n_table outside
 * [1, 65536]; lethal NaN or <= 0; d_table, d_dst or d_work NULL or not 4-byte aligned; an overlap. */
int rk_plan_inflate(const rk_plan_map_t *map, const rk_plan_inflate_t *spec, float *d_dst, void *d_work, void *stream);
/* Bytes of d_work for rk_plan_inflate; 0 for sizes it rejects. */
size_t rk_plan_inflate_work_bytes(int32_t n_maps, int32_t width, int32_t height);

/* =====================================================================================
 * RobotManager guard (SURVEY 8f-2): the vehicle-management block of RMT's routine_ros()
 * (src/RobotManager/RM_task_main.cpp:484-767), one call = K manager cycles of n robots.  Per
 * cycle: at most one ROS message is delivered through the callback the firmware runs for it
 * (sb_mecanumCmd_callback :206-218, sb_mecanumContOdr_callback :220-233, sb_mecanumCmdVel_callback
 * :235-248, sb_cmd_callback :159-204), the floor / wall sensors are read (FDT::get_now_FDinfo), and
 * the block decides what VDT receives: the command as it is, a wall-leave move (:546-577), a floor
 * veto -- MOVE_STOP for direction commands (:581-673), zeroed translation for continuous commands
 * by the sector the table arctangent UTIL::mymath::atan2f (src/Utility/util_mymath.cpp:98-126) puts
 * the heading in (:674-749) -- or the 200-cycle no-command watchdog stop (:752-767).  The output
 * record is the RK_CMD_MSG_* vocabulary rk_vdt_rollout's command layer takes (kind 0: nothing sent),
 * so guarded rollouts chain the two calls.  u32_time_ms travels in kind >> 8 (24 bits).
 * ===================================================================================== */
typedef struct rk_rmt_params {
  uint32_t no_cmd_stop_thre;      /* U32_MCN_NO_CMD_STOP_THRE       :62 */
  uint32_t wall_leave_time_ms;    /* U32_MCN_WALL_LEAVE_TIME_MS     :63 */
  uint32_t wall_leave_speed_mmps; /* U32_MCN_WALL_LEAVE_SPEED_MMPS  :64 */
} rk_rmt_params_t;
void rk_rmt_default_params(rk_rmt_params_t *p);

/* manager state per robot: one plane */
enum {
  RK_RS_CMD_STATUS   = 0, /* NOW_CMD_STATUS (CmdStatus :45-59; RELAX = 0 at power-on) */
  RK_RS_IGNORE_FLOOR = 1, /* IS_IGNORE_FLOOR_DETECTION */
  RK_RS_NO_CMD_CNT   = 2, /* U32_MCN_NO_CMD_CNT */
  RK_RS_ABORT        = 3, /* vdt_abort.val (VDT_REQ_ABORT :70-92): wall_abort x+/x-/y+/y- bits 0-3, fllr_abort
                             x+/x-/y+/y- bits 8-11, fllr_abort_vdt_cont_trans_dir bit 16 */
  RK_RS_WORDS        = 4
};
/* input record per robot per cycle: three 128-bit cells, cell c of cycle u, robot i at (u*3 + c)*n + i */
enum {
  RK_ROS_NONE = 0,
  RK_ROS_MECANUM_CMD  = 1, /* interfaces/MecanumCommand {cmd, time, speed}: words A, B, C */
  RK_ROS_MECANUM_CONT = 2, /* interfaces/MecanumContOrder {Twist speed, time_ms}: doubles X, Y, Z (linear.x, linear.y
                              in mm/s, angular.z), time_ms in word A */
  RK_ROS_CMD_VEL      = 3, /* geometry_msgs/Twist on cmd_vel: doubles X, Y (m/s, scaled x1000.0 in double), Z; 500 ms */
  RK_ROS_COMMAND      = 4  /* interfaces/Command {command}: word A */
};
enum {
  RK_RI_KIND = 0, RK_RI_A = 1, RK_RI_B = 2, RK_RI_C = 3,
  RK_RI_X = 4, RK_RI_Y = 6, RK_RI_Z = 8, /* IEEE doubles, low word first */
  RK_RI_FLOOR = 10, /* FDT::Info_FloorDetect (FD_task_main.hpp:24-33) as bytes from the low byte of word 10 up:
                       rForward, lForward, rBack, lBack, right, left, forward, back; 0 none, 1 floor, 2 wall */
  RK_RI_WORDS = 12
};
size_t rk_rmt_state_words(void);
size_t rk_rmt_state_bytes(int64_t n);
/* d_cmd_out: [K][n] rk_vdt_cmd_t (the message VDT::send_req_msg got this cycle, kind 0 if none);
 * d_abort_out: [K][n] vdt_abort.val after the cycle (VehicleInfo.fault, :828) or NULL */
int rk_rmt_guard(const rk_rmt_params_t *p, void *d_state, int64_t n, int32_t K, const void *d_in, rk_vdt_cmd_t *d_cmd_out,
                 uint32_t *d_abort_out, void *stream);
/* single-instance handle (drop-in for the manager's file-static state, RM_task_main.cpp:61-92): one routine_ros()
 * vehicle-management block per call, record in / message out on the host */
typedef struct rk_rmt rk_rmt_t;
int  rk_rmt_create(rk_rmt_t **out, const rk_rmt_params_t *p /* NULL = defaults */);
void rk_rmt_destroy(rk_rmt_t *h);
int  rk_rmt_cycle(rk_rmt_t *h, const uint32_t in[RK_RI_WORDS], rk_vdt_cmd_t *out, uint32_t *abort_val);
int  rk_rmt_get_state(rk_rmt_t *h, uint32_t words[RK_RS_WORDS]);

/* UTIL::mymath::atan2f on device arrays (the guard's sector test uses it; exposed for parity tests) */
int rk_mymath_atan2f(const float *d_y, const float *d_x, float *d_out, int64_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ROBOTICK_H_ */
