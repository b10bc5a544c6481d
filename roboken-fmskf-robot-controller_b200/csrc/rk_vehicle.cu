// rk_vehicle.cu -- vehicle kernels + their C-ABI entry points (include/robotick.h).
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>

#include "rk_vehicle_fast2.cuh"

namespace rk {

// -----------------------------------------------------------------------------------------
// Fused rollout: K ticks of VEHICLE_CTRL::update() per launch, one thread per robot, state
// loaded once with 128-bit loads, held in registers for all K ticks, stored once.
// MODE = RK_SENSOR_* ; TRACE writes the per-tick record (tests only).
// -----------------------------------------------------------------------------------------
constexpr int kRolloutThreads = 128;

// The yaw the ISR hands to set_now_yaw_world() (VD_task_main.cpp:368) before tick y * yaw_period, from one of three
// sources: the float stream d_yaw; the WT901C Yaw register stream d_yaw_reg; or the IMU's own register snapshots
// d_imu_regs (the cells rk_imt_update consumes) -- then the vehicle forms what IMT::get_status_now_yaw() would
// return after IMU update y without waiting for the IMU kernel:
//   angle[2] = reg / 32768.0f * 180.0f (IMU_IF_WT901C::updateData, imu_if_wt901c.cpp:100; /2^15 is exact) ->
//   getYawDate() (:160) -> mymath::deg2rad (util_mymath.hpp:16);
//   an update without a quaternion frame (d_imu_have_quat == 0) leaves the IMU's Data page as it was
//   (imu_if_wt901c.cpp:83-89), i.e. the yaw of the last good update -- before the first one of this launch that is
//   the Data page the IMU block held at launch (d_imu_yaw0_deg).
struct YawPf {
  uint32_t raw;  // float bits, or the sign-extended register
  uint32_t have; // 0: hold
};
RK_DEV YawPf load_yaw_pf(const rk_vdt_rollout_t &a, int64_t n, int64_t i, int yk) { // the loads only: nothing here waits for them
  YawPf         pf;
  const int64_t idx = (int64_t)yk * n + i;
  pf.have           = 1u;
  if(a.d_yaw) {
    pf.raw = __float_as_uint(__ldcs(a.d_yaw + idx));
  } else if(a.d_yaw_reg) {
    pf.raw = (uint32_t)(int)__ldcs(a.d_yaw_reg + idx);
    if(a.d_imu_have_quat) pf.have = (uint32_t)__ldcs(a.d_imu_have_quat + idx);
  } else {
    pf.raw = (uint32_t)(int)__ldcs(a.d_imu_regs + (((int64_t)yk * 2 + 1) * n + i) * 8 + (RK_IMT_REG_YAW - 8));
    if(a.d_imu_have_quat) pf.have = (uint32_t)__ldcs(a.d_imu_have_quat + idx);
  }
  return pf;
}
RK_DEV float yaw_of_reg(int32_t reg) { return fmul(fmul(fmul((float)reg, 1.0f / 32768.0f), 180.0f), RK_DEG2RAD); }
// false: the yaw word stays as it is
RK_DEV bool yaw_of_pf(const rk_vdt_rollout_t &a, const YawPf &pf, int yk, int64_t i, float &pth) {
  if(a.d_yaw) {
    pth = __uint_as_float(pf.raw);
    return true;
  }
  if(pf.have) {
    pth = yaw_of_reg((int32_t)pf.raw);
    return true;
  }
  if(yk == 0 && a.d_imu_yaw0_deg) {
    pth = fmul(__ldcs(a.d_imu_yaw0_deg + i), RK_DEG2RAD);
    return true;
  }
  return false;
}
RK_DEV bool yaw_enabled(const rk_vdt_rollout_t &a) {
  return (a.d_yaw != nullptr || a.d_yaw_reg != nullptr || a.d_imu_regs != nullptr) && a.yaw_period > 0 && a.n_yaw > 0;
}

// CAN_CTRL::tx_routine (VD_can_controller.hpp:43-55): half of the C610 current frame (id 0x200) -- two s16 currents,
// big-endian, wire order from the low byte of the word
RK_DEV uint32_t c610_tx_word(int32_t cur_a, int32_t cur_b) { return __byte_perm((uint32_t)cur_a, (uint32_t)cur_b, 0x4501); }

// rk_plan_rollout: the PLAN instantiations of the rollout kernels run candidate i = r * S + j of n = R * S from robot
// r's block of the source (pitch R, read only), form the stage cost at every segment end and store nothing else.
struct PlanArgs {
  int64_t       R;
  int32_t       S;
  const float2 *ref; // [n_seg][R], metres
  float         w_pos, w_goal, w_cur;
  float        *cost; // [R * S]
};
// J after the end of segment s (rk_plan_cost_t): the state is that after tick (s + 1) * seg_len - 1
RK_DEV float plan_stage_cost(float J, const Veh &v, const PlanArgs &pl, int s, int n_seg, int64_t r) {
  const float2 g = __ldg(pl.ref + (int64_t)s * pl.R + r);
  const float  dx = fsub(v.pos[0], g.x), dy = fsub(v.pos[1], g.y);
  const float  e = fadd(fmul(dx, dx), fmul(dy, dy));
  float        c[4];
#pragma unroll
  for(int k = 0; k < 4; k++) c[k] = (float)v.m[k].cur_tgt;
  const float q = fadd(fadd(fadd(fmul(c[0], c[0]), fmul(c[1], c[1])), fmul(c[2], c[2])), fmul(c[3], c[3]));
  return fadd(fadd(J, fmul(s < n_seg - 1 ? pl.w_pos : pl.w_goal, e)), fmul(pl.w_cur, q));
}
// rk_plan_rollout_obstacles: the keep-out discs on top of PlanArgs (the OBST instantiations; the others keep PlanArgs
// itself, so their parameter block is unchanged)
struct PlanObstArgs : PlanArgs {
  const float4 *obs; // [m][R]: {cx, cy, radius, -}, metres
  int32_t       m, P;
  float         w_obst;
};
template <bool OBST>
using PlanArgsOf = std::conditional_t<OBST, PlanObstArgs, PlanArgs>;
// O after the checkpoint at position (x, y) (rk_plan_obstacles_t).  The S candidates of robot r read the same m cells
// (one broadcast per warp); the discs are not staged in registers, the packed kernel has none to spare.  r fits 32 bits
// (2^32 robots would take 1.9 TB of state), which keeps one register fewer live across the hot loop.
RK_DEV float plan_obst_cost(float O, float x, float y, const PlanObstArgs &pl, uint32_t r) {
  const float4 *q = pl.obs + r;
#pragma unroll 1
  for(int k = 0; k < pl.m; k++, q += pl.R) {
    const float4 c   = __ldg(q);
    const float  dx  = fsub(x, c.x), dy = fsub(y, c.y);
    const float  pen = fsub(fmul(c.z, c.z), fadd(fmul(dx, dx), fmul(dy, dy)));
    if(pen > 0.0f) O = fadd(O, fmul(pl.w_obst, pen));
  }
  return O;
}

// The start state of thread i: under PLAN, candidate i = r * S + j starts from robot r's block (the S candidates of robot
// r read the same cells: one broadcast per warp).  Returns r (0 without PLAN).
template <bool PLAN>
RK_DEV int64_t rollout_load(const uint4 *state, int64_t n, int64_t i, const PlanArgs &pl, Veh &v) {
  if constexpr(PLAN) {
    const int64_t r = i / pl.S;
    load_veh(state, pl.R, r, v);
    return r;
  }
  load_veh(state, n, i, v);
  return 0;
}
// The end of a launch.  PLAN: the candidate's cost J (+ O after the last obstacle checkpoint, t = K: seg_len % P == 0);
// the end state is discarded, 448 B per candidate not written.  Otherwise the end state, and its squared distance to the
// goal if asked.
template <bool PLAN, bool OBST>
RK_DEV void rollout_store(uint4 *state, int64_t n, int64_t i, const rk_vdt_rollout_t &a, const PlanArgsOf<OBST> &pl, const Veh &v,
                          float J, float O, int64_t r) {
  if constexpr(OBST) {
    pl.cost[i] = fadd(plan_stage_cost(J, v, pl, a.n_seg - 1, a.n_seg, r), plan_obst_cost(O, v.pos[0], v.pos[1], pl, r));
  } else if constexpr(PLAN) {
    pl.cost[i] = plan_stage_cost(J, v, pl, a.n_seg - 1, a.n_seg, r);
  } else {
    store_veh(state, n, i, v);
    if(a.d_cost != nullptr && a.d_goal != nullptr) {
      const float2 g  = reinterpret_cast<const float2 *>(a.d_goal)[i];
      const float  dx = fsub(v.pos[0], g.x), dy = fsub(v.pos[1], g.y);
      a.d_cost[i]     = fadd(fmul(dx, dx), fmul(dy, dy));
    }
  }
}

template <bool TRACE>
RK_DEV void trace_row(uint32_t *d_trace, int64_t n, int64_t i, int t, float px, float py, float pth, const float vel[3],
                      const float tgt[3], int c0, int c1, int c2, int c3, uint32_t cnt) {
  if(!TRACE) return;
  uint32_t *tr = d_trace + (int64_t)t * RK_VDT_TRACE_WORDS * n + i;
  tr[0] = f2u(px), tr[n] = f2u(py), tr[2 * n] = f2u(pth);
#pragma unroll
  for(int j = 0; j < 3; j++) tr[(int64_t)(3 + j) * n] = f2u(vel[j]), tr[(int64_t)(6 + j) * n] = f2u(tgt[j]);
  tr[9 * n] = (uint32_t)c0, tr[10 * n] = (uint32_t)c1, tr[11 * n] = (uint32_t)c2, tr[12 * n] = (uint32_t)c3;
  tr[13 * n] = cnt, tr[14 * n] = c610_tx_word(c0, c1), tr[15 * n] = c610_tx_word(c2, c3);
}

template <int MODE, bool TRACE, bool PLAN = false, bool OBST = false>
__global__ void __launch_bounds__(kRolloutThreads)
vdt_rollout_kernel(const rk_vdt_params_t p, uint4 *__restrict__ state, int64_t n, const rk_vdt_rollout_t a, const PlanArgsOf<OBST> pl) {
  static_assert(PLAN || !OBST, "obstacles are a plan-rollout term");
  __shared__ float s_tab[513];
  stage_sin_table(s_tab);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;

  Veh           v;
  const int64_t r = rollout_load<PLAN>(state, n, i, pl, v);
  float         J = 0.0f;
  const Derived d = derive(p);
  float         cth, sth;
  yaw_trig(s_tab, v.pos[2], cth, sth);

  int   next_yaw = yaw_enabled(a) ? 0 : INT_MAX, yk = 0;
  Sched sc;
  sched_init(sc, a);

  // RK_SENSOR_STREAM: the four frames of tick t + 1 are in flight while tick t is computed
  const unsigned long long *fsrc = reinterpret_cast<const unsigned long long *>(a.d_frames) + i;
  uint64_t                  fpf[4] = {0, 0, 0, 0};
  if(MODE == RK_SENSOR_STREAM && a.steps > 0) {
#pragma unroll
    for(int k = 0; k < 4; k++) fpf[k] = __ldcs(fsrc + (int64_t)k * n);
  }

  float O = 0.0f;
  int   next_chk = 0;
  if constexpr(OBST) next_chk = pl.P;
  for(int t = 0; t < a.steps; t++) {
    if constexpr(PLAN)
      if(t == sc.next_cmd && sc.seg > 0) J = plan_stage_cost(J, v, pl, sc.seg - 1, a.n_seg, r);
    if constexpr(OBST)
      if(t == next_chk) { // the state after tick t - 1
        O = plan_obst_cost(O, v.pos[0], v.pos[1], pl, r);
        next_chk += pl.P;
      }
    sched_events(v, p, a, n, i, t, sc);
    if(t == next_yaw) { // can_tx_routine_intr -> set_now_yaw_world()   VD_task_main.cpp:368
      if(yaw_of_pf(a, load_yaw_pf(a, n, i, yk), yk, i, v.pos[2])) yaw_trig(s_tab, v.pos[2], cth, sth);
      yk++;
      next_yaw = (yk < a.n_yaw) ? next_yaw + a.yaw_period : INT_MAX;
    }
    if(MODE != RK_SENSOR_HOLD) {
      const int32_t us = ((t + 1) * 1000) & 0x7FFF;
      uint64_t      fr[4];
#pragma unroll
      for(int k = 0; k < 4; k++) fr[k] = (MODE == RK_SENSOR_PLANT) ? plant_frame(v.m[k]) : fpf[k];
      if(MODE == RK_SENSOR_STREAM && t + 1 < a.steps) {
#pragma unroll
        for(int k = 0; k < 4; k++) fpf[k] = __ldcs(fsrc + ((int64_t)(t + 1) * 4 + k) * n);
      }
#pragma unroll
      for(int k = 0; k < 4; k++) motor_rx(v.m[k], p.motor_dir[k], fr[k], us);
    }
    veh_update(v, p, d, cth, sth);
    trace_row<TRACE>(a.d_trace, n, i, t, v.pos[0], v.pos[1], v.pos[2], v.vel, v.tgt, v.m[0].cur_tgt, v.m[1].cur_tgt,
                     v.m[2].cur_tgt, v.m[3].cur_tgt, (a.task_period > 0) ? v.move_cnt : 0u);
  }
  rollout_store<PLAN, OBST>(state, n, i, a, pl, v, J, O, r);
}

// -----------------------------------------------------------------------------------------
// Closed-loop rollout, issue-optimised (rk_vehicle_fast.cuh / rk_vehicle_fast2.cuh).  Ticks between two
// command boundaries ("chunks") run on the fast tick when the thread's state satisfies fast_ok() and the
// chunk's constants bound the controller output (fast_u_bounded); command application, the last tick of
// the launch and any thread outside the fast path's domain run the transcription (veh_update), so the
// stored state is complete and identical.
// -----------------------------------------------------------------------------------------
constexpr int kFastThreads = 128;
constexpr int kFastUnroll  = 2;
constexpr int kMaxChunk    = 2048; // ticks per chunk: keeps the per-chunk angle sum exact (int32, or integers in float: |step| <= 4474)

RK_DEV void fast_consts(FastConsts &fc, const rk_vdt_params_t &p, const Derived &d) {
  fc.rcp_r = fdiv(1.0f, p.wheel_radius_mm), fc.rcp_s2 = fdiv(1.0f, p.sqrtf2), fc.rcp_l = fdiv(1.0f, p.wheel_l_mm);
  const double K = (double)RK_OUT_RAD_PER_RAW_ANGLE * (double)RK_GEAR_RATIO_INV;
  fc.k_hi        = __double2float_rn(K);
  fc.k_lo        = __double2float_rn(K - (double)fc.k_hi);
  fc.A1 = d.A1, fc.B0 = d.B0, fc.ki_dt = d.ki_dt, fc.s2l = d.s2l;
  fc.neg_i_limit = -p.i_limit, fc.neg_ff_limit = -p.ff_limit;
  fc.khi_pm = make_float2(fc.k_hi, -fc.k_hi), fc.klo_pm = make_float2(fc.k_lo, -fc.k_lo);
  asm volatile("" : "+f"(fc.khi_pm.x), "+f"(fc.khi_pm.y), "+f"(fc.klo_pm.x), "+f"(fc.klo_pm.y)); // not rematerialised per tick
}

// The yaw sample for the next boundary is fetched one period ahead, so its HBM latency hides behind
// yaw_period ticks of arithmetic instead of stalling every warp at once.
struct YawFeed {
  int   next, yk;
  YawPf pf;
};
RK_DEV void yaw_feed_init(YawFeed &y, const rk_vdt_rollout_t &a, int64_t n, int64_t i) {
  y.next = yaw_enabled(a) ? 0 : INT_MAX, y.yk = 0;
  y.pf.raw = 0u, y.pf.have = 0u;
  if(y.next == 0) y.pf = load_yaw_pf(a, n, i, 0);
}
// can_tx_routine_intr -> set_now_yaw_world()   VD_task_main.cpp:368
RK_DEV void yaw_feed_take(YawFeed &y, const rk_vdt_rollout_t &a, int64_t n, int64_t i, const float *s_tab, float &pth, float &cth,
                          float &sth) {
  if(yaw_of_pf(a, y.pf, y.yk, i, pth)) yaw_trig(s_tab, pth, cth, sth);
  y.yk++;
  if(y.yk < a.n_yaw) {
    y.next += a.yaw_period;
    y.pf = load_yaw_pf(a, n, i, y.yk);
  } else {
    y.next = INT_MAX;
  }
}

// The cold branch of vdt_rollout_fast_kernel at t == yf.next.  OBST: the obstacle checkpoint at (x, y), the state after
// tick t - 1; returns O with it added.  Otherwise the yaw boundary into (pth, cth, sth); returns O as it was.  (O by
// value: taken by reference, it changes ptxas' register assignment in the OBST kernels.)
template <bool OBST>
RK_DEV float yaw_boundary(YawFeed &yf, float O, float x, float y, const PlanArgsOf<OBST> &pl, int64_t r, const rk_vdt_rollout_t &a,
                          int64_t n, int64_t i, const float *s_tab, float &pth, float &cth, float &sth) {
  if constexpr(OBST) {
    O = plan_obst_cost(O, x, y, pl, r);
    yf.next += pl.P;
  } else {
    yaw_feed_take(yf, a, n, i, s_tab, pth, cth, sth);
  }
  return O;
}
// FLAGS: bit 0 FFSAT (ff_limit == 1: FMUL.SAT form of the feed-forward clamp), bit 1 KD0 (kd == 0, packed tick only)
// PLAN: rk_plan_rollout (PlanArgs); segment ends are command ticks, so they are chunk boundaries and the stage cost is
// formed outside the chunk loop.
// OBST (with PLAN): rk_plan_rollout_obstacles (PlanObstArgs).  Plan rollouts have no yaw stream, so the yaw boundary's
// cold branch inside the chunk loop takes the obstacle checkpoint instead (every P ticks, the same tick in every lane):
// no new chunk boundary and no new loop-carried register besides O.
template <bool TRACE, int OCC, int FLAGS, bool PACKED, bool RESET = false, bool PLAN = false, bool OBST = false>
__global__ void __launch_bounds__(kFastThreads, OCC * 128 / kFastThreads)
vdt_rollout_fast_kernel(const rk_vdt_params_t p, uint4 *__restrict__ state, int64_t n, const rk_vdt_rollout_t a, const CmdRcp rcp,
                        const PlanArgsOf<OBST> pl) {
  static_assert(PLAN || !OBST, "obstacles are a plan-rollout term");
  constexpr int  D0 = 1, D1 = 1, D2 = -1, D3 = -1; // VD_task_main.cpp:75-78 (host checks params match)
  constexpr bool FFSAT = (FLAGS & 1) != 0, KD0 = (FLAGS & 2) != 0;
  __shared__ float s_tab[513];
  stage_sin_table(s_tab);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;

  Veh     v;
  int64_t r = 0;
  float   J = 0.0f;
  if(RESET) v = Veh{}; // reset_state: the power-on block is all zeros -- nothing to load (and no memset in front of the kernel)
  else r = rollout_load<PLAN>(state, n, i, pl, v);
  const Derived d = derive(p);
  FastConsts    fc;
  fast_consts(fc, p, d);
  float cth, sth;
  yaw_trig(s_tab, v.pos[2], cth, sth);

  const int K = a.steps;
  Sched     sch;
  sched_init(sch, a);
  YawFeed yf;
  float   O = 0.0f;
  if constexpr(OBST) yf.next = pl.P; // the next checkpoint: the state after tick yf.next - 1
  else yaw_feed_init(yf, a, n, i);

  int t = 0;
  while(t < K) {
    if constexpr(PLAN)
      if(t == sch.next_cmd && sch.seg > 0) J = plan_stage_cost(J, v, pl, sch.seg - 1, a.n_seg, r);
    sched_events(v, p, a, n, i, t, sch, &rcp); // commands, VDT::main messages and the move-time countdown due at this tick
    // run to the next event: a command, the countdown's automatic stop, or the last tick of the launch
    // (always a transcription tick).  Lanes of a warp whose countdowns fire at different ticks leave
    // the fast loop at different times; results do not depend on it.
    const int t_end = min(min(min(sch.next_cmd, sched_fire_tick(v, a, sch)), K - 1), t + kMaxChunk);
    if(t < t_end && fast_ok<D0, D1, D2, D3>(v, p) && fast_u_bounded<false>(v, p, fc) &&
       !(PACKED && (f2u(v.pos[0]) == 0x80000000u || f2u(v.pos[1]) == 0x80000000u))) {
      const int t0  = t;
      float     pth = v.pos[2];
      if(PACKED) { // FADD2 / FFMA2 form of the same tick (rk_vehicle_fast2.cuh)
        FastVeh2 f;
        to_fast2(v, f, p.ts, fc.B0);
        const float nz = fmul(-0.0f, p.ts); // opaque -0.0f (p.ts > 0 is a fast-path precondition)
        // ONE loop over the chunk; the yaw boundary (every yaw_period ticks, the same tick in every lane) is a cold
        // branch inside it, so the tick's loop-carried registers stay where they are across boundaries
        float2 cs = make_float2(cth, sth), sc = make_float2(sth, cth);
#pragma unroll kFastUnroll
        for(; t < t_end; t++) {
          if(t == yf.next) {
            O = yaw_boundary<OBST>(yf, O, f.p.x, f.p.y, pl, r, a, n, i, s_tab, pth, cth, sth);
            if constexpr(!OBST) cs = make_float2(cth, sth), sc = make_float2(sth, cth);
          }
          float vel[3], tgt[3];
          fast_tick2<FFSAT, TRACE, KD0>(f, p, fc, cs, sc, nz, vel, tgt);
          trace_row<TRACE>(a.d_trace, n, i, t, f.p.x, f.p.y, pth, vel, tgt, f.w01.cur[0], f.w01.cur[1], f.w23.cur[0], f.w23.cur[1],
                           TRACE ? sched_cnt_at(v.move_cnt, a, sch, t) : 0u);
        }
        v.pos[2] = pth;
        from_fast2<D0, D1, D2, D3>(v, f, t - t0);
        sched_skip_to(v, a, sch, t);
      } else {
        FastVeh f;
        to_fast<D0, D1, D2, D3>(v, f, p.ts, fc.B0);
#pragma unroll kFastUnroll
        for(; t < t_end; t++) {
          if(t == yf.next) O = yaw_boundary<OBST>(yf, O, f.px, f.py, pl, r, a, n, i, s_tab, pth, cth, sth);
          float vel[3], tgt[3];
          fast_tick<D0, D1, D2, D3, FFSAT>(f, p, fc, cth, sth, vel, tgt);
          trace_row<TRACE>(a.d_trace, n, i, t, f.px, f.py, pth, vel, tgt, f.w[0].cur, f.w[1].cur, f.w[2].cur, f.w[3].cur,
                           TRACE ? sched_cnt_at(v.move_cnt, a, sch, t) : 0u);
        }
        v.pos[2] = pth;
        from_fast<D0, D1, D2, D3>(v, f, t - t0);
        sched_skip_to(v, a, sch, t);
      }
    } else {
      if(t == yf.next) O = yaw_boundary<OBST>(yf, O, v.pos[0], v.pos[1], pl, r, a, n, i, s_tab, v.pos[2], cth, sth);
      const int32_t us = ((t + 1) * 1000) & 0x7FFF;
#pragma unroll
      for(int k = 0; k < 4; k++) motor_rx(v.m[k], p.motor_dir[k], plant_frame(v.m[k]), us);
      veh_update(v, p, d, cth, sth);
      trace_row<TRACE>(a.d_trace, n, i, t, v.pos[0], v.pos[1], v.pos[2], v.vel, v.tgt, v.m[0].cur_tgt, v.m[1].cur_tgt,
                       v.m[2].cur_tgt, v.m[3].cur_tgt, (a.task_period > 0) ? v.move_cnt : 0u);
      t++;
    }
  }
  rollout_store<PLAN, OBST>(state, n, i, a, pl, v, J, O, r);
}

// -----------------------------------------------------------------------------------------
// RK_SENSOR_STREAM on the packed fast tick: the same chunk structure as vdt_rollout_fast_kernel, the wheel
// feedback decoded from the recorded frames (fast_tick2_stream); the four frames of tick t + 1 are in flight
// while tick t is computed.  Command ticks, the last tick and threads outside the fast domain run the
// transcription on the same frames.
// -----------------------------------------------------------------------------------------
// The recorded frames reach each thread through its own ring in shared memory, filled kStreamRing ticks ahead by
// cp.async (LDGSTS): the HBM latency of a tick's four frames hides behind kStreamRing ticks of arithmetic and costs no
// registers.  Every thread copies and reads only its own slots ([stage][wheel][thread], conflict-free LDS.64), so
// threads of a warp that sit in different chunk paths need no barrier between them.
constexpr int kStreamRing = 4;
struct FrameRing {
  uint32_t                  base; // shared-memory address of this thread's slot (stage 0, wheel 0)
  const unsigned long long *src;  // the thread's column of d_frames
  int64_t                   n;
  int                       K;
};
RK_DEV void frame_ring_issue(const FrameRing &r, int t) { // the four frames of tick t (nothing past the launch); one group per tick
  if(t < r.K) {
#pragma unroll
    for(int k = 0; k < 4; k++) {
      const uint32_t dst = r.base + (uint32_t)(((t & (kStreamRing - 1)) * 4 + k) * (kFastThreads * 8));
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(r.src + ((int64_t)t * 4 + k) * r.n) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}
RK_DEV void frame_ring_take(const FrameRing &r, int t, uint64_t fr[4]) { // groups 0..t have landed once all but the last R-1 have
  asm volatile("cp.async.wait_group %0;" ::"n"(kStreamRing - 1) : "memory");
#pragma unroll
  for(int k = 0; k < 4; k++) {
    const uint32_t src = r.base + (uint32_t)(((t & (kStreamRing - 1)) * 4 + k) * (kFastThreads * 8));
    unsigned long long v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(src) : "memory");
    fr[k] = v;
  }
}
template <bool TRACE, int FLAGS>
__global__ void __launch_bounds__(kFastThreads, 4)
vdt_rollout_stream_fast_kernel(const rk_vdt_params_t p, uint4 *__restrict__ state, int64_t n, const rk_vdt_rollout_t a, const CmdRcp rcp) {
  constexpr int  D0 = 1, D1 = 1, D2 = -1, D3 = -1;
  constexpr bool FFSAT = (FLAGS & 1) != 0, KD0 = (FLAGS & 2) != 0;
  __shared__ float s_tab[513];
  stage_sin_table(s_tab);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;

  Veh v;
  load_veh(state, n, i, v);
  const Derived d = derive(p);
  FastConsts    fc;
  fast_consts(fc, p, d);
  float cth, sth;
  yaw_trig(s_tab, v.pos[2], cth, sth);

  const int K = a.steps;
  Sched     sch;
  sched_init(sch, a);
  YawFeed yf;
  yaw_feed_init(yf, a, n, i);
  __shared__ __align__(16) unsigned long long s_ring[kStreamRing * 4 * kFastThreads];
  FrameRing ring;
  ring.base = (uint32_t)__cvta_generic_to_shared(s_ring + threadIdx.x), ring.n = n, ring.K = a.steps;
  ring.src  = reinterpret_cast<const unsigned long long *>(a.d_frames) + i;
#pragma unroll
  for(int s = 0; s < kStreamRing; s++) frame_ring_issue(ring, s);

  int t = 0;
  while(t < K) {
    sched_events(v, p, a, n, i, t, sch, &rcp);
    // chunks are capped so the 32-bit per-chunk angle sum cannot overflow (|step| <= 40960)
    const int t_end = min(min(min(sch.next_cmd, sched_fire_tick(v, a, sch)), K - 1), t + 32768);
    if(t < t_end && fast_ok<D0, D1, D2, D3, true>(v, p) && fast_u_bounded<true>(v, p, fc)) {
      const int   t0  = t;
      float       pth = v.pos[2];
      FastVeh2    f;
      StreamSense ss;
      to_fast2(v, f, p.ts, fc.B0);
      stream_sense_load(ss, v);
      const float nz = fmul(-0.0f, p.ts);
      float2 cs = make_float2(cth, sth), sc = make_float2(sth, cth);
      {
#pragma unroll 2
        for(; t < t_end; t++) {
          if(t == yf.next) {
            yaw_feed_take(yf, a, n, i, s_tab, pth, cth, sth);
            cs = make_float2(cth, sth), sc = make_float2(sth, cth);
          }
          uint64_t fr[4];
          frame_ring_take(ring, t, fr);
          float vel[3], tgt[3];
          fast_tick2_stream<FFSAT, TRACE, KD0>(f, ss, fr, p, fc, cs, sc, nz, vel, tgt);
          frame_ring_issue(ring, t + kStreamRing); // into the stage just read
          trace_row<TRACE>(a.d_trace, n, i, t, f.p.x, f.p.y, pth, vel, tgt, f.w01.cur[0], f.w01.cur[1], f.w23.cur[0], f.w23.cur[1],
                           TRACE ? sched_cnt_at(v.move_cnt, a, sch, t) : 0u);
        }
      }
      v.pos[2] = pth;
      from_fast2_stream(v, f, ss, t - t0);
      sched_skip_to(v, a, sch, t);
    } else {
      if(t == yf.next) yaw_feed_take(yf, a, n, i, s_tab, v.pos[2], cth, sth);
      const int32_t us = ((t + 1) * 1000) & 0x7FFF;
      uint64_t      fr[4];
      frame_ring_take(ring, t, fr);
#pragma unroll
      for(int k = 0; k < 4; k++) motor_rx(v.m[k], p.motor_dir[k], fr[k], us);
      veh_update(v, p, d, cth, sth);
      frame_ring_issue(ring, t + kStreamRing);
      trace_row<TRACE>(a.d_trace, n, i, t, v.pos[0], v.pos[1], v.pos[2], v.vel, v.tgt, v.m[0].cur_tgt, v.m[1].cur_tgt,
                       v.m[2].cur_tgt, v.m[3].cur_tgt, (a.task_period > 0) ? v.move_cnt : 0u);
      t++;
    }
  }
  rollout_store<false, false>(state, n, i, a, PlanArgs{}, v, 0.0f, 0.0f, 0);
}

// ---- small batched setters ------------------------------------------------------------
__global__ void vdt_set_power_kernel(uint4 *state, int64_t n, const uint8_t *on) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  uint4 q = state[i]; // plane 0
  bool  b = on ? (on[i] != 0) : true;
  q.w     = b ? (q.w | RK_VS_FLAG_POWER_ON) : (q.w & ~RK_VS_FLAG_POWER_ON);
  state[i] = q;
}

__global__ void vdt_set_target_kernel(uint4 *state, int64_t n, const float *v, const float *a, const float *j) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
#pragma unroll
  for(int k = 0; k < 3; k++) {
    Interp t;
    load_interp(state, n, i, k, t);
    interp_set(t, v[(int64_t)k * n + i], a[(int64_t)k * n + i], j[(int64_t)k * n + i]);
    store_interp(state, n, i, k, t);
  }
}

__global__ void vdt_motor_rx_kernel(const rk_vdt_params_t p, uint4 *state, int64_t n, int wheel,
                                    const unsigned long long *frames, const int16_t *usec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  Motor m;
  load_motor(state, n, i, wheel, m);
  motor_rx(m, p.motor_dir[wheel], frames[i], usec ? (int32_t)usec[i] : 0);
  store_motor(state, n, i, wheel, m);
}

// CAN_CTRL::tx_routine for every vehicle: the 8-byte C610 frame from the four s16_rawCurr_tgt of the state block
__global__ void vdt_tx_frames_kernel(const uint4 *state, int64_t n, unsigned long long *frames) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  int32_t c[4];
#pragma unroll
  for(int k = 0; k < 4; k++) c[k] = hi16(ld_plane(state, n, RK_VS_MOTOR0 / 4 + 2 * k + 1, i).y); // RK_VM_CUR_TGT: s16_rawCurr_tgt in the high half
  frames[i] = (unsigned long long)c610_tx_word(c[0], c[1]) | ((unsigned long long)c610_tx_word(c[2], c[3]) << 32);
}

// single-instance pokes used by the handle API (arguments by value, one thread)
__global__ void vdt_poke_word_kernel(uint32_t *state, int64_t idx, uint32_t val) { state[idx] = val; }
__global__ void vdt_set_target1_kernel(uint4 *state, float v0, float v1, float v2, float a0, float a1, float a2,
                                       float j0, float j1, float j2) {
  const float v[3] = {v0, v1, v2}, a[3] = {a0, a1, a2}, j[3] = {j0, j1, j2};
#pragma unroll
  for(int k = 0; k < 3; k++) {
    Interp t;
    load_interp(state, 1, 0, k, t);
    interp_set(t, v[k], a[k], j[k]);
    store_interp(state, 1, 0, k, t);
  }
}
// -----------------------------------------------------------------------------------------
// host side
// -----------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char *what) {
  set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return RK_ERR_CUDA;
}
int require_device() {
  int         cnt = 0;
  cudaError_t e   = cudaGetDeviceCount(&cnt);
  if(e != cudaSuccess || cnt == 0) {
    set_error("no CUDA device (%s): librobotick_b200 has no CPU fallback", cudaGetErrorString(e));
    cudaGetLastError();
    return RK_ERR_CUDA;
  }
  return RK_OK;
}

static int check_block(const void *p, const char *name) {
  if(p == nullptr || ((uintptr_t)p & 15u) != 0) {
    set_error("%s must be a non-NULL 16-byte aligned device pointer", name);
    return RK_ERR_ARG;
  }
  return RK_OK;
}

bool fast_path_proven(const rk_vdt_params_t &p); // rk_exact.cu
static CmdRcp make_cmd_rcp(const rk_vdt_params_t &p) { // the host's IEEE divisions (interp_set_rcp)
  CmdRcp r;
  for(int k = 0; k < 3; k++)
    r.ra_move[k] = 1.0f / p.accel_move[k], r.rj_move[k] = 1.0f / p.jerk_move[k], r.ra_stop[k] = 1.0f / p.accel_stop[k], r.rj_stop[k] = 1.0f / p.jerk_stop[k];
  return r;
}
int  tick_set_side_ctas(int v);                     // rk_tick.cu
int  stream_set_ctas(int v);                        // rk_stream.cu

static int g_fast_occupancy = 4;       // rk_set_option(RK_OPT_FAST_OCCUPANCY, 3|4): tuning
static int g_fast_packed = 1;          // rk_set_option(RK_OPT_FAST_PACKED, 0|1): packed FP32 tick (default) or scalar
static int g_fast_ffsat = 0;           // rk_set_option(RK_OPT_FAST_FFSAT, 0|1): FMUL.SAT form of the feed-forward clamp.  Off since
                                       // round 2: the packed tick is bound by FP32 lanes, the FMNMX form runs on the ALU pipe (8.83 vs 8.94 ms)
static int g_force_transcription = 0; // rk_vdt_set_option(RK_OPT_FORCE_TRANSCRIPTION, 1): tests

// The fast kernel is compiled for the firmware's wiring (directions +,+,-,-) and needs
// positive finite limits / profile tables and proven exact-division constants; anything else
// runs the transcription kernel.
static bool fast_path_usable(const rk_vdt_params_t &p) {
  if(g_force_transcription) return false;
  if(!(p.motor_dir[0] == 1 && p.motor_dir[1] == 1 && p.motor_dir[2] == -1 && p.motor_dir[3] == -1)) return false;
  if(!(p.raw_curr_lim >= 0 && p.raw_curr_lim <= 7000)) return false;
  auto pos = [](float x) { return x > 0.0f && x <= 1.0e9f; };
  auto fin = [](float x) { return x >= -1.0e9f && x <= 1.0e9f; };
  if(!(pos(p.i_limit) && pos(p.ff_limit) && pos(p.ts) && pos(p.ctrl_freq) && pos(p.lpf_freq))) return false;
  if(!(fin(p.kff) && fin(p.kp) && fin(p.ki) && fin(p.kd))) return false;
  for(int k = 0; k < 3; k++)
    if(!(pos(p.accel_move[k]) && pos(p.jerk_move[k]) && pos(p.accel_stop[k]) && pos(p.jerk_stop[k]))) return false;
  return fast_path_proven(p);
}

// The compile-time configuration of one fast-kernel launch, from the params and the RK_OPT_FAST_* options
struct FastCfg {
  bool trace;  // TRACE (compiled at occupancy 4 only)
  int  occ;    // OCC: resident CTAs per SM the kernel is compiled for (register budget), 3 or 4
  int  flags;  // FLAGS: bit 0 FFSAT, bit 1 KD0
  bool packed; // PACKED
};
static FastCfg fast_cfg(const rk_vdt_params_t &p, bool trace, bool stream) {
  FastCfg c;
  c.trace = trace;
  c.occ   = (trace || g_fast_occupancy != 3) ? 4 : 3;
  // KD0 specialises the packed tick only.  The stream kernel has no scalar form, so it is packed (and takes KD0)
  // whatever RK_OPT_FAST_PACKED says.
  c.packed = stream || g_fast_packed;
  c.flags  = ((p.ff_limit == 1.0f && g_fast_ffsat) ? 1 : 0) | ((p.kd == 0.0f && c.packed) ? 2 : 0);
  return c;
}
// Calls f(TRACE, OCC, FLAGS, PACKED) with c's values as std::integral_constants.  Only these combinations are compiled:
// TRACE at occupancy 4, and the scalar tick without KD0.
template <int V>
using Int = std::integral_constant<int, V>;
template <class F>
static void with_fast_cfg(const FastCfg &c, F &&f) {
  const auto flags = [&](auto tr, auto occ) {
    if(!c.packed) {
      if(c.flags & 1) f(tr, occ, Int<1>{}, std::false_type{});
      else f(tr, occ, Int<0>{}, std::false_type{});
      return;
    }
    switch(c.flags) {
    case 3: f(tr, occ, Int<3>{}, std::true_type{}); break;
    case 2: f(tr, occ, Int<2>{}, std::true_type{}); break;
    case 1: f(tr, occ, Int<1>{}, std::true_type{}); break;
    default: f(tr, occ, Int<0>{}, std::true_type{}); break;
    }
  };
  if(c.trace) flags(std::true_type{}, Int<4>{});
  else if(c.occ == 3) flags(std::false_type{}, Int<3>{});
  else flags(std::false_type{}, Int<4>{});
}

} // namespace rk

using namespace rk;

extern "C" {

int         rk_version(void) { return RK_VERSION; }
const char *rk_last_error(void) { return rk::g_err; }

int rk_device_info(int device, int *sm_count, int *sm_clock_khz, size_t *hbm_bytes) {
  if(int rc = require_device()) return rc;
  cudaDeviceProp prop;
  RK_CUDA(cudaGetDeviceProperties(&prop, device));
  if(sm_count) *sm_count = prop.multiProcessorCount;
  if(sm_clock_khz) {
    int khz = 0;
    RK_CUDA(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
    *sm_clock_khz = khz;
  }
  if(hbm_bytes) *hbm_bytes = prop.totalGlobalMem;
  return RK_OK;
}

int rk_set_option(int option, int value) {
  if(option == RK_OPT_FORCE_TRANSCRIPTION) {
    rk::g_force_transcription = value;
    return RK_OK;
  }
  if(option == RK_OPT_FAST_PACKED) {
    rk::g_fast_packed = value != 0;
    return RK_OK;
  }
  if(option == RK_OPT_FAST_OCCUPANCY && (value >= 3 && value <= 4)) {
    rk::g_fast_occupancy = value;
    return RK_OK;
  }
  if(option == RK_OPT_FAST_FFSAT) {
    rk::g_fast_ffsat = value != 0;
    return RK_OK;
  }
  if(option == RK_OPT_STREAM_CTAS && rk::stream_set_ctas(value) == RK_OK) return RK_OK;
  if(option == RK_OPT_TICK_SIDE_CTAS && rk::tick_set_side_ctas(value) == RK_OK) return RK_OK;
  set_error("rk_set_option: unknown option %d / bad value %d", option, value);
  return RK_ERR_ARG;
}

int rk_set_device(int device) {
  if(int rc = require_device()) return rc;
  RK_CUDA(cudaSetDevice(device));
  return RK_OK;
}

void rk_vdt_default_params(rk_vdt_params_t *p) {
  if(!p) return;
  memset(p, 0, sizeof(*p));
  p->wheel_radius_mm = 37.5f;
  p->wheel_l_mm      = 13.08148f;
  p->sqrtf2          = 1.41421356f;
  p->ts              = 1.0f / (float)1000;
  p->ctrl_freq       = (float)100;
  p->kff = 0.0075f, p->kp = 0.02f, p->ki = 0.01f, p->kd = 0.0f;
  p->i_limit  = 0.5f;
  p->lpf_freq = 10.0f;
  p->ff_limit = 1.0f;
  const float am[3] = {1000.0f, 1000.0f, 30.0f}, jm[3] = {10000.0f, 10000.0f, 300.0f};
  const float as[3] = {2000.0f, 2000.0f, 70.0f}, js[3] = {30000.0f, 30000.0f, 1000.0f};
  for(int k = 0; k < 3; k++) p->accel_move[k] = am[k], p->jerk_move[k] = jm[k], p->accel_stop[k] = as[k], p->jerk_stop[k] = js[k];
  p->motor_dir[0] = 1, p->motor_dir[1] = 1, p->motor_dir[2] = -1, p->motor_dir[3] = -1;
  p->raw_curr_lim = 3000;
  p->default_speed_mmps = 200.0f, p->limit_speed_mmps = 400.0f;                    // VD_task_main.cpp:24,26
  p->default_rot_radps = (float)(2.0f * M_PI / 1.0f), p->limit_rot_radps = (float)(6.0f * M_PI / 1.0f); // :25,27 (double expressions)
  p->task_freq_hz = 100; // :22
}

size_t rk_vdt_state_words(void) { return RK_VS_WORDS; }
size_t rk_vdt_state_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_VS_WORDS * 4u; }

int rk_vdt_rollout(const rk_vdt_params_t *p, void *d_state, int64_t n, const rk_vdt_rollout_t *args, void *stream) {
  if(!p || !args) {
    set_error("rk_vdt_rollout: NULL params/args");
    return RK_ERR_ARG;
  }
  if(n == 0 || args->steps == 0) return RK_OK;
  if(n < 0 || args->steps < 0) {
    set_error("rk_vdt_rollout: negative n or steps");
    return RK_ERR_ARG;
  }
  if(int rc = check_block(d_state, "d_state")) return rc;
  if(args->d_cmd && (((uintptr_t)args->d_cmd & 15u) != 0)) {
    set_error("rk_vdt_rollout: d_cmd must be 16-byte aligned");
    return RK_ERR_ARG;
  }
  if(args->sensor_mode == RK_SENSOR_STREAM && (!args->d_frames || ((uintptr_t)args->d_frames & 7u) != 0)) {
    set_error("rk_vdt_rollout: RK_SENSOR_STREAM needs 8-byte aligned d_frames");
    return RK_ERR_ARG;
  }
  if(args->task_period < 0 || (args->task_period > 0 && args->d_cmd && args->seg_len % args->task_period != 0)) {
    set_error("rk_vdt_rollout: task_period must be >= 0 and divide seg_len (messages are taken at task-period boundaries)");
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  cudaStream_t  st    = (cudaStream_t)stream;
  uint4        *state = (uint4 *)d_state;
  const int     mode  = args->sensor_mode;
  const bool    fast  = (mode == RK_SENSOR_PLANT || mode == RK_SENSOR_STREAM) && fast_path_usable(*p);
  const FastCfg c     = fast_cfg(*p, args->d_trace != nullptr, mode == RK_SENSOR_STREAM);
  // reset_state: the power-on block is all zeros (static initialisation).  Done as a memset in front of the kernel: a
  // second load path inside the rollout kernels cost the hot loop 2 % through ptxas' register allocation (8.83 -> 8.99 ms).
  // ... except in the default configuration of the packed fast kernel, which has an instantiation that starts from
  // zeros in registers: no memset, no state load.
  const bool reset_in_kernel = args->reset_state && mode == RK_SENSOR_PLANT && fast && !c.trace && c.occ == 4 && c.flags == 2 && c.packed;
  if(args->reset_state && !reset_in_kernel) RK_CUDA(cudaMemsetAsync(d_state, 0, (size_t)n * RK_VS_WORDS * 4u, st));
  const unsigned grid  = (unsigned)((n + kFastThreads - 1) / kFastThreads);
  const unsigned tgrid = (unsigned)((n + kRolloutThreads - 1) / kRolloutThreads);
  const auto     transcription = [&](auto m) {
    if(c.trace) vdt_rollout_kernel<m, true><<<tgrid, kRolloutThreads, 0, st>>>(*p, state, n, *args, PlanArgs{});
    else vdt_rollout_kernel<m, false><<<tgrid, kRolloutThreads, 0, st>>>(*p, state, n, *args, PlanArgs{});
  };
  switch(mode) {
  case RK_SENSOR_HOLD: transcription(Int<RK_SENSOR_HOLD>{}); break;
  case RK_SENSOR_PLANT:
    if(!fast) transcription(Int<RK_SENSOR_PLANT>{});
    else if(reset_in_kernel)
      vdt_rollout_fast_kernel<false, 4, 2, true, true><<<grid, kFastThreads, 0, st>>>(*p, state, n, *args, make_cmd_rcp(*p), PlanArgs{});
    else
      with_fast_cfg(c, [&](auto tr, auto occ, auto fl, auto pk) {
        vdt_rollout_fast_kernel<tr, occ, fl, pk><<<grid, kFastThreads, 0, st>>>(*p, state, n, *args, make_cmd_rcp(*p), PlanArgs{});
      });
    break;
  case RK_SENSOR_STREAM:
    if(!fast) transcription(Int<RK_SENSOR_STREAM>{});
    else
      with_fast_cfg(c, [&](auto tr, auto, auto fl, auto) {
        vdt_rollout_stream_fast_kernel<tr, fl><<<grid, kFastThreads, 0, st>>>(*p, state, n, *args, make_cmd_rcp(*p));
      });
    break;
  default: set_error("rk_vdt_rollout: bad sensor_mode %d", mode); return RK_ERR_ARG;
  }
  if(cudaError_t e = cudaGetLastError(); e != cudaSuccess) return cuda_fail(e, "vdt_rollout_kernel launch");
  return RK_OK;
}

} // extern "C"
namespace rk {
// rk_plan_rollout's kernel choice: the RK_SENSOR_PLANT dispatch of rk_vdt_rollout without trace and reset
template <bool OBST>
static void launch_plan(const rk_vdt_params_t &p, const void *d_src, int64_t n, const rk_vdt_rollout_t &a, const PlanArgsOf<OBST> &pl,
                        cudaStream_t st) {
  uint4 *src = (uint4 *)d_src; // read only under PLAN
  if(fast_path_usable(p)) {
    const unsigned grid = (unsigned)((n + kFastThreads - 1) / kFastThreads);
    with_fast_cfg(fast_cfg(p, false, false), [&](auto, auto occ, auto fl, auto pk) {
      vdt_rollout_fast_kernel<false, occ, fl, pk, false, true, OBST><<<grid, kFastThreads, 0, st>>>(p, src, n, a, make_cmd_rcp(p), pl);
    });
  } else {
    const unsigned grid = (unsigned)((n + kRolloutThreads - 1) / kRolloutThreads);
    vdt_rollout_kernel<RK_SENSOR_PLANT, false, true, OBST><<<grid, kRolloutThreads, 0, st>>>(p, src, n, a, pl);
  }
}
// rk_plan_rollout (ob == NULL) and rk_plan_rollout_obstacles: the same checks, and without discs the same kernels
static int plan_rollout(const char *who, const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S, const rk_vdt_cmd_t *d_cmd,
                        int32_t n_seg, int32_t seg_len, const rk_plan_cost_t *cost, const rk_plan_obstacles_t *ob, float *d_cost,
                        void *stream) {
  if(!p || !cost) {
    set_error("%s: NULL params/cost", who);
    return RK_ERR_ARG;
  }
  if(R < 0 || S < 1) {
    set_error("%s: need R >= 0 and S >= 1 (R = %lld, S = %d)", who, (long long)R, S);
    return RK_ERR_ARG;
  }
  if(n_seg < 1 || seg_len < 1 || (int64_t)n_seg * seg_len > INT_MAX) {
    set_error("%s: need n_seg >= 1, seg_len >= 1 and n_seg * seg_len < 2^31 (n_seg = %d, seg_len = %d)", who, n_seg, seg_len);
    return RK_ERR_ARG;
  }
  if((uint64_t)n_seg * (uint64_t)S >= (1ull << 32)) {
    set_error("%s: n_seg * S must be < 2^32", who);
    return RK_ERR_ARG;
  }
  if(ob) {
    if(ob->m < 0) {
      set_error("%s: need m >= 0 discs per robot (m = %d)", who, ob->m);
      return RK_ERR_ARG;
    }
    if(ob->check_period < 1 || seg_len % ob->check_period != 0) {
      set_error("%s: need check_period >= 1 dividing seg_len (check_period = %d, seg_len = %d)", who, ob->check_period, seg_len);
      return RK_ERR_ARG;
    }
    if(!(ob->w_obst >= 0.0f)) {
      set_error("%s: w_obst must be >= 0 (+inf allowed, NaN not)", who);
      return RK_ERR_ARG;
    }
  }
  if(R == 0) return RK_OK;
  if(int rc = check_block(d_src_state, "d_src_state")) return rc;
  if(int rc = check_block(d_cmd, "d_cmd")) return rc;
  if(!cost->d_ref || ((uintptr_t)cost->d_ref & 7u) || !d_cost || ((uintptr_t)d_cost & 3u)) {
    set_error("%s: cost->d_ref (8-byte aligned float2) and d_cost (float) must be non-NULL device pointers", who);
    return RK_ERR_ARG;
  }
  const bool obst = ob && ob->m > 0;
  if(obst && (!ob->d_obs || ((uintptr_t)ob->d_obs & 15u))) {
    set_error("%s: obst->d_obs must be a non-NULL 16-byte aligned device pointer when m > 0", who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  rk_vdt_rollout_t a;
  memset(&a, 0, sizeof(a));
  a.steps = n_seg * seg_len, a.sensor_mode = RK_SENSOR_PLANT;
  a.d_cmd = d_cmd, a.n_seg = n_seg, a.seg_len = seg_len;
  PlanObstArgs pl;
  pl.R = R, pl.S = S, pl.ref = reinterpret_cast<const float2 *>(cost->d_ref);
  pl.w_pos = cost->w_pos, pl.w_goal = cost->w_goal, pl.w_cur = cost->w_cur, pl.cost = d_cost;
  const int64_t n  = R * (int64_t)S;
  cudaStream_t  st = (cudaStream_t)stream;
  if(obst) {
    pl.obs = reinterpret_cast<const float4 *>(ob->d_obs), pl.m = ob->m, pl.P = ob->check_period, pl.w_obst = ob->w_obst;
    launch_plan<true>(*p, d_src_state, n, a, pl, st);
  } else {
    launch_plan<false>(*p, d_src_state, n, a, static_cast<const PlanArgs &>(pl), st);
  }
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}
} // namespace rk
extern "C" {

int rk_plan_rollout(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S, const rk_vdt_cmd_t *d_cmd, int32_t n_seg,
                    int32_t seg_len, const rk_plan_cost_t *cost, float *d_cost, void *stream) {
  return plan_rollout("rk_plan_rollout", p, d_src_state, R, S, d_cmd, n_seg, seg_len, cost, nullptr, d_cost, stream);
}

int rk_plan_rollout_obstacles(const rk_vdt_params_t *p, const void *d_src_state, int64_t R, int32_t S, const rk_vdt_cmd_t *d_cmd,
                              int32_t n_seg, int32_t seg_len, const rk_plan_cost_t *cost, const rk_plan_obstacles_t *obst, float *d_cost,
                              void *stream) {
  return plan_rollout("rk_plan_rollout_obstacles", p, d_src_state, R, S, d_cmd, n_seg, seg_len, cost, obst, d_cost, stream);
}

int rk_vdt_set_power(void *d_state, int64_t n, const uint8_t *d_on, void *stream) {
  if(n <= 0) return RK_OK;
  if(int rc = check_block(d_state, "d_state")) return rc;
  if(int rc = require_device()) return rc;
  vdt_set_power_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((uint4 *)d_state, n, d_on);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_vdt_set_target_vel(const rk_vdt_params_t *p, void *d_state, int64_t n, const float *d_v, const float *d_a,
                          const float *d_j, void *stream) {
  (void)p;
  if(n <= 0) return RK_OK;
  if(!d_v || !d_a || !d_j) {
    set_error("rk_vdt_set_target_vel: NULL v/a/j");
    return RK_ERR_ARG;
  }
  if(int rc = check_block(d_state, "d_state")) return rc;
  if(int rc = require_device()) return rc;
  vdt_set_target_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>((uint4 *)d_state, n, d_v, d_a, d_j);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_vdt_motor_rx(const rk_vdt_params_t *p, void *d_state, int64_t n, int wheel, const uint64_t *d_frames,
                    const int16_t *d_usec, void *stream) {
  if(n <= 0) return RK_OK;
  if(!p || !d_frames || wheel < 0 || wheel > 3) {
    set_error("rk_vdt_motor_rx: bad arguments");
    return RK_ERR_ARG;
  }
  if(int rc = check_block(d_state, "d_state")) return rc;
  if(int rc = require_device()) return rc;
  vdt_motor_rx_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      *p, (uint4 *)d_state, n, wheel, (const unsigned long long *)d_frames, d_usec);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_vdt_tx_frames(const void *d_state, int64_t n, uint64_t *d_frames, void *stream) {
  if(n <= 0) return RK_OK;
  if(!d_frames || ((uintptr_t)d_frames & 7u)) {
    set_error("rk_vdt_tx_frames: d_frames must be a non-NULL 8-byte aligned device pointer");
    return RK_ERR_ARG;
  }
  if(int rc = check_block(d_state, "d_state")) return rc;
  if(int rc = require_device()) return rc;
  vdt_tx_frames_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint4 *)d_state, n, (unsigned long long *)d_frames);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

// ---- single-instance handle: the drop-in for the static objects of VD_task_main.cpp:75-108 -------------
// The state block lives in MAPPED PINNED host memory (zero-copy): the one-thread kernels read and write it over the
// bus, the getters read it from the host side -- no device-to-host copy anywhere.  A 1 kHz firmware tick is
//   rx_callback x4, set_now_yaw_world   -> kept on the host side of the handle (no launch),
//   update()                            -> ONE launch that applies them in arrival order and runs the tick,
//   get_rawCurr_tgt x4 / tx_routine     -> ONE stream synchronisation, then plain loads from the mirror.
struct rk_vdt {
  rk_vdt_params_t p;
  uint32_t       *h_state = nullptr; // mapped pinned; the kernels use the same address (UVA)
  cudaStream_t    st      = nullptr;
  bool            in_flight = false; // a launch since the last synchronisation
  // calls not yet handed to the device
  uint32_t rx_mask = 0;
  uint64_t rx_frame[4] = {0, 0, 0, 0};
  int32_t  rx_usec[4]  = {0, 0, 0, 0};
  bool     has_yaw = false;
  float    yaw     = 0.0f;
};

} // extern "C"
namespace rk {
struct Tick1Args {
  uint32_t           rx_mask;
  unsigned long long frame[4];
  int32_t            usec[4];
  int32_t            has_yaw;
  float              yaw;
  int32_t            do_update;
};
// pending rx_callback()s (VD_motor_if_m2006.cpp:32-72), set_now_yaw_world() (VD_vehicle_controller.hpp:57) and, if asked,
// VEHICLE_CTRL::update() (VD_vehicle_controller.cpp:6-99) on the single instance
__global__ void vdt_tick1_kernel(const rk_vdt_params_t p, uint4 *state, const Tick1Args a) {
  Veh v;
  load_veh(state, 1, 0, v);
#pragma unroll
  for(int k = 0; k < 4; k++)
    if(a.rx_mask & (1u << k)) motor_rx(v.m[k], p.motor_dir[k], a.frame[k], a.usec[k]);
  if(a.has_yaw) v.pos[2] = a.yaw;
  if(a.do_update) {
    const Derived d = derive(p);
    float         c, s;
    yaw_trig(g_sin_table, v.pos[2], c, s);
    veh_update(v, p, d, c, s);
  }
  store_veh(state, 1, 0, v);
}
static int vdt_flush(rk_vdt *h, bool do_update) {
  if(!do_update && !h->rx_mask && !h->has_yaw) return RK_OK;
  Tick1Args a;
  a.rx_mask = h->rx_mask;
  for(int k = 0; k < 4; k++) a.frame[k] = h->rx_frame[k], a.usec[k] = h->rx_usec[k];
  a.has_yaw = h->has_yaw ? 1 : 0, a.yaw = h->yaw, a.do_update = do_update ? 1 : 0;
  vdt_tick1_kernel<<<1, 1, 0, h->st>>>(h->p, (uint4 *)h->h_state, a);
  h->rx_mask = 0, h->has_yaw = false, h->in_flight = true;
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}
// everything handed to the device has finished: the mirror is current
static int vdt_settle(rk_vdt *h) {
  if(int rc = vdt_flush(h, false)) return rc;
  if(h->in_flight) {
    RK_CUDA(cudaStreamSynchronize(h->st));
    h->in_flight = false;
  }
  return RK_OK;
}
} // namespace rk
extern "C" {

int rk_vdt_create(rk_vdt_t **out, const rk_vdt_params_t *p) {
  if(!out) {
    set_error("rk_vdt_create: NULL out");
    return RK_ERR_ARG;
  }
  *out = nullptr;
  if(int rc = require_device()) return rc;
  rk_vdt *h = new rk_vdt();
  if(p)
    h->p = *p;
  else
    rk_vdt_default_params(&h->p);
  cudaError_t e = cudaHostAlloc((void **)&h->h_state, RK_VS_WORDS * 4, cudaHostAllocMapped);
  if(e == cudaSuccess) memset(h->h_state, 0, RK_VS_WORDS * 4); // power-on = zero-initialised statics
  if(e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking);
  if(e != cudaSuccess) {
    int rc = cuda_fail(e, "rk_vdt_create");
    rk_vdt_destroy(h);
    return rc;
  }
  *out = h;
  return RK_OK;
}

void rk_vdt_destroy(rk_vdt_t *h) {
  if(!h) return;
  if(h->st) {
    cudaStreamSynchronize(h->st);
    cudaStreamDestroy(h->st);
  }
  if(h->h_state) cudaFreeHost(h->h_state);
  delete h;
}

int rk_vdt_update(rk_vdt_t *h) {
  if(!h) return RK_ERR_ARG;
  return vdt_flush(h, true);
}

static int poke(rk_vdt_t *h, int word, uint32_t val) {
  if(int rc = vdt_flush(h, false)) return rc;
  vdt_poke_word_kernel<<<1, 1, 0, h->st>>>(h->h_state, (int64_t)word, val); // n = 1: SoA index == word
  h->in_flight = true;
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_vdt_start(rk_vdt_t *h) {
  if(!h) return RK_ERR_ARG;
  if(int rc = vdt_flush(h, false)) return rc;
  h->in_flight = true;
  return rk_vdt_set_power(h->h_state, 1, nullptr, h->st);
}
int rk_vdt_stop(rk_vdt_t *h) {
  if(!h) return RK_ERR_ARG;
  // flags word only carries isPowerOn
  return poke(h, RK_VS_FLAGS, 0u);
}
int rk_vdt_set_target(rk_vdt_t *h, const float v[3], const float a[3], const float j[3]) {
  if(!h || !v || !a || !j) return RK_ERR_ARG;
  if(int rc = vdt_flush(h, false)) return rc;
  vdt_set_target1_kernel<<<1, 1, 0, h->st>>>((uint4 *)h->h_state, v[0], v[1], v[2], a[0], a[1], a[2], j[0], j[1], j[2]);
  h->in_flight = true;
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}
int rk_vdt_set_yaw(rk_vdt_t *h, float yaw_rad) {
  if(!h) return RK_ERR_ARG;
  h->has_yaw = true, h->yaw = yaw_rad; // rides with the next launch
  return RK_OK;
}
int rk_vdt_rx(rk_vdt_t *h, int wheel, const uint8_t frame[8], int16_t usec_id) {
  if(!h || !frame || wheel < 0 || wheel > 3) return RK_ERR_ARG;
  if(h->rx_mask & (1u << wheel)) // a second frame for the same wheel before the tick: keep the arrival order
    if(int rc = vdt_flush(h, false)) return rc;
  memcpy(&h->rx_frame[wheel], frame, 8);
  h->rx_usec[wheel] = (int32_t)usec_id;
  h->rx_mask |= 1u << wheel;
  return RK_OK;
}

int rk_vdt_get_state(rk_vdt_t *h, uint32_t words[RK_VS_WORDS]) {
  if(!h || !words) return RK_ERR_ARG;
  if(int rc = vdt_settle(h)) return rc;
  memcpy(words, h->h_state, RK_VS_WORDS * 4); // n = 1: SoA == AoS
  return RK_OK;
}
int rk_vdt_set_state(rk_vdt_t *h, const uint32_t words[RK_VS_WORDS]) {
  if(!h || !words) return RK_ERR_ARG;
  if(int rc = vdt_settle(h)) return rc;
  memcpy(h->h_state, words, RK_VS_WORDS * 4);
  return RK_OK;
}
static int get3(rk_vdt_t *h, int word0, float out[3]) {
  if(int rc = vdt_settle(h)) return rc;
  memcpy(out, &h->h_state[word0], 12);
  return RK_OK;
}
int rk_vdt_get_pos(rk_vdt_t *h, float out[3]) { return (h && out) ? get3(h, RK_VS_POS_X, out) : RK_ERR_ARG; }
int rk_vdt_get_vel(rk_vdt_t *h, float out[3]) { return (h && out) ? get3(h, RK_VS_VEL_X, out) : RK_ERR_ARG; }
int rk_vdt_get_vel_tgt(rk_vdt_t *h, float out[3]) { return (h && out) ? get3(h, RK_VS_TGT_X, out) : RK_ERR_ARG; }
int rk_vdt_get_raw_current(rk_vdt_t *h, int16_t out[4]) {
  if(!h || !out) return RK_ERR_ARG;
  if(int rc = vdt_settle(h)) return rc;
  for(int k = 0; k < 4; k++) out[k] = (int16_t)(h->h_state[RK_VS_MOTOR0 + 8 * k + RK_VM_CUR_TGT] >> 16);
  return RK_OK;
}
int rk_vdt_get_tx_frame(rk_vdt_t *h, uint8_t frame[8]) {
  if(!h || !frame) return RK_ERR_ARG;
  int16_t c[4];
  if(int rc = rk_vdt_get_raw_current(h, c)) return rc;
  for(int k = 0; k < 4; k++) frame[2 * k] = (uint8_t)(c[k] >> 8), frame[2 * k + 1] = (uint8_t)(c[k] & 0x00FF);
  return RK_OK;
}
int rk_vdt_get_angle_sum(rk_vdt_t *h, int64_t out[4]) {
  if(!h || !out) return RK_ERR_ARG;
  if(int rc = vdt_settle(h)) return rc;
  for(int k = 0; k < 4; k++) {
    const uint32_t *q = &h->h_state[RK_VS_MOTOR0 + 8 * k];
    out[k]            = (int64_t)(((uint64_t)q[RK_VM_SUM_HI] << 32) | q[RK_VM_SUM_LO]);
  }
  return RK_OK;
}

} // extern "C"
