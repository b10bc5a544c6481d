// rk_arm.cu -- 5-axis arm tick batched (src/ArmDrive): ADTModePositioningSeq::update() +
// the joint command packers, one ADT::main loop body per tick (AD_task_main.cpp:208-229).
//
// One thread per arm.  The 19 state planes (304 B) are loaded once with 128-bit loads, the
// live words stay in registers for the K fused ticks, and are stored once.  The command ring
// (4 slots x 65 planes per arm) lives in its own block and is touched only at a segment start
// (2 planes = one waypoint, + the slot header), so a 100 Hz tick costs no HBM traffic at all:
// the kernel is issue/latency bound, not bandwidth bound (SURVEY.md 8d, C4).
#include <string.h>

#include <type_traits>

#include "rk_vehicle_fast.cuh" // div_const(), rk_math.cuh

namespace rk {
int div_const_exact(float c); // rk_exact.cu: 2 = exact for all x, 1 = for x == 0 or |x| >= 2^-40, 0 = no

// IcsBaseClass::posDeg100   lib/IcsClass_V210/src/IcsBaseClass.cpp:105-137 (C division truncates toward zero)
RK_DEV int ics_posDeg100(int pos) {
  int deg;
  if(pos >= -2000000 && pos <= 2000000) { // every position a 14-bit ICS frame can carry: 32-bit arithmetic
    deg = ((pos - 7500) * 1000) / 296;
  } else { // arbitrary state words: the reference's 64-bit `long` arithmetic
    const long long a = (long long)pos - 7500;
    deg               = (int)((a * 1000) / 296);
  }
  if(deg > 18000) return 0x7FFF;
  if(deg < -18000) return -0x7FFF;
  return deg;
}
// JointIcsServo: fl_raw_now_deg from the position word the servo answers with (update() and init())
RK_DEV float ics_now_deg(int pos, float dir) { return fmul(fmul((float)ics_posDeg100(pos), 0.01f), dir); }

// mode axis J0..J4 -> joint object (AD_task_main.cpp:148)
RK_DEV constexpr int axis_joint(int ax) { return ax == 0 ? RK_AJ_Y0 : ax == 1 ? RK_AJ_P1 : ax == 2 ? RK_AJ_P2 : ax == 3 ? RK_AJ_R0 : RK_AJ_P3; }

RK_DEV uint32_t bldc_id_byte(uint32_t id) { return (id & 0xFFu) | ((id & 0x8000u) ? 0x80u : 0u); }

// ---------------------------------------------------------------------------------------------
// K fused ticks.  Only the words a tick reads or writes live in registers (ArmLoop); words that
// are constant during update() -- unused offsets / limits / measured angles, the reserved
// torque-control block -- stay in HBM and are merged back plane by plane at the end.  The tick
// is straight-line predicated code apart from the two rare FSM transitions, so ptxas can
// interleave its six independent chains (mode, MG, 3 x MyBldc, ICS) and their long-latency
// conversions (F2I / I2FP ~12 cycles each).  DIVC: the MG velocity limit divides by a launch
// constant through div_const() when rk_exact.cu has proven it exact for every finite input.
// ---------------------------------------------------------------------------------------------
struct MgFrame {
  uint32_t tx0, tx1, valid;
};
struct ArmLoop {
  uint32_t state, fsmflags, exec, head, cmd_idx;
  int32_t  cnt, cyc;
  uint32_t total_ms, now_dt;
  float    now_tgt[5], move[5], dfv_p, dfv_r;
  float    ofs[5], ofs_dfl, ofs_dfr; // offsets: mode axes J0..J4, DF_Left, DF_Right
  float    tgt[5], tgt_dfl, tgt_dfr; // fl_raw_tgt_deg of the same
  float    cl_dfl, cl_dfr, cl_p3;    // fl_curlim_A of the three MyBldc joints
  float    now_y0, mg_pre;
  float    mg_pp; // LAZY_MG: f_pre_tgt_deg as it stood before the last tick
  int32_t  y0_pos;  // LAZY_Y0: the position word of the ICS servo's last answer, converted after the last tick
  bool     y0_seen;
  uint32_t ics_pos, ics_servo;
  MgFrame  mg; // tx1data words 0, 1 and the valid word of the MG joint
  uint32_t bl0[3], bl1[3], bl2[3];   // txmsg word 0, word 1, u32_txcmdid per MyBldc joint
  bool     mg_prev, bl_prev[3];
  // command-ring prefetch: the lengths of the four slots (8 bits each) and the waypoint the FSM
  // will ask for next, fetched one segment ahead so its HBM latency never stalls a tick.  The
  // ring is read-only while update() runs (push_cmdseq is a separate call), so reading early
  // returns the same words.  Two register sets alternate (sel = the set holding the prefetched
  // waypoint): a set is only ever written by a predicated load and read by a select, so no copy
  // has to wait for a load in flight.
  uint32_t lens, pf_key; // pf_key = slot * 32 + index of the prefetched waypoint, or ~0u
  uint4    pa0, pb0;     // {u32_dt_ms, fl_tgt_pos_deg[0..2]}
  uint2    pa1, pb1;     // fl_tgt_pos_deg[3..4]
  bool     sel;
};

RK_DEV uint32_t ring_len(const ArmLoop &a, uint32_t slot) { return (a.lens >> (8 * (slot % RK_ACMD_SLOTS))) & 0xFFu; }
RK_DEV uint32_t ring_key(uint32_t slot, uint32_t idx) { return (slot % RK_ACMD_SLOTS) * RK_ACMD_MAX_LEN + (idx % RK_ACMD_MAX_LEN); }

// `if(pred) dst = *addr` as ONE predicated load into the registers dst already lives in.  The two
// register sets use different load flavours (read-only path / L2-coherent path): ptxas otherwise
// merges the complementary-predicate pair into one load plus moves that wait for it.
template <bool NC> RK_DEV void ldg_if(uint4 &d, const uint4 *addr, bool pred) {
  if(NC)
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %5, 0; @p ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4]; }"
                 : "+r"(d.x), "+r"(d.y), "+r"(d.z), "+r"(d.w) : "l"(addr), "r"((uint32_t)pred));
  else
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %5, 0; @p ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4]; }"
                 : "+r"(d.x), "+r"(d.y), "+r"(d.z), "+r"(d.w) : "l"(addr), "r"((uint32_t)pred));
}
template <bool NC> RK_DEV void ldg_if(uint2 &d, const uint4 *addr, bool pred) {
  if(NC)
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %3, 0; @p ld.global.nc.v2.u32 {%0, %1}, [%2]; }" : "+r"(d.x), "+r"(d.y) : "l"(addr), "r"((uint32_t)pred));
  else
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %3, 0; @p ld.global.cg.v2.u32 {%0, %1}, [%2]; }" : "+r"(d.x), "+r"(d.y) : "l"(addr), "r"((uint32_t)pred));
}
// waypoint (slot, idx) -> register set B when `into_b`, else set A
RK_DEV void ring_fetch(ArmLoop &a, const uint4 *__restrict__ tab, int64_t n, int64_t i, uint32_t slot, uint32_t idx, bool into_b) {
  const int    pl = (int)(slot % RK_ACMD_SLOTS) * (RK_ACMD_SLOT_WORDS / 4) + 1 + 2 * (int)(idx % RK_ACMD_MAX_LEN);
  const uint4 *p0 = &tab[(int64_t)pl * n + i], *p1 = &tab[(int64_t)(pl + 1) * n + i];
  ldg_if<true>(a.pa0, p0, !into_b), ldg_if<true>(a.pa1, p1, !into_b);
  ldg_if<false>(a.pb0, p0, into_b), ldg_if<false>(a.pb1, p1, into_b);
}
// what exec_move_start will read after the segment (slot, idx) that is starting now: the next waypoint
// of the sequence, else waypoint 0 of the next queued sequence, else (nothing to come) the same entry
RK_DEV void ring_next(const ArmLoop &a, uint32_t slot, uint32_t idx, uint32_t &nslot, uint32_t &nidx) {
  const bool more = idx + 1 < ring_len(a, slot) && idx + 1 < RK_ACMD_MAX_LEN;
  const bool next = !more && slot != a.head;
  uint32_t   nx   = (slot + 1) & 0xFFFFu;
  nx              = (nx >= RK_ACMD_SLOTS) ? 0u : nx;
  nslot = next ? nx : slot, nidx = more ? idx + 1 : (next ? 0u : idx);
}

// IEEE single-precision x / c through one double-precision reciprocal shared by several numerators:
//   RN32(x / c) == RN32(RN64((double)x * RN64(1 / (double)c)))   whenever the quotient is a NORMAL float (or 0, inf, NaN).
// Why: a normal-range quotient of two floats is never a midpoint of two adjacent floats, and is at least 2^-49
// (relative) away from every such midpoint (|A * 2^ea - B * M * 2^e| >= 2^e for the 24-bit significands A, B and a 25-bit
// odd M, over B * M * 2^e < 2^49 * 2^e), while the double product carries at most 2^-52 of relative error (2^-53 from the
// rounded reciprocal, 2^-53 from the product) -- so it lies on the same side of every float rounding boundary as the
// exact quotient.  Zeros keep the numerator's sign, x / inf = 0, x / 0 = inf, 0 / 0 = NaN as in the IEEE division.
// SUBNORMAL quotients can be exact ties (3 * 2^-149 / 6 = 2^-150), where the inexact reciprocal decides the rounding
// instead of ties-to-even: those (|q| < 2^-125, x != 0) take the IEEE division.  rk_selftest_div_rcp64
// (tests/test_arm_gpu.py) compares the function with div.rn.f32 on 2^32 (x, c) pairs, integer counts included.
RK_DEV float div_by_rcp64_raw(float x, double rc) { return __double2float_rn(__dmul_rn((double)x, rc)); }
RK_DEV bool  div_by_rcp64_unsafe(float x, float q) { return fabsf(q) < 2.3509887e-38f /* 2^-125 */ && x != 0.0f; }
RK_DEV float div_by_rcp64(float x, float c, double rc) {
  const float q = div_by_rcp64_raw(x, rc);
  return div_by_rcp64_unsafe(x, q) ? fdiv(x, c) : q;
}

RK_DEV uint4 ldp(const uint4 *st, int64_t n, int64_t i, int word) { return ld_plane(st, n, word / 4, i); }

RK_DEV void loop_load(const uint4 *st, int64_t n, int64_t i, ArmLoop &a, uint32_t &jflags) {
  const uint4 f0 = ldp(st, n, i, RK_AS_FSM), f1 = ldp(st, n, i, RK_AS_CYCLE);
  a.state = f0.x & 0xFFu, a.fsmflags = f0.x & ~0xFFu, a.exec = f0.y & 0xFFFFu, a.head = f0.y >> 16, a.cmd_idx = f0.z;
  a.cnt = (int32_t)f0.w, a.cyc = (int32_t)f1.x, a.total_ms = f1.y, a.now_dt = f1.z;
  const uint4 t0 = ldp(st, n, i, RK_AS_NOW_TGT), t1 = ldp(st, n, i, 12), t2 = ldp(st, n, i, 16);
  a.now_tgt[0] = u2f(t0.x), a.now_tgt[1] = u2f(t0.y), a.now_tgt[2] = u2f(t0.z), a.now_tgt[3] = u2f(t0.w), a.now_tgt[4] = u2f(t1.x);
  a.move[0] = u2f(t1.y), a.move[1] = u2f(t1.z), a.move[2] = u2f(t1.w), a.move[3] = u2f(t2.x), a.move[4] = u2f(t2.y);
  a.dfv_p = u2f(t2.z), a.dfv_r = u2f(t2.w);
#pragma unroll
  for(int ax = 0; ax < 5; ax++) {
    const uint4 j = ldp(st, n, i, RK_AS_JOINT0 + 4 * axis_joint(ax));
    a.ofs[ax] = u2f(j.x), a.tgt[ax] = u2f(j.y);
    if(ax == 0) a.now_y0 = u2f(j.w);
    if(ax == 4) a.cl_p3 = u2f(j.z);
  }
  const uint4 l = ldp(st, n, i, RK_AS_JOINT0 + 4 * RK_AJ_DFL), r = ldp(st, n, i, RK_AS_JOINT0 + 4 * RK_AJ_DFR);
  a.ofs_dfl = u2f(l.x), a.tgt_dfl = u2f(l.y), a.cl_dfl = u2f(l.z);
  a.ofs_dfr = u2f(r.x), a.tgt_dfr = u2f(r.y), a.cl_dfr = u2f(r.z);
  const uint4 m = ldp(st, n, i, RK_AS_JFLAGS), x = ldp(st, n, i, RK_AS_MG_TX);
  jflags = m.x, a.mg_pre = u2f(m.y), a.ics_pos = m.z, a.ics_servo = m.w;
  a.mg = {x.x, x.y, x.z};
#pragma unroll
  for(int s = 0; s < 3; s++) {
    const uint4 b = ldp(st, n, i, RK_AS_BLDC_TX0 + 4 * s);
    a.bl0[s] = b.x, a.bl1[s] = b.y, a.bl2[s] = b.z;
  }
  a.lens = 0u, a.pf_key = 0xFFFFFFFFu, a.sel = false;
  a.y0_pos = -1, a.y0_seen = false;
  a.pa0 = make_uint4(0u, 0u, 0u, 0u), a.pb0 = a.pa0, a.pa1 = make_uint2(0u, 0u), a.pb1 = a.pa1;
  a.mg_prev    = ((jflags >> (4 * RK_AJ_P1)) & RK_AJF_TORQUE_PREV) != 0;
  a.bl_prev[0] = ((jflags >> (4 * RK_AJ_DFL)) & RK_AJF_TORQUE_PREV) != 0;
  a.bl_prev[1] = ((jflags >> (4 * RK_AJ_DFR)) & RK_AJF_TORQUE_PREV) != 0;
  a.bl_prev[2] = ((jflags >> (4 * RK_AJ_P3)) & RK_AJF_TORQUE_PREV) != 0;
}

RK_DEV void loop_store(uint4 *st, int64_t n, int64_t i, const ArmLoop &a, uint32_t jflags, bool ticked) {
  st_plane(st, n, 0, i, make_uint4(a.state | a.fsmflags, a.exec | (a.head << 16), a.cmd_idx, (uint32_t)a.cnt));
  uint4 f1 = ldp(st, n, i, RK_AS_CYCLE);
  f1.x = (uint32_t)a.cyc, f1.y = a.total_ms, f1.z = a.now_dt;
  st_plane(st, n, 1, i, f1);
  st_plane(st, n, 2, i, make_uint4(f2u(a.now_tgt[0]), f2u(a.now_tgt[1]), f2u(a.now_tgt[2]), f2u(a.now_tgt[3])));
  st_plane(st, n, 3, i, make_uint4(f2u(a.now_tgt[4]), f2u(a.move[0]), f2u(a.move[1]), f2u(a.move[2])));
  st_plane(st, n, 4, i, make_uint4(f2u(a.move[3]), f2u(a.move[4]), f2u(a.dfv_p), f2u(a.dfv_r)));
#pragma unroll
  for(int ax = 0; ax < 5; ax++) {
    const int pl = (RK_AS_JOINT0 + 4 * axis_joint(ax)) / 4;
    uint4     j  = ld_plane(st, n, pl, i);
    j.y          = f2u(a.tgt[ax]);
    if(ax == 0) j.w = f2u(a.now_y0);
    st_plane(st, n, pl, i, j);
  }
  {
    const int pl = (RK_AS_JOINT0 + 4 * RK_AJ_DFL) / 4;
    uint4     l = ld_plane(st, n, pl, i), r = ld_plane(st, n, pl + 1, i);
    l.y = f2u(a.tgt_dfl), r.y = f2u(a.tgt_dfr);
    st_plane(st, n, pl, i, l);
    st_plane(st, n, pl + 1, i, r);
  }
  if(ticked) { // is_torque_on_prev = is_torque_on after any tick
    const uint32_t prevbits = ((uint32_t)RK_AJF_TORQUE_PREV << (4 * RK_AJ_P1)) | ((uint32_t)RK_AJF_TORQUE_PREV << (4 * RK_AJ_DFL)) |
                              ((uint32_t)RK_AJF_TORQUE_PREV << (4 * RK_AJ_DFR)) | ((uint32_t)RK_AJF_TORQUE_PREV << (4 * RK_AJ_P3));
    const uint32_t onbits   = ((uint32_t)RK_AJF_TORQUE_ON << (4 * RK_AJ_P1)) | ((uint32_t)RK_AJF_TORQUE_ON << (4 * RK_AJ_DFL)) |
                            ((uint32_t)RK_AJF_TORQUE_ON << (4 * RK_AJ_DFR)) | ((uint32_t)RK_AJF_TORQUE_ON << (4 * RK_AJ_P3));
    jflags = (jflags & ~prevbits) | ((jflags & onbits) << 2); // TORQUE_PREV = TORQUE_ON << 2
  }
  st_plane(st, n, RK_AS_JFLAGS / 4, i, make_uint4(jflags, f2u(a.mg_pre), a.ics_pos, a.ics_servo));
  uint4 x = ldp(st, n, i, RK_AS_MG_TX);
  x.x = a.mg.tx0, x.y = a.mg.tx1, x.z = a.mg.valid;
  st_plane(st, n, RK_AS_MG_TX / 4, i, x);
#pragma unroll
  for(int s = 0; s < 3; s++) st_plane(st, n, (RK_AS_BLDC_TX0 + 4 * s) / 4, i, make_uint4(a.bl0[s], a.bl1[s], a.bl2[s], 1u));
}

struct ArmConsts { // loop invariants derived from params + flags once per launch
  float    gear_p2, gear_r0, gear_dir[3], dir_y0, mg_ctrl_time, mg_rcp;
  uint32_t bl_ms[3];
  bool     y0_conn, y0_on, mg_pos, mg_on, mg_ini, bl_on[3];
};

// exec_standby + exec_move_start: the rare, divergent part of ADTModePositioningSeq::update
RK_DEV void loop_fsm_transitions(ArmLoop &a, const rk_adt_params_t &p, const uint4 *__restrict__ tab, int64_t n, int64_t i) {
  if(a.state == RK_ASTATE_STANDBY) { // exec_standby :24-42
    a.fsmflags |= RK_AS_FSM_IS_COMP;
    if(a.exec != a.head) {
      a.exec = (a.exec + 1) & 0xFFFFu;
      a.exec = (a.exec >= RK_ACMD_SLOTS) ? 0u : a.exec;
      a.cmd_idx  = 0;
      a.total_ms = 0;
      a.state    = RK_ASTATE_MOVE_START;
      a.fsmflags &= ~RK_AS_FSM_FIRSTCALL;
    }
  }
  if(a.state == RK_ASTATE_MOVE_START) { // exec_move_start :48-83
    const uint32_t len = ring_len(a, a.exec);
    const uint32_t idx = a.cmd_idx & 0xFFu;
    if(idx >= len) {
      a.state = RK_ASTATE_STANDBY;
    } else {
      // now_cmd_ = cmd_seq_[exec].cmd_seq[idx]: one waypoint = two 128-bit planes, normally already prefetched
      if(a.pf_key != ring_key(a.exec, idx)) ring_fetch(a, tab, n, i, a.exec, idx, a.sel);
      const uint4 w0 = a.sel ? a.pb0 : a.pa0;
      const uint2 w1 = a.sel ? a.pb1 : a.pa1;
      uint32_t    ns, ni;
      ring_next(a, a.exec, idx, ns, ni);
      a.sel = !a.sel;
      ring_fetch(a, tab, n, i, ns, ni, a.sel);
      a.pf_key = ring_key(ns, ni);
      a.now_dt       = w0.x;
      a.now_tgt[0] = u2f(w0.y), a.now_tgt[1] = u2f(w0.z), a.now_tgt[2] = u2f(w0.w), a.now_tgt[3] = u2f(w1.x), a.now_tgt[4] = u2f(w1.y);
      // a zero numerator (dt equal to the previous one; an axis that does not move) would send the
      // IEEE division down its slow path: 0 / c = 0 with the numerator's sign for c > 0
      const float span = fmul(__uint2float_rn(a.now_dt - a.total_ms), 0.001f);
      int32_t     cnt  = f2i_x86((span == 0.0f && p.cycle_time_s > 0.0f) ? span : fdiv(span, p.cycle_time_s));
      cnt              = (cnt <= 0) ? 1 : cnt;
      const float fc   = (float)cnt; // >= 1
      // the five divisions by the same count through one double-precision reciprocal (div_by_rcp64)
      const double rc = __drcp_rn((double)fc);
      float        d[5];
      bool  slow = false; // one test for the five quotients: the IEEE division is out of the way of the common case
#pragma unroll
      for(int k = 0; k < 5; k++) {
        d[k]      = fsub(a.now_tgt[k], fsub(a.tgt[k], a.ofs[k]));
        a.move[k] = div_by_rcp64_raw(d[k], rc);
        slow |= div_by_rcp64_unsafe(d[k], a.move[k]);
      }
      if(slow) { // (static indices: a rolled loop would put d[] and move[] into local memory)
#pragma unroll
        for(int k = 0; k < 5; k++) a.move[k] = fdiv(d[k], fc);
      }
      a.cnt      = cnt;
      a.total_ms = a.now_dt;
      a.cyc      = 0;
      a.fsmflags &= ~RK_AS_FSM_IS_COMP;
      a.state = RK_ASTATE_MOVING;
    }
  }
}

// the five set_tgt_ang_deg() calls of exec_moving (JointBase :42, DfGear overrides), predicated on `moving`
RK_DEV void loop_set_targets(ArmLoop &a, const ArmConsts &c, bool moving, float rem, const float now_tgt[5], const float move[5]) {
  float raw[5];
#pragma unroll
  for(int k = 0; k < 5; k++) {
    raw[k]   = fadd(fsub(now_tgt[k], fmul(move[k], rem)), a.ofs[k]);
    a.tgt[k] = moving ? raw[k] : a.tgt[k];
  }
  const float P = fmul(raw[2], c.gear_p2), R = fmul(raw[3], c.gear_r0);
  a.dfv_p = moving ? P : a.dfv_p, a.dfv_r = moving ? R : a.dfv_r;
  a.tgt_dfl = moving ? fadd(fsub(P, R), a.ofs_dfl) : a.tgt_dfl;
  a.tgt_dfr = moving ? fadd(-fadd(P, R), a.ofs_dfr) : a.tgt_dfr;
}

// (int32_t)(double) as cvttsd2si
RK_DEV int32_t d2i_x86(double d) { return (fabs(d) < 2147483648.0) ? __double2int_rz(d) : (int32_t)0x80000000u; }

// The three branches of JointMgServo::update() other than position control (AD_joint_mg_servo.cpp:50-73):
// PI_D reset on the torque on->off edge, torque control while not initialised, InitGain + torque
// control while torque is off (subproc_torquectrl :104-134, UTIL::PI_D util_controller.hpp:86-153, the
// double-precision current->raw map AD_joint_mg_servo.hpp:120-136).  q0, q1: the eight RK_AS_MG_CTRL words as
// two planes; jp: the MG joint's plane {ofs, raw_tgt, curlim, raw_now}.
RK_DEV MgFrame mg_torque_ctrl(MgFrame f, uint4 &q0, uint4 &q1, uint4 jp, float tgt, float ctrl_time_s, bool prev, bool on, bool ini) {
  f.valid = 0u;
  if(prev && !on) { // pos_ctrl_.reset(): everything but the gains
    q0 = make_uint4(0u, 0u, 0u, 0u);
    q1.x = 0u, q1.y = 0u, q1.z = 0u;
  } else {
    if(!on) { // set_myctrl_gain_params(InitGain): gains + set_VelLpf_CutOff -> IIR reset
      q1.w = 1u;
      q0.z = 0u, q0.w = 0u;
    }
    const float freq = fdiv(1.0f, ctrl_time_s), dt = fdiv(1.0f, freq), lpf = 10.0f;
    const float den  = fadd(fmul(2.0f, freq), lpf);
    const float A1 = fdiv(fsub(fmul(2.0f, freq), lpf), den), B0 = fdiv(lpf, den);
    const float pg = q1.w ? 0.01f : 0.0f, ig = 0.0f, dg = 0.0f, ilim = 0.0f;
    const float now = u2f(jp.w), curlim = u2f(jp.z);
    const float err = fsub(tgt, now);
    const float x   = fmul(fsub(now, u2f(q0.x)), freq);
    const float y   = fadd(fadd(fmul(A1, u2f(q0.z)), fmul(B0, x)), fmul(B0, u2f(q0.w)));
    float integ     = fadd(u2f(q0.y), fmul(fmul(ig, dt), err));
    integ           = (integ >= ilim) ? ilim : ((integ <= -ilim) ? -ilim : integ);
    float iq        = fsub(fadd(fmul(pg, err), integ), fmul(dg, y));
    q0 = make_uint4(f2u(now), f2u(integ), f2u(y), f2u(x));
    q1.x = f2u(tgt), q1.y = f2u(err), q1.z = f2u(iq);
    if(ini) iq = fsub(iq, fmul(0.05f, arm_sin(g_sin_table, fmul(fsub(now, u2f(jp.x)), RK_DEG2RAD))));
    iq = (iq > curlim) ? curlim : ((iq < -curlim) ? -curlim : iq);
    const double C_A = 0.0000057204, C_B = -0.0000485371, d = (double)iq;
    double       raw;
    if(d >= 0) raw = __ddiv_rn(__dadd_rn(-C_B, (double)arm_sqrt(__double2float_rn(__dadd_rn(C_B * C_B, __dmul_rn(4.0 * C_A, d))))), 2.0 * C_A);
    else raw = __ddiv_rn(__dsub_rn(C_B, (double)arm_sqrt(__double2float_rn(__dsub_rn(C_B * C_B, __dmul_rn(4.0 * C_A, d))))), 2.0 * C_A);
    int32_t s = sext16(d2i_x86(__dmul_rn(-1.0, raw)));
    s         = (s > 450) ? 450 : ((s < -450) ? -450 : s);
    f.tx0 = 0xA1u, f.tx1 = (uint32_t)s & 0xFFFFu, f.valid = 1u;
  }
  return f;
}
// The sequence tick's form: rare there (an arm that is being homed or is limp), so the PI_D block is read and
// written in HBM and the function is kept out of line.
__device__ __noinline__ MgFrame mg_update_slow(MgFrame f, float tgt, float ctrl_time_s, bool prev, bool on, bool ini, uint4 *st,
                                               int64_t n, int64_t i) {
  uint4       q0 = ld_plane(st, n, RK_AS_MG_CTRL / 4, i), q1 = ld_plane(st, n, RK_AS_MG_CTRL / 4 + 1, i);
  const uint4 jp = ld_plane(st, n, (RK_AS_JOINT0 + 4 * RK_AJ_P1) / 4, i); // {ofs, raw_tgt (stale), curlim, raw_now}
  f              = mg_torque_ctrl(f, q0, q1, jp, tgt, ctrl_time_s, prev, on, ini);
  st_plane(st, n, RK_AS_MG_CTRL / 4, i, q0);
  st_plane(st, n, RK_AS_MG_CTRL / 4 + 1, i, q1);
  return f;
}

template <int DIVC, bool MGSLOW, bool LAZY_Y0 = false, bool STEADY = false, bool LAZY_MG = false>
RK_DEV void loop_joints(ArmLoop &a, const rk_adt_params_t &p, const ArmConsts &c, uint4 *st, int64_t n, int64_t i);

// LAZY (no trace attached): what nobody reads inside the launch is not formed per tick.  Inside a segment the five targets
// are a pure function of the segment's constants and the tick count (now_cmd_ - move * rem + offset), and between two
// segment ends only the ICS joint (axis 0, which converts its target every tick) looks at them: exec_move_start measures
// the next segment from the targets of the tick that ENDED the previous one, the MyBldc / MG frames and the stored block
// need those of the launch's last ticks.  So axes 1..4 and the differential are formed on the ticks that end a segment
// and on the last two ticks of the launch (`eager`), with the same operations on the same operands; the MG joint's
// position frame is formed once after the last tick (LAZY_MG of loop_joints).  Not for an MG joint in torque control
// (its PI_D consumes the target every tick).
template <int DIVC, bool MGSLOW, bool STEADY = false, bool LAZY = false>
RK_DEV void loop_tick(ArmLoop &a, const rk_adt_params_t &p, const ArmConsts &c, uint4 *st, const uint4 *__restrict__ tab, int64_t n, int64_t i,
                      bool eager = true) {
  if(a.state != RK_ASTATE_MOVING) loop_fsm_transitions(a, p, tab, n, i);
  // ---- exec_moving :89-117
  const bool  moving = a.state == RK_ASTATE_MOVING;
  const bool  fin    = moving && (a.cnt <= a.cyc);
  const float rem    = (float)(a.cnt - a.cyc);
  if(LAZY) {
    const float raw0 = fadd(fsub(a.now_tgt[0], fmul(a.move[0], rem)), a.ofs[0]);
    a.tgt[0]         = moving ? raw0 : a.tgt[0];
    if(fin || eager) loop_set_targets(a, c, moving, rem, a.now_tgt, a.move);
  } else {
    loop_set_targets(a, c, moving, rem, a.now_tgt, a.move);
  }
  a.cmd_idx      = fin ? ((a.cmd_idx + 1) & 0xFFu) : a.cmd_idx;
  a.state        = fin ? (uint32_t)RK_ASTATE_MOVE_START : a.state;
  a.cyc          = (moving && !fin) ? a.cyc + 1 : a.cyc;
  loop_joints<DIVC, MGSLOW, true, STEADY, LAZY>(a, p, c, st, n, i);
}

// JointMgServo::subproc_posctrl  AD_joint_mg_servo.cpp:136-149: the 0xA4 frame (velocity limit from the step since the
// last target, position) from the raw target and the previous one; ct = fl_ctrl_time_s, rcp = RN(1 / ct) when DIVC > 0.
template <int DIVC>
RK_DEV MgFrame mg_posctrl_frame(float tgt, float pre, float ct, float rcp) {
  const float d = fsub(tgt, pre);
  float       q;
  if(DIVC == 2) {
    q = div_const(d, ct, rcp);
  } else if(DIVC == 1) { // proven for zero and 2^-40 <= |d| <= 2^64; anything else takes the IEEE division
    const float ad = fabsf(d);
    if(d == 0.0f || (ad >= 9.094947017729282e-13f && ad <= 18446744073709551616.0f)) q = div_const(d, ct, rcp);
    else q = fdiv(d, ct);
  } else { // 0 / c = 0 with the numerator's sign for c > 0; keeps an idle joint off the division's slow path
    q = (d == 0.0f && ct > 0.0f) ? d : fdiv(d, ct);
  }
  const float    v  = fabsf(fmul(q, -10.0f));
  const uint32_t vl = (uint32_t)f2i_x86((v > 1800.0f) ? 1800.0f : v) & 0xFFFFu;
  const uint32_t w1 = (uint32_t)f2i_x86(fmul(tgt, -100.0f * 10.0f));
  return {0xA4u | (vl << 16), w1, 1u};
}
template <int DIVC>
RK_DEV void loop_finish_mg(ArmLoop &a, const ArmConsts &c) { a.mg = mg_posctrl_frame<DIVC>(a.mg_pre, a.mg_pp, c.mg_ctrl_time, c.mg_rcp); }

// The MyBldc and ICS packers are shared by the sequence tick and the homing tick as statement macros rather than
// functions: written as inline functions, the different inlining order changes how ptxas schedules the sequence kernel.
//
// JointMyBldcServo::update  AD_joint_mybldc_servo.cpp:7-36 for joint k: txmsg words 0 and 1 and u32_txcmdid (w0..w2)
// from the raw target, the current limit and the control period in ms (bldc_ms)
RK_DEV uint32_t bldc_ms(float ctrl_time_s) { return (uint32_t)f2i_x86(fmul(ctrl_time_s, 1000.0f)) & 0xFFFFu; }
#define RK_BLDC_FRAME(p, k, tg, cl, ms, on, prev_, w0, w1, w2)                                                 \
  {                                                                                                        \
    const int32_t  ang   = f2i_x86(fmul(fmul(fmul(tg, (p).gear_ratio[k]), (p).motor_dir[k]), 65536.0f));   \
    const uint32_t clq   = (uint32_t)f2i_x86(fmul(cl, 256.0f)) & 0xFFFFu;                                    \
    const bool     prev  = prev_;                                                                          \
    const bool     drive = (on) && prev;                                                                   \
    w0                   = drive ? (uint32_t)ang : 0u;                                                     \
    w1                   = drive ? ((ms) | (clq << 16)) : 0u;                                              \
    w2                   = !(on) ? 0x8002u : (prev ? 0x8010u : 0x8001u);                                   \
  }
// JointIcsServo::update  AD_joint_ics_servo.cpp:5-29 over the ideal servo (IcsBaseClass::degPos100, setPos / setFree):
// updates the position word handed to setPos and what the servo reports, and declares `active` (the servo answered)
// and `now_pos` (the position word of its answer).
#define RK_ICS_UPDATE(tgt, dir, conn, on, ics_pos, ics_servo)                                              \
  const int  deg100  = f2i_x86(fmul(fmul(tgt, dir), 100.0f));                                            \
  const bool in_deg  = deg100 <= 18000 && deg100 >= -18000;                                              \
  const int  tp      = (deg100 * 2963) / 10000 + 7500; /* garbage when !in_deg, never used then */       \
  const bool active  = (conn) && in_deg;                                                                  \
  const bool send    = active && (on) && tp <= 11500 && tp >= 3500;                                       \
  const bool fre     = active && !(on);                                                                   \
  const int  now_pos = send ? tp : (fre ? (int)(int32_t)(ics_servo) + 7500 : -1);                        \
  ics_pos            = send ? (uint32_t)tp : (fre ? 0xFFFFFFFFu : (ics_pos));                             \
  ics_servo          = send ? (uint32_t)(tp - 7500) : (ics_servo);

// ADT::main's joint updates (AD_task_main.cpp:213-228): j_P1, j_DF_Left, j_DF_Right, j_P3, [CAN tx], j_Y0
// MGSLOW: the thread's MG joint is NOT in position control (c.mg_pos is invariant over the launch); the
// kernel runs such threads through a separate instantiation of the tick loop so that the common loop
// carries none of the torque-control code.
// LAZY_Y0: the ICS joint's fl_raw_now_deg (the position the servo answers with) is read by nobody inside
// ADTModePositioningSeq's tick -- the mode measures from the targets -- so the sequence kernel only remembers the last
// answer (y0_pos, y0_seen) and converts it once after its last tick (loop_finish_y0); ADTModePositioning measures
// from get_now_deg() and keeps the eager form.
// STEADY: not the first tick of the launch -- is_torque_on_prev already equals is_torque_on (a launch invariant), so the
// torque-edge logic of the three MyBldc joints and of the MG joint folds into per-launch constants.
// LAZY_MG: the MG joint's position-control frame is a function of this tick's target and the previous one only, and
// nobody reads it inside the launch unless a trace is attached -- the loop carries the two targets and loop_finish_mg()
// forms the frame of the last tick once.
template <int DIVC, bool MGSLOW, bool LAZY_Y0, bool STEADY, bool LAZY_MG>
RK_DEV void loop_joints(ArmLoop &a, const rk_adt_params_t &p, const ArmConsts &c, uint4 *st, int64_t n, int64_t i) {
  // ---- JointMgServo::update -> subproc_posctrl  AD_joint_mg_servo.cpp:50-73,136-149
  if(MGSLOW) {
    a.mg      = mg_update_slow(a.mg, a.tgt[1], c.mg_ctrl_time, STEADY ? c.mg_on : a.mg_prev, c.mg_on, c.mg_ini, st, n, i);
    a.mg_prev = c.mg_on;
    a.mg_pre  = a.tgt[1];
  } else if(LAZY_MG) {
    a.mg_pp  = a.mg_pre;
    a.mg_pre = a.tgt[1];
  } else {
    a.mg     = mg_posctrl_frame<DIVC>(a.tgt[1], a.mg_pre, c.mg_ctrl_time, c.mg_rcp);
    a.mg_pre = a.tgt[1];
  }
  // ---- JointMyBldcServo::update x3
#pragma unroll
  for(int s = 0; s < 3; s++) {
    const float tg = s == 0 ? a.tgt_dfl : s == 1 ? a.tgt_dfr : a.tgt[4];
    const float cl = s == 0 ? a.cl_dfl : s == 1 ? a.cl_dfr : a.cl_p3;
    RK_BLDC_FRAME(p, s == 0 ? RK_AJ_DFL : s == 1 ? RK_AJ_DFR : RK_AJ_P3, tg, cl, c.bl_ms[s], c.bl_on[s], STEADY ? c.bl_on[s] : a.bl_prev[s],
                  a.bl0[s], a.bl1[s], a.bl2[s])
    a.bl_prev[s] = c.bl_on[s];
  }
  // ---- JointIcsServo::update
  RK_ICS_UPDATE(a.tgt[0], c.dir_y0, c.y0_conn, c.y0_on, a.ics_pos, a.ics_servo)
  if(LAZY_Y0) {
    a.y0_pos  = active ? now_pos : a.y0_pos;
    a.y0_seen = a.y0_seen || active;
  } else {
    const float nn = ics_now_deg(now_pos, c.dir_y0);
    a.now_y0       = active ? nn : a.now_y0;
  }
}
RK_DEV void loop_finish_y0(ArmLoop &a, const ArmConsts &c) {
  if(a.y0_seen) a.now_y0 = ics_now_deg(a.y0_pos, c.dir_y0);
}

RK_DEV ArmConsts make_consts(const rk_adt_params_t &p, uint32_t jflags, float mg_rcp) {
  ArmConsts c;
  auto      fl = [&](int k) { return (jflags >> (4 * k)) & 0xFu; };
  c.gear_p2 = p.gear_ratio[RK_AJ_P2], c.gear_r0 = p.gear_ratio[RK_AJ_R0], c.dir_y0 = p.motor_dir[RK_AJ_Y0];
  c.mg_ctrl_time = p.ctrl_time_s[RK_AJ_P1], c.mg_rcp = mg_rcp;
  c.y0_conn = (fl(RK_AJ_Y0) & RK_AJF_CONNECTED) != 0, c.y0_on = (fl(RK_AJ_Y0) & RK_AJF_TORQUE_ON) != 0;
  c.mg_on  = (fl(RK_AJ_P1) & RK_AJF_TORQUE_ON) != 0;
  c.mg_ini = (fl(RK_AJ_P1) & RK_AJF_INITIALIZED) != 0;
  c.mg_pos = c.mg_on && c.mg_ini; // position control on every tick (the branch a running arm is in)
  const int jk[3] = {RK_AJ_DFL, RK_AJ_DFR, RK_AJ_P3};
#pragma unroll
  for(int s = 0; s < 3; s++) {
    c.bl_on[s] = (fl(jk[s]) & RK_AJF_TORQUE_ON) != 0;
    c.bl_ms[s] = bldc_ms(p.ctrl_time_s[jk[s]]);
  }
  return c;
}

RK_DEV void arm_trace_row(uint32_t *tr, int64_t n, const ArmLoop &a, uint32_t w11, uint32_t w12) {
#pragma unroll
  for(int k = 0; k < 5; k++) tr[(int64_t)k * n] = f2u(fsub(a.tgt[k], a.ofs[k]));
  tr[5 * n] = a.mg.tx0 >> 16, tr[6 * n] = a.mg.tx1;
#pragma unroll
  for(int s = 0; s < 3; s++) tr[(int64_t)(7 + s) * n] = a.bl0[s];
  tr[10 * n] = a.ics_pos;
  tr[11 * n] = w11;
  tr[12 * n] = w12;
  tr[13 * n] = bldc_id_byte(a.bl2[0]) | (bldc_id_byte(a.bl2[1]) << 8) | (bldc_id_byte(a.bl2[2]) << 16);
  tr[14 * n] = 0u, tr[15 * n] = 0u;
}

// Jumping over ticks (the untraced launch with the MG joint in position control).  Inside a segment a LAZY tick only
// advances cyc, forms tgt[0] and runs the ICS update on it (the MG targets it shifts are constant there, and the last two
// ticks of the launch, which stay real, rewrite them), so the non-final ticks of a segment can be replaced by their end
// state.  The ICS update of one tick is exact to reproduce over a window: its deg100 is a chain of RN operations with
// one fixed operand and a truncation toward zero on the remaining count, so it is monotone over the window, and tp is
// monotone in deg100.  So "active" (|deg100| <= 18000) and "send" (active, torque on, 3500 <= tp <= 11500) each hold on
// one contiguous run of ticks; the window leaves what the last sending tick and then the last active tick leave.

// the ICS joint's raw target, and the argument of its deg100 conversion, on the segment tick with remaining count r
RK_DEV float seg_tgt0(const ArmLoop &a, int32_t r) { return fadd(fsub(a.now_tgt[0], fmul(a.move[0], (float)r)), a.ofs[0]); }
RK_DEV float ics_arg(const ArmLoop &a, const ArmConsts &c, int32_t r) { return fmul(fmul(seg_tgt0(a, r), c.dir_y0), 100.0f); }
// where the tick with remaining count r lies against the interval of `active` (send = false) or of `send` (send = true):
// -1 below, 0 inside, +1 above; monotone in deg100
RK_DEV int ics_side(const ArmLoop &a, const ArmConsts &c, int32_t r, bool send) {
  const int deg100 = f2i_x86(ics_arg(a, c, r));
  if(deg100 < -18000 || deg100 > 18000) return deg100 < 0 ? -1 : 1;
  const int tp = (deg100 * 2963) / 10000 + 7500;
  return !send ? 0 : (tp < 3500 ? -1 : (tp > 11500 ? 1 : 0));
}
// the last of the window's j ticks (tick k has remaining count left - k) inside the interval, or -1: the last tick if it
// is inside; else the ticks past the same bound form a suffix, and the one before it is checked against the other bound
RK_DEV int32_t ics_last(const ArmLoop &a, const ArmConsts &c, int32_t left, int32_t j, bool send) {
  const int s = ics_side(a, c, left - (j - 1), send);
  if(s == 0) return j - 1;
  int32_t lo = 0, hi = j - 1;
#pragma unroll 1
  while(lo < hi) {
    const int32_t m = lo + (hi - lo) / 2;
    if(ics_side(a, c, left - m, send) == s) hi = m;
    else lo = m + 1;
  }
  return (lo > 0 && ics_side(a, c, left - (lo - 1), send) == 0) ? lo - 1 : -1;
}
RK_DEV void ics_window_tick(ArmLoop &a, const ArmConsts &c, int32_t r) {
  RK_ICS_UPDATE(seg_tgt0(a, r), c.dir_y0, c.y0_conn, c.y0_on, a.ics_pos, a.ics_servo)
  a.y0_pos  = active ? now_pos : a.y0_pos;
  a.y0_seen = a.y0_seen || active;
}
RK_DEV bool arm_idle(const ArmLoop &a) { return a.state == RK_ASTATE_STANDBY && a.exec == a.head; }

// The index of the next tick to run for real, after ticks [0, t) have run (`idle`: the last of them started in STANDBY
// with nothing queued).  Ticks K-2 and K-1 always run: loop_finish_mg needs their MG targets, the stored block their
// targets and frames.  An idle tick is a fixed point -- IS_COMP is set, and the ICS update of an unchanged target rewrites
// what it wrote -- so the ticks after it are skipped.  Inside a segment, the next min(cnt - cyc, K-2 - t) ticks are its
// non-final ticks, jumped over in one step unless the ICS conversion of a target at either end of the window is out of
// f2i_x86's range or NaN (huge or infinite waypoints), which breaks the monotonicity: those windows run tick by tick.
RK_DEV int loop_jump(ArmLoop &a, const ArmConsts &c, int t, int K, bool idle) {
  if(t >= K - 2) return t;
  if(idle) return K - 2;
  const int32_t left = (int32_t)((uint32_t)a.cnt - (uint32_t)a.cyc); // remaining count of the next tick
  if(a.state != RK_ASTATE_MOVING || a.cnt <= a.cyc || left <= 0) return t;
  const int32_t j = min(left, K - 2 - t), last = left - (j - 1);
  if(!(fabsf(ics_arg(a, c, left)) < 2147483648.0f && fabsf(ics_arg(a, c, last)) < 2147483648.0f)) return t;
  if(c.y0_conn) {
    const int32_t ls = c.y0_on ? ics_last(a, c, left, j, true) : -1, la = ics_last(a, c, left, j, false);
    if(ls >= 0) ics_window_tick(a, c, left - ls);
    if(la >= 0) ics_window_tick(a, c, left - la);
  }
  a.tgt[0] = seg_tgt0(a, last);
  a.mg_pp  = j > 1 ? a.tgt[1] : a.mg_pre;
  a.mg_pre = a.tgt[1];
  a.cyc += j;
  return t + j;
}

template <bool TRACE, int DIVC>
RK_DEV void adt_update_body(int64_t i, const rk_adt_params_t &p, uint4 *__restrict__ state, const uint4 *__restrict__ tab, int64_t n, int K,
                            uint32_t *__restrict__ trace, float mg_rcp) {
  ArmLoop  a;
  uint32_t jflags;
  loop_load(state, n, i, a, jflags);
  const ArmConsts c = make_consts(p, jflags, mg_rcp);
  {
    uint32_t lens = 0;
#pragma unroll
    for(int sl = 0; sl < RK_ACMD_SLOTS; sl++) lens |= (__ldg(&tab[(int64_t)sl * (RK_ACMD_SLOT_WORDS / 4) * n + i]).y & 0xFFu) << (8 * sl);
    a.lens = lens;
    // what the FSM will read first: the waypoint of a pending MOVE_START, else the one after the running segment
    uint32_t fs = a.exec, fi = a.cmd_idx & 0xFFu;
    if(a.state == RK_ASTATE_MOVING) ring_next(a, a.exec, a.cmd_idx & 0xFFu, fs, fi);
    else if(a.state != RK_ASTATE_MOVE_START) fs = (a.exec + 1 >= RK_ACMD_SLOTS) ? 0u : a.exec + 1, fi = 0u;
    ring_fetch(a, tab, n, i, fs, fi, a.sel);
    a.pf_key = ring_key(fs, fi);
  }
  // the first tick sees the stored is_torque_on_prev flags, the others run on launch constants (STEADY)
  if(c.mg_pos && !TRACE) { // one real tick per iteration, then as far as loop_jump allows
    if(K > 0) {
      bool idle = arm_idle(a);
      loop_tick<DIVC, false, false, true>(a, p, c, state, tab, n, i, K <= 2);
#pragma unroll 1
      for(int t = loop_jump(a, c, 1, K, idle); t < K; t = loop_jump(a, c, t + 1, K, idle)) {
        idle = arm_idle(a);
        loop_tick<DIVC, false, true, true>(a, p, c, state, tab, n, i, t >= K - 2);
      }
      loop_finish_mg<DIVC>(a, c);
    }
  } else if(c.mg_pos) { // every tick writes a trace row
    if(K > 0) {
      loop_tick<DIVC, false, false, false>(a, p, c, state, tab, n, i, K <= 2);
      arm_trace_row(trace + i, n, a, a.state, a.cmd_idx);
    }
#pragma unroll 1
    for(int t = 1; t < K; t++) {
      loop_tick<DIVC, false, true, false>(a, p, c, state, tab, n, i, t >= K - 2);
      arm_trace_row(trace + (int64_t)t * RK_ADT_TRACE_WORDS * n + i, n, a, a.state, a.cmd_idx);
    }
  } else {
#pragma unroll 1
    for(int t = 0; t < K; t++) {
      loop_tick<DIVC, true>(a, p, c, state, tab, n, i);
      if(TRACE) arm_trace_row(trace + (int64_t)t * RK_ADT_TRACE_WORDS * n + i, n, a, a.state, a.cmd_idx);
    }
  }
  loop_finish_y0(a, c);
  loop_store(state, n, i, a, jflags, K > 0);
}
// One thread per arm; CTAs stride over the batch when the grid is capped (see imt_update_kernel).
template <bool TRACE, int DIVC>
__global__ void __launch_bounds__(128, 5)
adt_update_kernel(const rk_adt_params_t p, uint4 *__restrict__ state, const uint4 *__restrict__ tab, int64_t n, int K,
                  uint32_t *__restrict__ trace, float mg_rcp) {
  for(int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    adt_update_body<TRACE, DIVC>(i, p, state, tab, n, K, trace, mg_rcp);
}

// ---------------------------------------------------------------------------------------------
// ADTModePositioning (AD_mode_positioning.cpp): same joints, single-command FIFO mode.
// The FIFO (front first) stays in HBM; a command start (rare) pops it there.
// ---------------------------------------------------------------------------------------------
RK_DEV float joint_now_deg(const uint4 *st, int64_t n, int64_t i, int k) { // JointBase::get_now_deg  AD_joint_base.hpp:48
  const uint4 j = ld_plane(st, n, (RK_AS_JOINT0 + 4 * k) / 4, i);
  return fsub(u2f(j.w), u2f(j.x));
}

template <bool TRACE, int DIVC>
__global__ void __launch_bounds__(128)
adp_update_kernel(const rk_adt_params_t p, uint4 *__restrict__ state, uint4 *__restrict__ ps, int64_t n, int K,
                  uint32_t *__restrict__ trace, float mg_rcp) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  ArmLoop  a;
  uint32_t jflags;
  loop_load(state, n, i, a, jflags);
  const ArmConsts c = make_consts(p, jflags, mg_rcp);
  uint4    h0 = ld_plane(ps, n, 0, i), h1 = ld_plane(ps, n, 1, i);
  uint32_t pstate = h0.x & 0xFFu, pflags = h0.x & ~0xFFu, cnt = h0.y, cyc = h0.z, qsize = h0.w;
  uint4    c0 = ld_plane(ps, n, 2, i), c1 = ld_plane(ps, n, 3, i);
  const uint4 m0 = ld_plane(ps, n, 4, i), m1 = ld_plane(ps, n, 5, i);
  uint32_t now_id = c0.x, now_dt = c0.y;
  float    now_tgt[5] = {u2f(c0.z), u2f(c0.w), u2f(c1.x), u2f(c1.y), u2f(c1.z)};
  float    move[5]    = {u2f(m0.x), u2f(m0.y), u2f(m0.z), u2f(m0.w), u2f(m1.x)};
  for(int t = 0; t < K; t++) {
    const bool was_moving = pstate == 1u; // switch(nowState): ONE handler per update  :9-20
    if(pstate == 0u) {                    // exec_standby :27-58
      pflags |= RK_AS_FSM_IS_COMP;
      if(qsize > 0) {
        c0 = ld_plane(ps, n, RK_PS_QUEUE / 4, i), c1 = ld_plane(ps, n, RK_PS_QUEUE / 4 + 1, i); // cmd_q_.front()
        for(uint32_t e = 1; e < qsize && e < 4; e++) {                                          // pop_front()
          st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (e - 1), i, ld_plane(ps, n, RK_PS_QUEUE / 4 + 2 * e, i));
          st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (e - 1) + 1, i, ld_plane(ps, n, RK_PS_QUEUE / 4 + 2 * e + 1, i));
        }
        qsize = (qsize > 4u ? 4u : qsize) - 1u;
        st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (int)qsize, i, make_uint4(0u, 0u, 0u, 0u)); // entries past size() are kept zero
        st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (int)qsize + 1, i, make_uint4(0u, 0u, 0u, 0u));
        now_id = c0.x, now_dt = c0.y;
        now_tgt[0] = u2f(c0.z), now_tgt[1] = u2f(c0.w), now_tgt[2] = u2f(c1.x), now_tgt[3] = u2f(c1.y), now_tgt[4] = u2f(c1.z);
        cnt = (uint32_t)f2i_x86(fdiv(fmul(__uint2float_rn(now_dt), 0.001f), p.cycle_time_s));
        cnt = (cnt == 0u) ? 1u : cnt;
        const float fc = __uint2float_rn(cnt);
        // get_now_deg() of the five axes; J2 / J3 through the differential (AD_joint_dfgear.hpp:76-77,98)
        const float ln = joint_now_deg(state, n, i, RK_AJ_DFL), rn = joint_now_deg(state, n, i, RK_AJ_DFR);
        const float ofs_p2 = a.ofs[2], ofs_r0 = a.ofs[3];
        float       now[5];
        now[0] = fsub(a.now_y0, a.ofs[0]);
        now[1] = joint_now_deg(state, n, i, RK_AJ_P1);
        now[2] = fsub(fdiv(fmul(fsub(ln, rn), 0.5f), p.gear_ratio[RK_AJ_P2]), ofs_p2);
        now[3] = fsub(fdiv(fmul(-fadd(ln, rn), 0.5f), p.gear_ratio[RK_AJ_R0]), ofs_r0);
        now[4] = joint_now_deg(state, n, i, RK_AJ_P3);
#pragma unroll
        for(int k = 0; k < 5; k++) move[k] = fdiv(fsub(now_tgt[k], now[k]), fc);
        cyc = 0;
        pflags &= ~RK_AS_FSM_IS_COMP;
        pstate = 1u;
      }
    }
    // exec_moving :64-110 (only when the update STARTED in MOVING)
    loop_set_targets(a, c, was_moving, __uint2float_rn(cnt - cyc), now_tgt, move);
    if(was_moving) {
      if(cnt <= cyc) {
        h1.y = h1.x, h1.x = now_id; // u32_prev_cmd_id_
        pstate = 0u;
      } else {
        cyc++;
      }
    }
    if(c.mg_pos) loop_joints<DIVC, false>(a, p, c, state, n, i);
    else loop_joints<DIVC, true>(a, p, c, state, n, i);
    if(TRACE) arm_trace_row(trace + (int64_t)t * RK_ADT_TRACE_WORDS * n + i, n, a, pstate, qsize);
  }
  loop_store(state, n, i, a, jflags, K > 0);
  st_plane(ps, n, 0, i, make_uint4(pstate | pflags, cnt, cyc, qsize));
  st_plane(ps, n, 1, i, h1);
  st_plane(ps, n, 2, i, make_uint4(now_id, now_dt, f2u(now_tgt[0]), f2u(now_tgt[1])));
  st_plane(ps, n, 3, i, make_uint4(f2u(now_tgt[2]), f2u(now_tgt[3]), f2u(now_tgt[4]), c1.w));
  st_plane(ps, n, 4, i, make_uint4(f2u(move[0]), f2u(move[1]), f2u(move[2]), f2u(move[3])));
  st_plane(ps, n, 5, i, make_uint4(f2u(move[4]), m1.y, m1.z, m1.w));
}

// ---------------------------------------------------------------------------------------------
// Homing modes: ADTModeInitialize (AD_mode_initialize.cpp) and ADTModeInitPosMove (AD_mode_initpos_move.cpp).
// They rewrite what the positioning tick treats as launch constants (torque / initialised flags, current limits,
// offsets), and run once per power-up, so this is a plain transcription: the whole arm block lives in registers
// as words (every index below is a compile-time constant), and the servo updates run the sequence tick's servo code
// on it.
// ---------------------------------------------------------------------------------------------
// plane pl of a block held as words, and a whole block of W words (W / 4 planes) to and from registers
RK_DEV uint4 w_plane(const uint32_t *w, int pl) { return make_uint4(w[4 * pl], w[4 * pl + 1], w[4 * pl + 2], w[4 * pl + 3]); }
RK_DEV void  w_set_plane(uint32_t *w, int pl, uint4 v) { w[4 * pl] = v.x, w[4 * pl + 1] = v.y, w[4 * pl + 2] = v.z, w[4 * pl + 3] = v.w; }
template <int W> RK_DEV void ld_words(const uint4 *blk, int64_t n, int64_t i, uint32_t (&w)[W]) {
#pragma unroll
  for(int pl = 0; pl < W / 4; pl++) w_set_plane(w, pl, ld_plane(blk, n, pl, i));
}
template <int W> RK_DEV void st_words(uint4 *blk, int64_t n, int64_t i, const uint32_t (&w)[W]) {
#pragma unroll
  for(int pl = 0; pl < W / 4; pl++) st_plane(blk, n, pl, i, w_plane(w, pl));
}
#define AJW(w, k, f) ((w)[RK_AS_JOINT0 + 4 * (k) + (f)])
RK_DEV uint32_t hj_flag(const uint32_t *w, int k) { return (w[RK_AS_JFLAGS] >> (4 * k)) & 0xFu; }
RK_DEV void     hj_set_flag(uint32_t *w, int k, uint32_t b) { w[RK_AS_JFLAGS] = (w[RK_AS_JFLAGS] & ~(0xFu << (4 * k))) | (b << (4 * k)); }
RK_DEV void     hj_set_bit(uint32_t *w, int k, uint32_t bit, bool on) { hj_set_flag(w, k, (hj_flag(w, k) & ~bit) | (on ? bit : 0u)); }
RK_DEV float    hj_absf(float x) { return (x < 0.0f) ? -x : x; } // mymath::absf  util_mymath.hpp:40

template <int AX> RK_DEV float hj_get_tgt(const uint32_t *w) { // JointBase::get_tgt_deg :47
  return fsub(u2f(AJW(w, axis_joint(AX), RK_AJ_RAW_TGT)), u2f(AJW(w, axis_joint(AX), RK_AJ_OFS)));
}
template <int AX> RK_DEV float hj_get_now(const rk_adt_params_t &p, const uint32_t *w) { // ::get_now_deg :48; DfGear :76-77,98
  constexpr int k = axis_joint(AX);
  if(k == RK_AJ_P2 || k == RK_AJ_R0) {
    const float ln = fsub(u2f(AJW(w, RK_AJ_DFL, RK_AJ_RAW_NOW)), u2f(AJW(w, RK_AJ_DFL, RK_AJ_OFS)));
    const float rn = fsub(u2f(AJW(w, RK_AJ_DFR, RK_AJ_RAW_NOW)), u2f(AJW(w, RK_AJ_DFR, RK_AJ_OFS)));
    const float m  = (k == RK_AJ_P2) ? fsub(ln, rn) : -fadd(ln, rn);
    return fsub(fdiv(fmul(m, 0.5f), p.gear_ratio[k]), u2f(AJW(w, k, RK_AJ_OFS)));
  }
  return fsub(u2f(AJW(w, k, RK_AJ_RAW_NOW)), u2f(AJW(w, k, RK_AJ_OFS)));
}
template <int AX> RK_DEV void hj_set_tgt(const rk_adt_params_t &p, uint32_t *w, float tgt) { // ::set_tgt_ang_deg :42; DfGear :14-37,60-63,93-96
  constexpr int k = axis_joint(AX);
  const float   raw = fadd(tgt, u2f(AJW(w, k, RK_AJ_OFS)));
  AJW(w, k, RK_AJ_RAW_TGT) = f2u(raw);
  if(k == RK_AJ_P2 || k == RK_AJ_R0) {
    if(k == RK_AJ_P2) w[RK_AS_DFV_P] = f2u(fmul(raw, p.gear_ratio[k]));
    else w[RK_AS_DFV_R] = f2u(fmul(raw, p.gear_ratio[k]));
    const float P = u2f(w[RK_AS_DFV_P]), R = u2f(w[RK_AS_DFV_R]);
    AJW(w, RK_AJ_DFL, RK_AJ_RAW_TGT) = f2u(fadd(fsub(P, R), u2f(AJW(w, RK_AJ_DFL, RK_AJ_OFS))));
    AJW(w, RK_AJ_DFR, RK_AJ_RAW_TGT) = f2u(fadd(-fadd(P, R), u2f(AJW(w, RK_AJ_DFR, RK_AJ_OFS))));
  }
}
template <int AX> RK_DEV void hj_set_torque_on(uint32_t *w, bool on) { // :39; DfGear forwards to both motors :50-53
  constexpr int k = axis_joint(AX);
  if(k == RK_AJ_P2 || k == RK_AJ_R0) hj_set_bit(w, RK_AJ_DFL, RK_AJF_TORQUE_ON, on), hj_set_bit(w, RK_AJ_DFR, RK_AJF_TORQUE_ON, on);
  else hj_set_bit(w, k, RK_AJF_TORQUE_ON, on);
}
template <int AX> RK_DEV void hj_set_curlim(uint32_t *w, float lim) { // :43; DfGear forwards :55-58
  constexpr int k = axis_joint(AX);
  if(k == RK_AJ_P2 || k == RK_AJ_R0) AJW(w, RK_AJ_DFL, RK_AJ_CURLIM) = f2u(lim), AJW(w, RK_AJ_DFR, RK_AJ_CURLIM) = f2u(lim);
  else AJW(w, k, RK_AJ_CURLIM) = f2u(lim);
}
template <int AX> RK_DEV void hj_mech_reset(const rk_adt_params_t &p, uint32_t *w) { // :36-38; DfGear :65-71,100-106
  constexpr int k = axis_joint(AX);
  if(k == RK_AJ_P2) { // the pitch joint resets both motors, the roll joint does not
    AJW(w, RK_AJ_DFL, RK_AJ_OFS) = f2u(fsub(u2f(AJW(w, RK_AJ_DFL, RK_AJ_RAW_NOW)), p.mechend_pos_deg[RK_AJ_DFL]));
    AJW(w, RK_AJ_DFR, RK_AJ_OFS) = f2u(fsub(u2f(AJW(w, RK_AJ_DFR, RK_AJ_RAW_NOW)), p.mechend_pos_deg[RK_AJ_DFR]));
  }
  AJW(w, k, RK_AJ_OFS) = f2u(fsub(u2f(AJW(w, k, RK_AJ_RAW_NOW)), p.mechend_pos_deg[k]));
}
template <int AX> RK_DEV void hj_joint_init(const rk_adt_params_t &p, uint32_t *w) { // JointBase::init() and its overrides
  constexpr int k = axis_joint(AX);
  if(k == RK_AJ_Y0) { // JointIcsServo::init  AD_joint_ics_servo.cpp:35-55 over the ideal servo (setFree answers the last position)
    const float now = ics_now_deg((int)(int32_t)w[RK_AS_ICS_SERVO] + 7500, p.motor_dir[RK_AJ_Y0]);
    AJW(w, k, RK_AJ_RAW_NOW) = f2u(now), AJW(w, k, RK_AJ_RAW_TGT) = f2u(now);
    w[RK_AS_ICS_POS] = 0xFFFFFFFFu;
    hj_set_bit(w, k, RK_AJF_CONNECTED, true);
  } else if(k == RK_AJ_P1) { // JointMgServo::init  AD_joint_mg_servo.cpp:38-48
    hj_set_flag(w, k, (hj_flag(w, k) & ~(RK_AJF_TORQUE_PREV | RK_AJF_TORQUE_ON)) | RK_AJF_CONNECTED);
    w[RK_AS_MG_CTRL + 7] = 1u; // set_myctrl_gain_params(InitGain): gains, and set_VelLpf_CutOff resets the IIR
    w[RK_AS_MG_CTRL + 2] = 0u, w[RK_AS_MG_CTRL + 3] = 0u;
  }
}
// exec_move_initpos of either mode (AD_mode_initialize.cpp:113-143 / AD_mode_initpos_move.cpp:70-95), one axis
template <int AX> RK_DEV bool hj_ramp_axis(const rk_adt_params_t &p, uint32_t *w, float dir_vel) {
  constexpr int k = axis_joint(AX);
  const float initpos = p.initpos_deg[k], nowpos = hj_get_tgt<AX>(w);
  const float vel     = fmul(dir_vel, hj_absf(p.vel_init_degps[k]));
  float       tgtpos  = fadd(nowpos, fmul(vel, p.cycle_time_s));
  const bool  arrived = ((vel > 0.0f) && (tgtpos > initpos)) || ((vel < 0.0f) && (tgtpos < initpos));
  if(arrived) tgtpos = initpos;
  hj_set_tgt<AX>(p, w, tgtpos);
  hj_set_curlim<AX>(w, p.curlim_default_A[k]);
  return arrived;
}
template <int AX> RK_DEV void hj_move_mechend(const rk_adt_params_t &p, uint32_t *w) { // ax_move_mechend :150-167
  constexpr int k = axis_joint(AX);
  const float vel = p.vel_init_degps[k], nowpos = hj_get_now<AX>(p, w), tgtpos = hj_get_tgt<AX>(w);
  if(hj_absf(fsub(nowpos, tgtpos)) > 45.0f) hj_set_tgt<AX>(p, w, tgtpos); // gone too far: hold
  else hj_set_tgt<AX>(p, w, fadd(tgtpos, fmul(vel, p.cycle_time_s)));
  hj_set_curlim<AX>(w, p.curlim_init_A[k]);
}
template <int AX> RK_DEV void hj_reset_angle(const rk_adt_params_t &p, uint32_t *w) { // ax_reset_angle :174-179
  hj_mech_reset<AX>(p, w);
  hj_set_tgt<AX>(p, w, hj_get_now<AX>(p, w));
}
template <int AX> RK_DEV bool hj_init_ramp(const rk_adt_params_t &p, uint32_t *w) {
  const float d = fsub(p.initpos_deg[axis_joint(AX)], hj_get_tgt<AX>(w));
  hj_set_bit(w, axis_joint(AX), RK_AJF_INITIALIZED, true);
  return hj_ramp_axis<AX>(p, w, (d >= 0.0f) ? 1.0f : -1.0f);
}
template <int AX> RK_DEV void hj_ipm_init(const rk_adt_params_t &p, uint32_t *w, uint32_t *hw) { // ADTModeInitPosMove::exec_init :37-45
  hj_set_tgt<AX>(p, w, hj_get_now<AX>(p, w));
  hw[RK_HS_VEL_DIR + AX] = f2u((p.initpos_deg[axis_joint(AX)] >= hj_get_now<AX>(p, w)) ? 1.0f : -1.0f);
}

RK_DEV void hj_mode_update(const rk_adt_params_t &p, uint32_t *w, uint32_t *hw) {
  uint32_t       state = hw[RK_HS_STATE] & 0xFFu, comp = hw[RK_HS_STATE] & RK_AS_FSM_IS_COMP;
  const uint32_t mode  = hw[RK_HS_STATE] >> 16;
  uint32_t       cnt   = hw[RK_HS_WAIT_CNT] & 0xFFFFu;
  const bool     torque_state = state == 1u && (mode == RK_ADH_MODE_INIT || mode == RK_ADH_MODE_INIT_POS_MOVE);
  if(torque_state) { // exec_torqueon of both modes
    if(cnt == 0u) {
      hj_set_torque_on<0>(w, true), hj_set_torque_on<1>(w, true), hj_set_torque_on<2>(w, true), hj_set_torque_on<3>(w, true), hj_set_torque_on<4>(w, true);
      cnt++;
    } else if(cnt == 100u) state = 2u, cnt = 0u;
    else cnt++;
  } else if(mode == RK_ADH_MODE_INIT) {
    if(state == 0u) { // exec_init :43-50
      hj_joint_init<0>(p, w), hj_joint_init<1>(p, w);
      hj_set_bit(w, RK_AJ_Y0, RK_AJF_INITIALIZED, false), hj_set_bit(w, RK_AJ_P1, RK_AJF_INITIALIZED, false);
      hj_set_bit(w, RK_AJ_P2, RK_AJF_INITIALIZED, false), hj_set_bit(w, RK_AJ_R0, RK_AJF_INITIALIZED, false);
      hj_set_bit(w, RK_AJ_P3, RK_AJF_INITIALIZED, false);
      state = 1u;
    } else if(state == 2u) { // exec_move_mechend :79-94
      if(cnt < 500u) {
        hj_move_mechend<1>(p, w);
        hj_move_mechend<4>(p, w);
        cnt++;
      } else if(cnt == 500u) state = 3u, cnt = 0u;
    } else if(state == 3u) { // exec_resetangle :100-109
      hj_reset_angle<1>(p, w), hj_reset_angle<2>(p, w), hj_reset_angle<3>(p, w), hj_reset_angle<4>(p, w);
      state = 4u;
    } else if(state == 4u) { // exec_move_initpos :115-143
      bool all = hj_init_ramp<0>(p, w);
      all &= hj_init_ramp<1>(p, w);
      all &= hj_init_ramp<2>(p, w);
      all &= hj_init_ramp<3>(p, w);
      all &= hj_init_ramp<4>(p, w);
      if(all) state = 5u;
    } else if(state == 5u) comp = RK_AS_FSM_IS_COMP;
  } else if(mode == RK_ADH_MODE_INIT_POS_MOVE) {
    if(state == 0u) {
      hj_ipm_init<0>(p, w, hw), hj_ipm_init<1>(p, w, hw), hj_ipm_init<2>(p, w, hw), hj_ipm_init<3>(p, w, hw), hj_ipm_init<4>(p, w, hw);
      state = 1u;
    } else if(state == 2u) { // exec_move_initpos :73-95
      bool all = hj_ramp_axis<0>(p, w, u2f(hw[RK_HS_VEL_DIR + 0]));
      all &= hj_ramp_axis<1>(p, w, u2f(hw[RK_HS_VEL_DIR + 1]));
      all &= hj_ramp_axis<2>(p, w, u2f(hw[RK_HS_VEL_DIR + 2]));
      all &= hj_ramp_axis<3>(p, w, u2f(hw[RK_HS_VEL_DIR + 3]));
      all &= hj_ramp_axis<4>(p, w, u2f(hw[RK_HS_VEL_DIR + 4]));
      if(all) state = 3u;
    } else if(state == 3u) comp = RK_AS_FSM_IS_COMP;
  }
  hw[RK_HS_STATE]    = state | comp | (mode << 16);
  hw[RK_HS_WAIT_CNT] = cnt;
}

// JointMgServo::update on the word block: all four branches  AD_joint_mg_servo.cpp:50-73
RK_DEV void hj_mg_update(const rk_adt_params_t &p, uint32_t *w) {
  const uint32_t b = hj_flag(w, RK_AJ_P1);
  const bool     on = (b & RK_AJF_TORQUE_ON) != 0, prev = (b & RK_AJF_TORQUE_PREV) != 0, ini = (b & RK_AJF_INITIALIZED) != 0;
  const float    tgt = u2f(AJW(w, RK_AJ_P1, RK_AJ_RAW_TGT)), ct = p.ctrl_time_s[RK_AJ_P1];
  MgFrame        f   = {w[RK_AS_MG_TX], w[RK_AS_MG_TX + 1], w[RK_AS_MG_TX + 2]};
  if(on && ini) {
    f = mg_posctrl_frame<0>(tgt, u2f(w[RK_AS_MG_PRE_TGT]), ct, 0.0f);
  } else {
    uint4 q0 = w_plane(w, RK_AS_MG_CTRL / 4), q1 = w_plane(w, RK_AS_MG_CTRL / 4 + 1);
    f        = mg_torque_ctrl(f, q0, q1, w_plane(w, (RK_AS_JOINT0 + 4 * RK_AJ_P1) / 4), tgt, ct, prev, on, ini);
    w_set_plane(w, RK_AS_MG_CTRL / 4, q0), w_set_plane(w, RK_AS_MG_CTRL / 4 + 1, q1);
  }
  w[RK_AS_MG_TX] = f.tx0, w[RK_AS_MG_TX + 1] = f.tx1, w[RK_AS_MG_TX + 2] = f.valid;
  hj_set_bit(w, RK_AJ_P1, RK_AJF_TORQUE_PREV, on);
  w[RK_AS_MG_PRE_TGT] = f2u(tgt);
}
// JointMyBldcServo::update on the word block
template <int SLOT> RK_DEV void hj_bldc_update(const rk_adt_params_t &p, uint32_t *w) {
  constexpr int  k  = SLOT == 0 ? RK_AJ_DFL : SLOT == 1 ? RK_AJ_DFR : RK_AJ_P3;
  const uint32_t b  = hj_flag(w, k);
  const bool     on = (b & RK_AJF_TORQUE_ON) != 0;
  uint32_t      *q  = w + RK_AS_BLDC_TX0 + 4 * SLOT;
  RK_BLDC_FRAME(p, k, u2f(AJW(w, k, RK_AJ_RAW_TGT)), u2f(AJW(w, k, RK_AJ_CURLIM)), bldc_ms(p.ctrl_time_s[k]), on, (b & RK_AJF_TORQUE_PREV) != 0,
                q[0], q[1], q[2])
  q[3] = 1u;
  hj_set_bit(w, k, RK_AJF_TORQUE_PREV, on);
}
// JointIcsServo::update on the word block
RK_DEV void hj_ics_update(const rk_adt_params_t &p, uint32_t *w) {
  const uint32_t b = hj_flag(w, RK_AJ_Y0);
  RK_ICS_UPDATE(u2f(AJW(w, RK_AJ_Y0, RK_AJ_RAW_TGT)), p.motor_dir[RK_AJ_Y0], (b & RK_AJF_CONNECTED) != 0, (b & RK_AJF_TORQUE_ON) != 0,
                w[RK_AS_ICS_POS], w[RK_AS_ICS_SERVO])
  if(active) AJW(w, RK_AJ_Y0, RK_AJ_RAW_NOW) = f2u(ics_now_deg(now_pos, p.motor_dir[RK_AJ_Y0]));
}

template <bool TRACE>
__global__ void __launch_bounds__(128)
adh_update_kernel(const rk_adt_params_t p, uint4 *__restrict__ state, uint4 *__restrict__ hs, int64_t n, int K,
                  const float *__restrict__ now, uint32_t *__restrict__ trace) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  uint32_t w[RK_AS_WORDS], hw[RK_HS_WORDS];
  ld_words(state, n, i, w);
  ld_words(hs, n, i, hw);
#pragma unroll 1
  for(int t = 0; t < K; t++) {
    if(now) { // what the CAN rx callbacks stored since the last tick
      const float *f = now + (int64_t)t * 4 * n + i;
      AJW(w, RK_AJ_P1, RK_AJ_RAW_NOW) = f2u(__ldcs(f)), AJW(w, RK_AJ_DFL, RK_AJ_RAW_NOW) = f2u(__ldcs(f + n));
      AJW(w, RK_AJ_DFR, RK_AJ_RAW_NOW) = f2u(__ldcs(f + 2 * n)), AJW(w, RK_AJ_P3, RK_AJ_RAW_NOW) = f2u(__ldcs(f + 3 * n));
    }
    hj_mode_update(p, w, hw);
    hj_mg_update(p, w);
    hj_bldc_update<0>(p, w), hj_bldc_update<1>(p, w), hj_bldc_update<2>(p, w);
    hj_ics_update(p, w);
    if(TRACE) {
      uint32_t *tr = trace + (int64_t)t * RK_ADT_TRACE_WORDS * n + i;
      tr[0] = f2u(hj_get_tgt<0>(w)), tr[n] = f2u(hj_get_tgt<1>(w)), tr[2 * n] = f2u(hj_get_tgt<2>(w));
      tr[3 * n] = f2u(hj_get_tgt<3>(w)), tr[4 * n] = f2u(hj_get_tgt<4>(w));
      tr[5 * n] = w[RK_AS_MG_TX] >> 16, tr[6 * n] = w[RK_AS_MG_TX + 1];
      tr[7 * n] = w[RK_AS_BLDC_TX0], tr[8 * n] = w[RK_AS_BLDC_TX0 + 4], tr[9 * n] = w[RK_AS_BLDC_TX0 + 8];
      tr[10 * n] = w[RK_AS_ICS_POS];
      tr[11 * n] = hw[RK_HS_STATE] & 0xFFu, tr[12 * n] = hw[RK_HS_WAIT_CNT];
      tr[13 * n] = bldc_id_byte(w[RK_AS_BLDC_TX0 + 2]) | (bldc_id_byte(w[RK_AS_BLDC_TX0 + 6]) << 8) | (bldc_id_byte(w[RK_AS_BLDC_TX0 + 10]) << 16);
      tr[14 * n] = 0u, tr[15 * n] = 0u;
    }
  }
  st_words(state, n, i, w);
  st_words(hs, n, i, hw);
}
__global__ void __launch_bounds__(128) adh_mode_init_kernel(uint4 *__restrict__ hs, int64_t n, uint32_t mode) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  // ADTModeBase::init(): is_comp = false; doInit(): nowState = INIT, u16_wait_cnt_ = 0, flags / directions zeroed
  st_plane(hs, n, 0, i, make_uint4(mode << 16, 0u, 0u, 0u));
  st_plane(hs, n, 1, i, make_uint4(0u, 0u, 0u, 0u));
  st_plane(hs, n, 2, i, make_uint4(0u, 0u, 0u, 0u));
}

__global__ void __launch_bounds__(128) adp_mode_init_kernel(uint4 *__restrict__ ps, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  uint4 h = ld_plane(ps, n, 0, i);
  h.x     = 0u; // is_comp = false; nowState = STANDBY
  st_plane(ps, n, 0, i, h);
}

// ADTModePositioning::push_cmd :118-124
__global__ void __launch_bounds__(128) adp_push_kernel(uint4 *__restrict__ ps, int64_t n, const uint4 *__restrict__ cmd, const uint8_t *__restrict__ valid) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  if(valid && !valid[i]) return;
  uint4    h     = ld_plane(ps, n, 0, i);
  uint32_t qsize = h.w > 4u ? 4u : h.w;
  if(qsize >= 4u) { // pop_front()
    for(int e = 1; e < 4; e++) {
      st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (e - 1), i, ld_plane(ps, n, RK_PS_QUEUE / 4 + 2 * e, i));
      st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (e - 1) + 1, i, ld_plane(ps, n, RK_PS_QUEUE / 4 + 2 * e + 1, i));
    }
    qsize = 3u;
  }
  uint4 c1 = __ldcs(cmd + n + i);
  c1.w     = 0u;
  st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (int)qsize, i, __ldcs(cmd + i));
  st_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (int)qsize + 1, i, c1);
  h.w = qsize + 1u;
  st_plane(ps, n, 0, i, h);
}

// ADTModePositioning::get_q_cmd_status :134-148
__global__ void __launch_bounds__(128) adp_status_kernel(const uint4 *__restrict__ ps, int64_t n, const uint32_t *__restrict__ ids, int32_t *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  const uint4    h = ld_plane(ps, n, 0, i), h1 = ld_plane(ps, n, 1, i);
  const uint32_t id = ids[i], qsize = h.w > 4u ? 4u : h.w;
  int32_t        sts = 0x63;
  for(uint32_t e = 0; e < qsize; e++)
    if(ld_plane(ps, n, RK_PS_QUEUE / 4 + 2 * (int)e, i).x == id) sts = 0;
  if(h1.x == id || h1.y == id) sts = 1;
  out[i] = sts;
}

// prepare_task() + a finished INIT mode + ADTModeBase::init() -> doInit()
// (AD_task_main.cpp:170-193, AD_mode_initialize.cpp:58-63,133-135, AD_mode_positioning_seq.cpp:5-11)
__global__ void __launch_bounds__(128) adt_mode_init_kernel(const rk_adt_params_t p, uint4 *__restrict__ state, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  uint32_t w[RK_AS_WORDS];
  ld_words(state, n, i, w);
  hj_joint_init<0>(p, w); // JointIcsServo::init: free command, target := present position
  hj_joint_init<1>(p, w); // JointMgServo::init: InitGain, whose set_VelLpf_CutOff() resets the IIR
  const uint32_t all = RK_AJF_CONNECTED | RK_AJF_TORQUE_ON | RK_AJF_INITIALIZED;
  hj_set_flag(w, RK_AJ_Y0, all), hj_set_flag(w, RK_AJ_P1, all); // JointMgServo::init clears torque_on_prev
  hj_set_torque_on<2>(w, true), hj_set_torque_on<4>(w, true);
  hj_set_bit(w, RK_AJ_P2, RK_AJF_INITIALIZED, true), hj_set_bit(w, RK_AJ_R0, RK_AJF_INITIALIZED, true);
  hj_set_bit(w, RK_AJ_P3, RK_AJF_INITIALIZED, true);
  hj_set_curlim<0>(w, p.curlim_default_A[RK_AJ_Y0]), hj_set_curlim<1>(w, p.curlim_default_A[RK_AJ_P1]);
  hj_set_curlim<3>(w, p.curlim_default_A[RK_AJ_R0]); // J3 (Roll) is the last to set both motors
  hj_set_curlim<4>(w, p.curlim_default_A[RK_AJ_P3]);
  w[RK_AS_FSM]     = RK_ASTATE_STANDBY | RK_AS_FSM_FIRSTCALL;
  w[RK_AS_SEQ_IDX] = (RK_ACMD_SLOTS - 1) | ((RK_ACMD_SLOTS - 1) << 16); // exec = head: nothing queued
  st_words(state, n, i, w);
}

// ADTModePositioningSeq::push_cmdseq   AD_mode_positioning_seq.cpp:124-137
__global__ void __launch_bounds__(128)
adt_push_kernel(uint4 *__restrict__ state, uint4 *__restrict__ tab, int64_t n, const uint4 *__restrict__ seq, const uint8_t *__restrict__ valid) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  if(valid && !valid[i]) return;
  uint4          s0   = ld_plane(state, n, 0, i);
  const uint32_t exec = s0.y & 0xFFFFu, head = s0.y >> 16;
  uint32_t       nw   = (head + 1) & 0xFFFFu;
  nw                  = (nw >= RK_ACMD_SLOTS) ? 0u : nw;
  if(nw == exec) return; // ring full: dropped silently
  const int base = (int)nw * (RK_ACMD_SLOT_WORDS / 4);
  for(int pl = 0; pl < RK_ACMD_SLOT_WORDS / 4; pl++) {
    uint4 v = __ldcs(seq + (int64_t)pl * n + i);
    if(pl == 0) v.y &= 0xFFu; // u8_cmd_seq_len
    tab[(int64_t)(base + pl) * n + i] = v;
  }
  s0.y = exec | (nw << 16);
  st_plane(state, n, 0, i, s0);
}

// ADTModePositioningSeq::get_q_cmdseq_status   AD_mode_positioning_seq.cpp:146-184
__global__ void __launch_bounds__(128)
adt_status_kernel(const uint4 *__restrict__ state, const uint4 *__restrict__ tab, int64_t n, const uint32_t *__restrict__ ids, int32_t *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  const uint4    s0   = ld_plane(state, n, 0, i);
  const uint32_t exec = s0.y & 0xFFFFu, head = s0.y >> 16, id = ids[i];
  int32_t        sts  = 99;
  if((s0.x & RK_AS_FSM_FIRSTCALL) && id == 0) {
    out[i] = 99;
    return;
  }
#pragma unroll
  for(uint32_t s = 0; s < RK_ACMD_SLOTS; s++) {
    if(__ldg(&tab[(int64_t)s * (RK_ACMD_SLOT_WORDS / 4) * n + i]).x != id) continue;
    if(exec == head) {
      const uint32_t len = __ldg(&tab[(int64_t)(exec % RK_ACMD_SLOTS) * (RK_ACMD_SLOT_WORDS / 4) * n + i]).y & 0xFFu;
      sts                = ((s0.z & 0xFFu) >= len) ? 1 : 0;
    } else if(exec < head) {
      sts = (exec <= s && s <= head) ? 0 : 1;
    } else {
      sts = ((exec <= s && s < RK_ACMD_SLOTS) || s <= head) ? 0 : 1;
    }
  }
  out[i] = sts;
}

// JointBase::get_tgt_deg() of the five mode axes (AD_joint_base.hpp:47)
__global__ void adt_targets_kernel(const uint4 *__restrict__ state, int64_t n, int64_t i, float *__restrict__ out5) {
  if(threadIdx.x != 0 || blockIdx.x != 0) return;
  uint32_t w[RK_AS_WORDS];
  ld_words(state, n, i, w);
  out5[0] = hj_get_tgt<0>(w), out5[1] = hj_get_tgt<1>(w), out5[2] = hj_get_tgt<2>(w), out5[3] = hj_get_tgt<3>(w), out5[4] = hj_get_tgt<4>(w);
}

} // namespace rk

namespace rk {
// ---------------------------------------------------------------------------------------------
// Servo feedback (SURVEY 8f-3, arm side): the CAN rx callbacks of the arm's servos, one frame per arm.
// KIND 0..2: JointMyBldcServo::rx_callback -> rx_summary_status of DF_Left / DF_Right / P3
//   (AD_joint_mybldc_servo.cpp:45-70; RES_STATUS_SUMMAY AD_joint_mybldc_servo.hpp:49-60: byte 0 flags, 1 mode,
//   2..3 s16_out_ang_deg_Q4, 4 s8_motor_curr_A_Q4); ids other than CMD_ID_RES_STATUS_SUMMARY are ignored.
// KIND 3: JointMgServo::rx_callback (AD_joint_mg_servo.cpp:75-92): 0x9C / 0xA1 -> the current through the
//   double-precision quadratic conv_raw_to_current (AD_joint_mg_servo.hpp:120-128); 0x92 -> the multi-turn angle.
//   The firmware assembles it as `u64 |= u8_ang[i] << (i * 8)`, i = 0..6, the byte promoted to a 32-bit int: shifts of
//   32 and more are undefined in C++.  A Cortex-M7 register shift by >= 32 gives 0 and the i = 3 term sign-extends,
//   so the value is the sign-extended low 32 bits -- restated here.  (The x86 build masks the count to 5 bits; the
//   two agree whenever bytes 5..7 of the frame are zero, which is where the compiled reference pins this.)
// The joint's fl_raw_now_deg is stored; fl_raw_tgt_deg follows it while torque is off; fl_out_now_cur, which
// nothing on the tick reads, goes to the optional cur[] (left untouched by frames that carry no current).
// ---------------------------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(128)
adt_rx_kernel(const rk_adt_params_t p, uint4 *__restrict__ state, int64_t n, const unsigned long long *__restrict__ frames,
              const uint32_t *__restrict__ cmdid, float *__restrict__ cur) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  constexpr int  k  = KIND == 0 ? RK_AJ_DFL : KIND == 1 ? RK_AJ_DFR : KIND == 2 ? RK_AJ_P3 : RK_AJ_P1;
  const uint64_t f  = frames[i];
  const uint32_t lo = (uint32_t)f, hi = (uint32_t)(f >> 32);
  const int      pl = (RK_AS_JOINT0 + 4 * k) / 4;
  const bool     on = ((ld_plane(state, n, RK_AS_JFLAGS / 4, i).x >> (4 * k)) & RK_AJF_TORQUE_ON) != 0;
  bool           have_now = false;
  float          now      = 0.0f;
  if(KIND < 3) {
    if((cmdid ? cmdid[i] : 0x1000u) != 0x1000u) return;
    now      = fmul(fdiv(fdiv((float)hi16(lo), 16.0f), p.gear_ratio[k]), p.motor_dir[k]);
    have_now = true;
    if(cur) cur[i] = fmul(fdiv((float)(int32_t)(int8_t)(hi & 0xFFu), 16.0f), p.motor_dir[k]);
  } else {
    const uint32_t cmd = lo & 0xFFu;
    if(cmd == 0x92u) {
      const int32_t a32 = (int32_t)((lo >> 8) | (hi << 24)); // bytes 1..4, little-endian
      const int64_t ang = (int64_t)((uint64_t)(int64_t)a32 << 8);
      const float   dbf = -1.0f / 100.0f / 10.0f / 256.0f;   // DB_ANG_RAW_TO_DEG: float arithmetic, then widened
      now      = __double2float_rn(__dmul_rn((double)ang, (double)dbf));
      have_now = true;
    } else if(cmd == 0x9Cu || cmd == 0xA1u) {
      const double C_A = 0.0000057204, C_B = -0.0000485371, raw = (double)hi16(lo); // s16_iq = bytes 2..3
      double       c;
      if(raw >= 0) c = __dadd_rn(__dmul_rn(__dmul_rn(C_A, raw), raw), __dmul_rn(C_B, raw));
      else c = -__dsub_rn(__dmul_rn(__dmul_rn(C_A, raw), raw), __dmul_rn(C_B, raw));
      if(cur) cur[i] = fmul(-1.0f, __double2float_rn(c));
    }
  }
  if(have_now) {
    uint4 j = ld_plane(state, n, pl, i);
    j.w     = f2u(now);
    if(!on) j.y = f2u(now);
    st_plane(state, n, pl, i, j);
  }
}

} // namespace rk

using namespace rk;

extern "C" {

void rk_adt_default_params(rk_adt_params_t *p) {
  if(!p) return;
  // AD_task_main.cpp:38-107 in RK_AJ_* order (Y0, P1, DF_Left, DF_Right, P2, R0, P3)
  const float gear[RK_AJ_NUM] = {1.0f, 1.0f, 1.0f, 1.0f, 24.0f / 7.0f, 48.0f / 7.0f, 48.0f / 19.0f};
  const float dir[RK_AJ_NUM]  = {-1.0f, 1.0f, 1.0f, 1.0f, 1.0f, 1.0f, -1.0f};
  const float cl[RK_AJ_NUM]   = {3.0f, 0.7f, 0.5f, 0.5f, 1.0f, 1.0f, 0.8f};
  for(int k = 0; k < RK_AJ_NUM; k++) p->ctrl_time_s[k] = 0.01f, p->gear_ratio[k] = gear[k], p->motor_dir[k] = dir[k], p->curlim_default_A[k] = cl[k];
  p->cycle_time_s = 0.01f; // AD_task_main.cpp:149
  const float mech[RK_AJ_NUM] = {-45.0f, 150.0f, 0.0f, 0.0f, 0.0f, 0.0f, -90.0f};
  const float vin[RK_AJ_NUM]  = {15.0f, 30.0f, 10.0f, 10.0f, 30.0f, 30.0f, -60.0f};
  const float cin[RK_AJ_NUM]  = {1.0f, 0.15f, 0.5f, 0.5f, 1.0f, 1.0f, 0.5f};
  const float ipos[RK_AJ_NUM] = {0.0f, 145.0f, 0.0f, 0.0f, -90.0f, 0.0f, 0.0f};
  for(int k = 0; k < RK_AJ_NUM; k++) p->mechend_pos_deg[k] = mech[k], p->vel_init_degps[k] = vin[k], p->curlim_init_A[k] = cin[k], p->initpos_deg[k] = ipos[k];
}

size_t rk_adt_state_words(void) { return RK_AS_WORDS; }
size_t rk_adt_state_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_AS_WORDS * 4u; }
size_t rk_adt_cmdtab_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_ACMD_WORDS * 4u; }

static int adt_check(const char *who, const void *a, const void *b, int64_t n) {
  if(n < 0) {
    set_error("%s: n < 0", who);
    return RK_ERR_ARG;
  }
  if(!a || ((uintptr_t)a & 15u) || ((uintptr_t)b & 15u)) {
    set_error("%s: blocks must be non-NULL and 16-byte aligned", who);
    return RK_ERR_ARG;
  }
  return require_device();
}
static unsigned adt_grid(int64_t n) { return (unsigned)((n + 127) / 128); }

// div_by_rcp64 against div.rn.f32 on `total` pseudo-random (x, c) pairs: all bit patterns of x, c alternately any
// float and an integer count in 1 .. 2^24; counts the mismatches (NaNs compare as NaNs).
__global__ void selftest_div_rcp64_kernel(unsigned long long total, unsigned long long seed, unsigned int *bad) {
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  unsigned int             mine   = 0;
  for(unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride) {
    unsigned long long z = (k + seed) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull, z = (z ^ (z >> 27)) * 0x94D049BB133111EBull, z ^= z >> 31;
    const uint32_t hi = (uint32_t)(z >> 32);
    // every fourth pair: a subnormal / tiny numerator over a small count -- the domain of exact ties
    const float x = ((k & 3) == 2) ? u2f(((uint32_t)z & 0x81FFFFFFu)) : u2f((uint32_t)z);
    const float c = (k & 1) ? u2f(hi) : (float)((hi & (((k & 3) == 2) ? 0xFFFu : 0xFFFFFFu)) + 1u);
    const float want = fdiv(x, c), got = div_by_rcp64(x, c, __drcp_rn((double)c));
    const bool  same = (f2u(want) == f2u(got)) || (want != want && got != got);
    mine += same ? 0u : 1u;
  }
  if(mine) atomicAdd(bad, mine);
}

int rk_adt_mode_init(const rk_adt_params_t *p, void *d_state, int64_t n, void *stream) {
  if(n == 0) return RK_OK;
  if(!p) {
    set_error("rk_adt_mode_init: params NULL");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adt_mode_init", d_state, nullptr, n)) return rc;
  adt_mode_init_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>(*p, (uint4 *)d_state, n);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adt_push_cmdseq(void *d_state, void *d_cmdtab, int64_t n, const void *d_seq, const uint8_t *d_valid, void *stream) {
  if(n == 0) return RK_OK;
  if(!d_cmdtab || !d_seq || ((uintptr_t)d_seq & 15u)) {
    set_error("rk_adt_push_cmdseq: d_cmdtab / d_seq must be non-NULL and 16-byte aligned");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adt_push_cmdseq", d_state, d_cmdtab, n)) return rc;
  adt_push_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>((uint4 *)d_state, (uint4 *)d_cmdtab, n, (const uint4 *)d_seq, d_valid);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adt_update(const rk_adt_params_t *p, void *d_state, const void *d_cmdtab, int64_t n, int32_t K, uint32_t *d_trace, void *stream) {
  return rk::adt_update_launch(p, d_state, d_cmdtab, n, K, d_trace, 0, stream);
}
} // extern "C"

// Calls f(DIVC, rcp) for the MG joint's control time ct: DIVC = div_const_exact(ct) (an exhaustive on-device proof, cached
// per constant) as a std::integral_constant, rcp = RN(1 / ct) from one correctly rounded host division (0 when DIVC == 0).
template <class F>
static void with_divc(float ct, F &&f) {
  const int   divc = div_const_exact(ct);
  const float rcp  = divc ? 1.0f / ct : 0.0f;
  if(divc == 2) f(std::integral_constant<int, 2>{}, rcp);
  else if(divc == 1) f(std::integral_constant<int, 1>{}, rcp);
  else f(std::integral_constant<int, 0>{}, rcp);
}

// max_ctas > 0: at most that many CTAs (each strides over the batch)
int rk::adt_update_launch(const rk_adt_params_t *p, void *d_state, const void *d_cmdtab, int64_t n, int32_t K, uint32_t *d_trace,
                          int max_ctas, void *stream) {
  if(n == 0 || K == 0) return RK_OK;
  if(!p || K < 0 || !d_cmdtab) {
    set_error("rk_adt_update: params / cmdtab NULL or K < 0");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adt_update", d_state, d_cmdtab, n)) return rc;
  cudaStream_t st   = (cudaStream_t)stream;
  unsigned     grid = adt_grid(n);
  if(max_ctas > 0 && grid > (unsigned)max_ctas) grid = (unsigned)max_ctas;
  with_divc(p->ctrl_time_s[RK_AJ_P1], [&](auto dv, float rcp) {
    uint4       *s = (uint4 *)d_state;
    const uint4 *t = (const uint4 *)d_cmdtab;
    if(d_trace) adt_update_kernel<true, dv><<<grid, 128, 0, st>>>(*p, s, t, n, K, d_trace, rcp);
    else adt_update_kernel<false, dv><<<grid, 128, 0, st>>>(*p, s, t, n, K, d_trace, rcp);
  });
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

extern "C" {

int rk_adt_bldc_rx(const rk_adt_params_t *p, void *d_state, int64_t n, int slot, const uint64_t *d_frames, const uint32_t *d_cmdid,
                   float *d_cur_A, void *stream) {
  if(n == 0) return RK_OK;
  if(!p || !d_frames || slot < 0 || slot > 2 || ((uintptr_t)d_frames & 7u)) {
    set_error("rk_adt_bldc_rx: params / frames NULL or misaligned, or slot outside 0..2");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adt_bldc_rx", d_state, nullptr, n)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const auto  *fr = (const unsigned long long *)d_frames;
  if(slot == 0) adt_rx_kernel<0><<<adt_grid(n), 128, 0, st>>>(*p, (uint4 *)d_state, n, fr, d_cmdid, d_cur_A);
  else if(slot == 1) adt_rx_kernel<1><<<adt_grid(n), 128, 0, st>>>(*p, (uint4 *)d_state, n, fr, d_cmdid, d_cur_A);
  else adt_rx_kernel<2><<<adt_grid(n), 128, 0, st>>>(*p, (uint4 *)d_state, n, fr, d_cmdid, d_cur_A);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adt_mg_rx(const rk_adt_params_t *p, void *d_state, int64_t n, const uint64_t *d_frames, float *d_cur_A, void *stream) {
  if(n == 0) return RK_OK;
  if(!p || !d_frames || ((uintptr_t)d_frames & 7u)) {
    set_error("rk_adt_mg_rx: params / frames NULL or misaligned");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adt_mg_rx", d_state, nullptr, n)) return rc;
  adt_rx_kernel<3><<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>(*p, (uint4 *)d_state, n, (const unsigned long long *)d_frames, nullptr, d_cur_A);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adt_cmdseq_status(const void *d_state, const void *d_cmdtab, int64_t n, const uint32_t *d_id, int32_t *d_status, void *stream) {
  if(n == 0) return RK_OK;
  if(!d_cmdtab || !d_id || !d_status) {
    set_error("rk_adt_cmdseq_status: NULL argument");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adt_cmdseq_status", d_state, d_cmdtab, n)) return rc;
  adt_status_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>((const uint4 *)d_state, (const uint4 *)d_cmdtab, n, d_id, d_status);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

size_t rk_adp_state_words(void) { return RK_PS_WORDS; }
size_t rk_adp_state_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_PS_WORDS * 4u; }

int rk_adp_mode_init(void *d_pstate, int64_t n, void *stream) {
  if(n == 0) return RK_OK;
  if(int rc = adt_check("rk_adp_mode_init", d_pstate, nullptr, n)) return rc;
  adp_mode_init_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>((uint4 *)d_pstate, n);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adp_push_cmd(void *d_pstate, int64_t n, const void *d_cmd, const uint8_t *d_valid, void *stream) {
  if(n == 0) return RK_OK;
  if(!d_cmd || ((uintptr_t)d_cmd & 15u)) {
    set_error("rk_adp_push_cmd: d_cmd must be non-NULL and 16-byte aligned");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adp_push_cmd", d_pstate, nullptr, n)) return rc;
  adp_push_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>((uint4 *)d_pstate, n, (const uint4 *)d_cmd, d_valid);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adp_update(const rk_adt_params_t *p, void *d_state, void *d_pstate, int64_t n, int32_t K, uint32_t *d_trace, void *stream) {
  if(n == 0 || K == 0) return RK_OK;
  if(!p || K < 0) {
    set_error("rk_adp_update: params NULL or K < 0");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adp_update", d_state, d_pstate, n)) return rc;
  if(!d_pstate) {
    set_error("rk_adp_update: d_pstate NULL");
    return RK_ERR_ARG;
  }
  with_divc(p->ctrl_time_s[RK_AJ_P1], [&](auto dv, float rcp) {
    if(d_trace) adp_update_kernel<true, dv><<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>(*p, (uint4 *)d_state, (uint4 *)d_pstate, n, K, d_trace, rcp);
    else adp_update_kernel<false, dv><<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>(*p, (uint4 *)d_state, (uint4 *)d_pstate, n, K, d_trace, rcp);
  });
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adp_cmd_status(const void *d_pstate, int64_t n, const uint32_t *d_id, int32_t *d_status, void *stream) {
  if(n == 0) return RK_OK;
  if(!d_id || !d_status) {
    set_error("rk_adp_cmd_status: NULL argument");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adp_cmd_status", d_pstate, nullptr, n)) return rc;
  adp_status_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>((const uint4 *)d_pstate, n, d_id, d_status);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

// ---- single-instance handle: a batch of one over the same kernels ---------------------------
size_t rk_adh_state_words(void) { return RK_HS_WORDS; }
size_t rk_adh_state_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_HS_WORDS * 4u; }

int rk_adh_mode_init(void *d_hstate, int64_t n, int mode, void *stream) {
  if(n == 0) return RK_OK;
  if(n < 0 || !d_hstate || ((uintptr_t)d_hstate & 15u) || (mode != RK_ADH_MODE_INIT && mode != RK_ADH_MODE_INIT_POS_MOVE)) {
    set_error("rk_adh_mode_init: bad n / mode, or d_hstate NULL / not 16-byte aligned");
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  adh_mode_init_kernel<<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>((uint4 *)d_hstate, n, (uint32_t)mode);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_adh_update(const rk_adt_params_t *p, void *d_state, void *d_hstate, int64_t n, int32_t K, const float *d_now, uint32_t *d_trace,
                  void *stream) {
  if(n == 0 || K == 0) return RK_OK;
  if(K < 0) {
    set_error("rk_adh_update: K < 0");
    return RK_ERR_ARG;
  }
  if(!d_hstate || ((uintptr_t)d_now & 3u) || ((uintptr_t)d_trace & 3u)) {
    set_error("rk_adh_update: d_hstate NULL or misaligned d_now / d_trace");
    return RK_ERR_ARG;
  }
  if(int rc = adt_check("rk_adh_update", d_state, d_hstate, n)) return rc;
  rk_adt_params_t q;
  if(p) q = *p;
  else rk_adt_default_params(&q);
  if(int rc = require_device()) return rc;
  if(d_trace) adh_update_kernel<true><<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>(q, (uint4 *)d_state, (uint4 *)d_hstate, n, K, d_now, d_trace);
  else adh_update_kernel<false><<<adt_grid(n), 128, 0, (cudaStream_t)stream>>>(q, (uint4 *)d_state, (uint4 *)d_hstate, n, K, d_now, d_trace);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

// All blocks of the handle live in ONE mapped pinned allocation (zero-copy): the kernels read / write them over the
// bus, the host writes inputs and reads results directly -- no cudaMemcpy anywhere; a reader synchronises the stream
// only if a launch is still in flight.
struct rk_adt {
  rk_adt_params_t p;
  uint32_t       *h_mem = nullptr;
  cudaStream_t    st    = nullptr;
  bool            in_flight = false;
  uint32_t *state() { return h_mem; }
  uint32_t *tab() { return h_mem + 80; }                                     // RK_ACMD_WORDS
  uint32_t *seq() { return h_mem + 80 + RK_ACMD_WORDS; }                     // RK_ACMD_SLOT_WORDS
  uint32_t *misc() { return h_mem + 80 + RK_ACMD_WORDS + RK_ACMD_SLOT_WORDS; } // [0] id, [1] status, [2..6] targets
  uint32_t *hs() { return misc() + 8; }                                      // homing block (RK_HS_WORDS) + 4 floats of feedback
  static size_t words() { return 80 + RK_ACMD_WORDS + RK_ACMD_SLOT_WORDS + 8 + RK_HS_WORDS + 4; }
};
static_assert(RK_AS_WORDS <= 80 && (80 + RK_ACMD_WORDS + RK_ACMD_SLOT_WORDS + 8) % 4 == 0, "16-byte aligned sub-blocks");
static int adt_settle(rk_adt *h) {
  if(h->in_flight) {
    RK_CUDA(cudaStreamSynchronize(h->st));
    h->in_flight = false;
  }
  return RK_OK;
}

int rk_adt_create(rk_adt_t **out, const rk_adt_params_t *p) {
  if(!out) return RK_ERR_ARG;
  *out = nullptr;
  if(int rc = require_device()) return rc;
  rk_adt *h = new rk_adt();
  if(p) h->p = *p;
  else rk_adt_default_params(&h->p);
  cudaError_t e = cudaHostAlloc((void **)&h->h_mem, rk_adt::words() * 4, cudaHostAllocMapped);
  if(e == cudaSuccess) memset(h->h_mem, 0, rk_adt::words() * 4);
  if(e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking);
  if(e != cudaSuccess) {
    int rc = cuda_fail(e, "rk_adt_create");
    rk_adt_destroy(h);
    return rc;
  }
  *out = h;
  return RK_OK;
}
void rk_adt_destroy(rk_adt_t *h) {
  if(!h) return;
  if(h->st) {
    cudaStreamSynchronize(h->st);
    cudaStreamDestroy(h->st);
  }
  if(h->h_mem) cudaFreeHost(h->h_mem);
  delete h;
}
int rk_adt_init(rk_adt_t *h) {
  if(!h) return RK_ERR_ARG;
  h->in_flight = true;
  return rk_adt_mode_init(&h->p, h->state(), 1, h->st);
}
int rk_adt_push(rk_adt_t *h, const rk_adt_poscmdseq_t *seq) {
  if(!h || !seq) return RK_ERR_ARG;
  if(int rc = adt_settle(h)) return rc; // the previous push may still read the image
  uint32_t *w = h->seq();
  memset(w, 0, RK_ACMD_SLOT_WORDS * 4);
  w[0] = seq->id, w[1] = seq->len;
  for(int k = 0; k < RK_ACMD_MAX_LEN; k++) {
    w[4 + 8 * k] = seq->cmd[k].dt_ms;
    memcpy(&w[4 + 8 * k + 1], seq->cmd[k].tgt_deg, 20);
  }
  h->in_flight = true;
  return rk_adt_push_cmdseq(h->state(), h->tab(), 1, h->seq(), nullptr, h->st);
}
int rk_adt_home_init(rk_adt_t *h, int mode) { // set_next_mode(INIT / INIT_POS_MOVE) -> m_nowProcess->init()
  if(!h) return RK_ERR_ARG;
  h->in_flight = true;
  return rk_adh_mode_init(h->hs(), 1, mode, h->st);
}
int rk_adt_home_tick(rk_adt_t *h, const float servo_now_deg[4], int *completed) {
  if(!h) return RK_ERR_ARG;
  float *now = nullptr;
  if(servo_now_deg) {
    if(int rc = adt_settle(h)) return rc;
    now = (float *)(h->hs() + RK_HS_WORDS);
    memcpy(now, servo_now_deg, 16);
  }
  h->in_flight = true;
  if(int rc = rk_adh_update(&h->p, h->state(), h->hs(), 1, 1, now, nullptr, h->st)) return rc;
  if(completed) { // ADTModeBase::isCompleted()
    if(int rc = adt_settle(h)) return rc;
    *completed = (h->hs()[0] & RK_AS_FSM_IS_COMP) ? 1 : 0;
  }
  return RK_OK;
}
int rk_adt_tick(rk_adt_t *h) {
  if(!h) return RK_ERR_ARG;
  h->in_flight = true;
  return rk_adt_update(&h->p, h->state(), h->tab(), 1, 1, nullptr, h->st);
}
int rk_adt_status(rk_adt_t *h, uint32_t id, int32_t *status) {
  if(!h || !status) return RK_ERR_ARG;
  if(int rc = adt_settle(h)) return rc;
  h->misc()[0] = id;
  h->in_flight = true;
  if(int rc = rk_adt_cmdseq_status(h->state(), h->tab(), 1, h->misc(), (int32_t *)(h->misc() + 1), h->st)) return rc;
  if(int rc = adt_settle(h)) return rc;
  *status = (int32_t)h->misc()[1];
  return RK_OK;
}
int rk_adt_get_state(rk_adt_t *h, uint32_t words[RK_AS_WORDS]) {
  if(!h || !words) return RK_ERR_ARG;
  if(int rc = adt_settle(h)) return rc;
  memcpy(words, h->state(), RK_AS_WORDS * 4);
  return RK_OK;
}
int rk_adt_set_state(rk_adt_t *h, const uint32_t words[RK_AS_WORDS]) {
  if(!h || !words) return RK_ERR_ARG;
  if(int rc = adt_settle(h)) return rc;
  memcpy(h->state(), words, RK_AS_WORDS * 4);
  return RK_OK;
}
int rk_adt_get_targets_deg(rk_adt_t *h, float out[5]) {
  if(!h || !out) return RK_ERR_ARG;
  adt_targets_kernel<<<1, 32, 0, h->st>>>((const uint4 *)h->state(), 1, 0, (float *)(h->misc() + 2));
  h->in_flight = true;
  RK_CUDA(cudaGetLastError());
  if(int rc = adt_settle(h)) return rc;
  memcpy(out, h->misc() + 2, 20);
  return RK_OK;
}
/* JointMyBldcServo / JointMgServo::rx_callback on the single instance (see rk_adt_bldc_rx / rk_adt_mg_rx); slot 0..2 =
 * DF_Left, DF_Right, P3, slot 3 = the MG servo.  *cur_A (optional) receives fl_out_now_cur when the frame carries one. */
int rk_adt_rx(rk_adt_t *h, int slot, uint32_t cmdid, const uint8_t frame[8], float *cur_A) {
  if(!h || !frame || slot < 0 || slot > 3) return RK_ERR_ARG;
  if(int rc = adt_settle(h)) return rc;
  uint32_t *m = h->misc();
  memcpy(m + 4, frame, 8); // misc words 4-5: the frame, 6: command id, 7: current (a NaN tag = "not written")
  m[6] = cmdid, m[7] = 0x7FC12345u;
  h->in_flight = true;
  int rc = (slot == 3) ? rk_adt_mg_rx(&h->p, h->state(), 1, (const uint64_t *)(m + 4), (float *)(m + 7), h->st)
                       : rk_adt_bldc_rx(&h->p, h->state(), 1, slot, (const uint64_t *)(m + 4), m + 6, (float *)(m + 7), h->st);
  if(rc) return rc;
  if(cur_A) {
    if(int rc2 = adt_settle(h)) return rc2;
    if(m[7] != 0x7FC12345u) memcpy(cur_A, m + 7, 4);
  }
  return RK_OK;
}
}

/* Self-test of the shared-reciprocal division the arm tick uses (div_by_rcp64): `pairs` pseudo-random (x, c) pairs
 * against div.rn.f32; *mismatches receives the number that differ.  Synchronous. */
extern "C" int rk_selftest_div_rcp64(uint64_t pairs, uint64_t seed, uint32_t *mismatches) {
  if(!mismatches) return RK_ERR_ARG;
  if(int rc = require_device()) return rc;
  unsigned int *d = nullptr;
  RK_CUDA(cudaMalloc((void **)&d, 4));
  cudaMemset(d, 0, 4);
  selftest_div_rcp64_kernel<<<148 * 8, 256>>>(pairs, seed, d);
  const cudaError_t e = cudaMemcpy(mismatches, d, 4, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if(e != cudaSuccess) return cuda_fail(e, "rk_selftest_div_rcp64");
  return RK_OK;
}
