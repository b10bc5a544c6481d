// rk_vehicle_fast2.cuh -- the closed-loop fast tick of rk_vehicle_fast.cuh, re-expressed on
// Blackwell's packed FP32 instructions (FADD2 / FFMA2, sm_100) and cut down to the values a
// fused rollout can observe.
//
// Why: the tick is bound by the SM's ISSUE rate (one warp-instruction per clock per
// sub-partition), not by the FP32 lanes themselves -- bit parity forbids FMA contraction, so
// every algorithmic flop is an instruction, and a third of the instruction stream is
// integer / select / convert work competing for the same issue slots.  A packed instruction
// retires two IEEE-rounded FP32 operations for ONE issue slot (it occupies the FMA pipe for
// two cycles, so the lane throughput is unchanged; measured with tools/ubench/f32x2_probe.cu).
//
// Lane assignment (round 2) -- every packed op has two useful lanes and no operand needs a MOV:
//   * wheel speed -> controller input (Mvel * GEAR_RATIO): lanes = {FL, BL} and {BR, FR};
//   * odometry increment: the four wheel steps are formed as {m0, -m0}, {m2, -m2} (odd symmetry of
//     the product) and {m1, m3}; the two sums of conv_Mdir_to_Vdir then run as lanes = {x, y};
//   * odometry rotation: lanes = {x, y};
//   * jerk-limited targets: lanes = {x interpolator, y interpolator} (theta stays scalar);
//   * inverse kinematics and the four FF_PI_D loops: lanes = {FL, BL} and {BR, FR}.
// Values nobody can observe inside a fused chunk are not formed per tick: the measured body
// velocity (VD_vehicle_controller.cpp:26-33: written every tick, read by nobody but the getters; the
// transcription tick that ends every launch stores it), acl_now_ of the three interpolators (read
// only by set_target_params and the final store: rebuilt from the last tick's operands when a
// chunk ends) and the IIR's prev_X_ (likewise).  With a trace attached they are all formed.
// Results are bit-identical to the scalar code: each lane performs the same single-rounding
// IEEE operation (packed ops are .rn, denormals preserved).
//
// ptxas (12.9) contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even with --fmad=false, which
// would break parity.  Every packed multiply is therefore written as fma(a, b, nz) with nz an
// OPAQUE -0.0f (derived from a kernel parameter at run time): a*b + (-0) is exactly RN(a*b)
// including the sign of a zero product, and an FMA cannot be contracted with the add that
// follows it.  cuobjdump shows FFMA2 ... Rnz.F32 followed by separate FADD2s.
#pragma once
#include "rk_vehicle_fast.cuh"

namespace rk {

RK_DEV float2 bc2(float s) { return make_float2(s, s); }
RK_DEV float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
RK_DEV float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
RK_DEV float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, neg2(b)); } // a - b == a + (-b) exactly
RK_DEV float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
RK_DEV float2 mul2(float2 a, float2 b, float nz) { return __ffma2_rn(a, b, make_float2(nz, nz)); }

// exact x / c per lane (div_const of rk_vehicle_fast.cuh)
RK_DEV float2 div_const2(float2 x, float c, float rcp, float nz) {
  const float2 q = mul2(x, bc2(rcp), nz);
  const float2 e = fma2(q, bc2(c), neg2(x));
  return fma2(neg2(e), bc2(rcp), q);
}

// x and y VelInterpConstJerk, lane-paired.  tm = max(t1, t2, t3): "one of the three phase conditions holds".
struct FastInterp2 {
  float2 vel, dt;
  float2 t1, t2, tm;
  float2 vel_tgt, acl_max, jerk_p, jerk_m, dt1, dt2, vel_ini, acl_ini;
  // operands of the last executed update, from which acl_now_ is rebuilt when the chunk ends
  float2 a1_l, a23_l;
  bool   p1x_l, p1y_l, acx_l, acy_l;
};
struct FastInterp1 { // the theta interpolator, same scheme
  float vel, dt;
  float t1, t2, tm;
  float vel_tgt, acl_max, jerk_p, jerk_m, dt1, dt2, vel_ini, acl_ini;
  float a1_l, a23_l;
  bool  p1_l, ac_l;
};
struct FastWheel2 { // two wheels of equal direction, lane-paired
  int32_t rpm[2], cur[2], dsum[2];
  float2  dsf; // fast_tick2: the chunk's angle sums kept as exact integers in float (|sum| < 2^24, see kMaxChunk);
               // w01.dsf = {wheel 0, wheel 2}, w23.dsf = {wheel 1, wheel 3} -- the pairing the odometry consumes the steps in
  float2  prev_val, integ, lpf_y, b0x;
  float2  x_l; // the IIR input of the last executed tick (prev_X_)
};
struct FastVeh2 {
  float2      p; // pos x, y
  FastInterp2 xy;
  FastInterp1 th;
  FastWheel2  w01, w23;
};

RK_DEV float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

RK_DEV void fast_interp1_load(FastInterp1 &f, const Interp &t, float ts) {
  f.vel = t.vel, f.dt = t.dt;
  f.vel_tgt = t.vel_tgt, f.acl_max = t.acl_max, f.jerk_p = t.jerk_p, f.jerk_m = t.jerk_m;
  f.dt1 = t.dt1, f.dt2 = t.dt2, f.vel_ini = t.vel_ini, f.acl_ini = t.acl_ini;
  f.t1 = fadd(t.dt1, ts);
  f.t2 = fadd(fadd(t.dt1, t.dt2), ts);
  f.tm = max3(f.t1, f.t2, fadd(fadd(fadd(t.dt1, t.dt2), t.dt3), ts));
  // keep the thresholds in registers: without this ptxas rematerialises the adds every tick
  asm volatile("" : "+f"(f.t1), "+f"(f.t2), "+f"(f.tm));
  f.a1_l = 0.0f, f.a23_l = 0.0f, f.p1_l = false, f.ac_l = false;
}
RK_DEV void fast_interp2_load(FastInterp2 &f, const Interp &a, const Interp &b, float ts) {
  FastInterp1 fa, fb;
  fast_interp1_load(fa, a, ts);
  fast_interp1_load(fb, b, ts);
  f.vel = make_float2(fa.vel, fb.vel), f.dt = make_float2(fa.dt, fb.dt);
  f.t1 = make_float2(fa.t1, fb.t1), f.t2 = make_float2(fa.t2, fb.t2), f.tm = make_float2(fa.tm, fb.tm);
  f.vel_tgt = make_float2(fa.vel_tgt, fb.vel_tgt), f.acl_max = make_float2(fa.acl_max, fb.acl_max);
  f.jerk_p = make_float2(fa.jerk_p, fb.jerk_p), f.jerk_m = make_float2(fa.jerk_m, fb.jerk_m);
  f.dt1 = make_float2(fa.dt1, fb.dt1), f.dt2 = make_float2(fa.dt2, fb.dt2);
  f.vel_ini = make_float2(fa.vel_ini, fb.vel_ini), f.acl_ini = make_float2(fa.acl_ini, fb.acl_ini);
  f.a1_l = bc2(0.0f), f.a23_l = bc2(0.0f), f.p1x_l = f.p1y_l = f.acx_l = f.acy_l = false;
}
// after >= 1 executed updates: acl_now_ as the last update assigned it (util_vel_interp.hpp:114,119,124,129)
RK_DEV float acl_of_last(bool p1, bool ac, float a1, float a23) { return p1 ? a1 : (ac ? a23 : 0.0f); }
RK_DEV void  fast_interp1_store(const FastInterp1 &f, Interp &t) {
  t.vel = f.vel, t.dt = f.dt, t.acl = acl_of_last(f.p1_l, f.ac_l, f.a1_l, f.a23_l);
}
RK_DEV void fast_interp2_store(const FastInterp2 &f, Interp &a, Interp &b) {
  a.vel = f.vel.x, a.dt = f.dt.x, a.acl = acl_of_last(f.p1x_l, f.acx_l, f.a1_l.x, f.a23_l.x);
  b.vel = f.vel.y, b.dt = f.dt.y, b.acl = acl_of_last(f.p1y_l, f.acy_l, f.a1_l.y, f.a23_l.y);
}

// util_vel_interp.hpp:110-136.  The if / else-if chain takes the FIRST true condition:
//   p1                      -> phase 1 (closed form in dt)
//   !p1 && (p2 || p3)       -> vel += a23 * ts with a23 = p2 ? acl_max : acl_max + jerk_m * ((dt - dt1) - dt2)
//   none                    -> vel = vel_tgt, dt stays
// and (p1 || p2 || p3) == (dt <= max(t1, t2, t3)).
RK_DEV float2 fast_interp2_update(FastInterp2 &f, float ts, float nz) {
  const float2 a1  = add2(f.acl_ini, mul2(f.jerk_p, f.dt, nz));
  const float2 v1  = add2(f.vel_ini, mul2(mul2(add2(f.acl_ini, a1), f.dt, nz), bc2(0.5f), nz));
  const float2 a3  = add2(f.acl_max, mul2(f.jerk_m, sub2(sub2(f.dt, f.dt1), f.dt2), nz));
  const bool   p1x = f.dt.x <= f.t1.x, p2x = f.dt.x <= f.t2.x, acx = f.dt.x <= f.tm.x;
  const bool   p1y = f.dt.y <= f.t1.y, p2y = f.dt.y <= f.t2.y, acy = f.dt.y <= f.tm.y;
  const float2 a23 = make_float2(p2x ? f.acl_max.x : a3.x, p2y ? f.acl_max.y : a3.y);
  const float2 v23 = add2(f.vel, mul2(a23, bc2(ts), nz));
  f.vel            = make_float2(p1x ? v1.x : (acx ? v23.x : f.vel_tgt.x), p1y ? v1.y : (acy ? v23.y : f.vel_tgt.y));
  if(acx) f.dt.x = fadd(f.dt.x, ts);
  if(acy) f.dt.y = fadd(f.dt.y, ts);
  f.a1_l = a1, f.a23_l = a23, f.p1x_l = p1x, f.p1y_l = p1y, f.acx_l = acx, f.acy_l = acy;
  return f.vel;
}
RK_DEV float fast_interp1_update(FastInterp1 &f, float ts) {
  const bool  p1 = f.dt <= f.t1, p2 = f.dt <= f.t2, ac = f.dt <= f.tm;
  const float a1  = fadd(f.acl_ini, fmul(f.jerk_p, f.dt));
  const float v1  = fadd(f.vel_ini, fmul(fmul(fadd(f.acl_ini, a1), f.dt), 0.5f));
  const float a3  = fadd(f.acl_max, fmul(f.jerk_m, fsub(fsub(f.dt, f.dt1), f.dt2)));
  const float a23 = p2 ? f.acl_max : a3;
  const float v23 = fadd(f.vel, fmul(a23, ts));
  f.vel           = p1 ? v1 : (ac ? v23 : f.vel_tgt);
  if(ac) f.dt = fadd(f.dt, ts);
  f.a1_l = a1, f.a23_l = a23, f.p1_l = p1, f.ac_l = ac;
  return f.vel;
}

RK_DEV void to_fast_wheel2(FastWheel2 &w, const Veh &v, int a, int b, float b0) {
  w.rpm[0] = v.m[a].p_rpm, w.rpm[1] = v.m[b].p_rpm, w.cur[0] = v.m[a].cur_tgt, w.cur[1] = v.m[b].cur_tgt;
  w.dsum[0] = 0, w.dsum[1] = 0, w.dsf = make_float2(0.0f, 0.0f);
  w.prev_val = make_float2(v.c[a].prev_val, v.c[b].prev_val), w.integ = make_float2(v.c[a].integ, v.c[b].integ);
  w.lpf_y = make_float2(v.c[a].lpf_y, v.c[b].lpf_y);
  w.x_l   = make_float2(v.c[a].lpf_x, v.c[b].lpf_x);
  w.b0x   = make_float2(fmul(b0, v.c[a].lpf_x), fmul(b0, v.c[b].lpf_x));
}
RK_DEV void to_fast2(const Veh &v, FastVeh2 &f, float ts, float b0) {
  f.p = make_float2(v.pos[0], v.pos[1]);
  fast_interp2_load(f.xy, v.it[0], v.it[1], ts);
  fast_interp1_load(f.th, v.it[2], ts);
  to_fast_wheel2(f.w01, v, 0, 1, b0);
  to_fast_wheel2(f.w23, v, 2, 3, b0);
}
RK_DEV FastWheel lane_wheel(const FastWheel2 &w, int l) {
  FastWheel s;
  s.rpm = w.rpm[l], s.cur = w.cur[l], s.dsum = w.dsum[l];
  s.prev_val = l ? w.prev_val.y : w.prev_val.x, s.integ = l ? w.integ.y : w.integ.x;
  s.lpf_y = l ? w.lpf_y.y : w.lpf_y.x, s.lpf_x = l ? w.x_l.y : w.x_l.x, s.b0x = l ? w.b0x.y : w.b0x.x;
  return s;
}
// requires nticks >= 1 (the *_l operands are those of an executed tick)
RK_DEV void from_fast2_common(Veh &v, const FastVeh2 &f, FastWheel w[4]) {
  v.pos[0] = f.p.x, v.pos[1] = f.p.y;
  fast_interp2_store(f.xy, v.it[0], v.it[1]);
  fast_interp1_store(f.th, v.it[2]);
  w[0] = lane_wheel(f.w01, 0), w[1] = lane_wheel(f.w01, 1), w[2] = lane_wheel(f.w23, 0), w[3] = lane_wheel(f.w23, 1);
  // the float angle sums of fast_tick2 (zero on the stream tick, which sums in dsum) in their odometry pairing
  w[0].dsum += (int32_t)f.w01.dsf.x, w[2].dsum += (int32_t)f.w01.dsf.y, w[1].dsum += (int32_t)f.w23.dsf.x, w[3].dsum += (int32_t)f.w23.dsf.y;
#pragma unroll
  for(int k = 0; k < 4; k++) v.c[k].prev_val = w[k].prev_val, v.c[k].integ = w[k].integ, v.c[k].lpf_y = w[k].lpf_y, v.c[k].lpf_x = w[k].lpf_x;
}
template <int D0, int D1, int D2, int D3>
RK_DEV void from_fast2(Veh &v, const FastVeh2 &f, int nticks) {
  if(nticks <= 0) return;
  FastWheel w[4];
  from_fast2_common(v, f, w);
  from_fast_motor<D0>(v.m[0], w[0], nticks);
  from_fast_motor<D1>(v.m[1], w[1], nticks);
  from_fast_motor<D2>(v.m[2], w[2], nticks);
  from_fast_motor<D3>(v.m[3], w[3], nticks);
}

// One tick's wheel feedback as the core consumes it: wheel-frame rpm and encoder step, as floats.
struct Sense {
  float2 rw01, rw23; // (float)s16_rawSpeedRpm, direction applied        VD_motor_if_m2006.cpp:45
  float  d0, d2;     // (float)(s64_rawAngleSum - s64_rawAngleSumPrev) of wheels 0, 2   VD_vehicle_controller.cpp:37-41
  float2 d13;        // ... and of wheels 1, 3, paired as the odometry consumes them
};

// ---- RK_SENSOR_STREAM on the fast tick: the wheel feedback comes from recorded C610 frames, so rx_callback
// (VD_motor_if_m2006.cpp:32-72) runs in full -- big-endian fields, direction, the +-4096 unwrap -- instead of the
// collapsed plant.  The odometry product fma(d, K_hi, d*K_lo) is proven for every step the unwrap can produce
// (|d| <= 2^17, rk_exact.cu), so no frame can leave the fast path's domain.
struct StreamSense {
  int32_t ang[4]; // head Status s16_rawAngle (direction applied): the one status word the next frame's unwrap needs.
                  // s16_rawSpeedRpm / s16_rawCurr are rewritten by the next rx_callback before anything reads them, and
                  // every launch ends on a transcription tick, so they are not carried through the fast ticks.
};
RK_DEV void stream_sense_load(StreamSense &ss, const Veh &v) {
#pragma unroll
  for(int k = 0; k < 4; k++) ss.ang[k] = v.m[k].ang;
}
// prmt.b32 with the selector's bit 3 (replicate the byte's sign) -- __byte_perm() only honours three bits per nibble
RK_DEV int32_t prmt_sx(uint32_t x, uint32_t sel) {
  int32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0u), "r"(sel));
  return r;
}
template <int DIR>
RK_DEV void fast_wheel_rx2(StreamSense &ss, int k, int32_t &dsum, uint64_t frame, float &rwf, float &df) {
  const uint32_t lo = (uint32_t)frame;
  // one PRMT each: the big-endian halfword with its sign replicated into the upper bytes (selector bit 3)
  const int32_t a = prmt_sx(lo, 0x8801); // (int16_t)((b0 << 8) | b1)
  const int32_t r = prmt_sx(lo, 0xAA23); // (int16_t)((b2 << 8) | b3)
  const int32_t raw_ang = (DIR == 1) ? a : sext16(8192 - a);
  int32_t       d       = sext16(raw_ang - ss.ang[k]);
  // +-8192 once when the step leaves +-4096 (VD_motor_if_m2006.cpp:50-55); d is an int16, so neither sum can wrap
  d += (d > 4096) ? -8192 : ((d < -4096) ? 8192 : 0);
  dsum += d;
  ss.ang[k] = raw_ang;
  rwf = (float)((DIR == 1) ? r : sext16(-r)), df = (float)d;
}
RK_DEV void from_fast2_stream(Veh &v, const FastVeh2 &f, const StreamSense &ss, int nticks) {
  if(nticks <= 0) return;
  FastWheel w[4];
  from_fast2_common(v, f, w);
#pragma unroll
  for(int k = 0; k < 4; k++) {
    Motor &m = v.m[k];
    m.sum += (int64_t)w[k].dsum;
    m.prev = m.sum;
    m.ang = ss.ang[k]; // rpm / cur: see StreamSense
    m.cur_tgt = w[k].cur;
    m.head    = (m.head + nticks) % 3;
  }
}

// FF_PI_D::update + set_CurrA_tgt for a pair of wheels of direction DIR (see fast_wheel_ctrl).
// tgt, now: controller target / input, already x GEAR_RATIO.
// (int16_t)(u * 1000.0f) * dir: trunc(-x) == -trunc(x) and sext16(-sext16(t)) == sext16(-t), so the direction
// folds into the multiplier.  The chunk only runs here when |u * 1000| < 2^31 is guaranteed (fast_u_bounded),
// so the conversion never saturates and equals x86's cvttss2si.
// KD0: Dgain_ == 0 (the firmware's setting, VD_task_main.cpp:86-89).  Kd * y is then +-0 for every finite y (the chunk
// bound keeps y finite), and (Kp*e + I) - (+-0) is (Kp*e + I) -- except that a zero result may come out as +0 where the
// subtraction gives -0; the sum only feeds the integer conversion of u * 1000, which maps both zeros to 0.  So the product
// and the subtraction are dropped; the filter itself still runs (its state is stored).
template <int DIR, bool FFSAT, bool KD0>
RK_DEV void fast_wheel_ctrl2(FastWheel2 &w, const rk_vdt_params_t &p, const FastConsts &fc, float2 tgt, float2 now, float nz) {
  const float2 err = sub2(tgt, now);
  const float2 x   = mul2(sub2(now, w.prev_val), bc2(p.ctrl_freq), nz);
  const float2 b0x = mul2(x, bc2(fc.B0), nz);
  const float2 y   = add2(add2(mul2(w.lpf_y, bc2(fc.A1), nz), b0x), w.b0x);
  w.lpf_y = y, w.x_l = x, w.b0x = b0x;
  const float2 ig = add2(w.integ, mul2(err, bc2(fc.ki_dt), nz));
  w.integ         = make_float2(clamp_sym(ig.x, p.i_limit, fc.neg_i_limit), clamp_sym(ig.y, p.i_limit, fc.neg_i_limit));
  float2 u        = add2(mul2(err, bc2(p.kp), nz), w.integ);
  if(!KD0) u = sub2(u, mul2(y, bc2(p.kd), nz));
  w.prev_val      = now;
  float2 ff;
  if(FFSAT) {
    const float2 sp = make_float2(__saturatef(fmul(tgt.x, p.kff)), __saturatef(fmul(tgt.y, p.kff)));
    const float2 sn = make_float2(__saturatef(fmul(tgt.x, -p.kff)), __saturatef(fmul(tgt.y, -p.kff)));
    ff              = sub2(sp, sn);
  } else {
    const float2 m = mul2(tgt, bc2(p.kff), nz);
    ff             = make_float2(clamp_sym(m.x, p.ff_limit, fc.neg_ff_limit), clamp_sym(m.y, p.ff_limit, fc.neg_ff_limit));
  }
  u               = add2(u, ff);
  const float2 tq = mul2(u, bc2(DIR > 0 ? RK_AMPERE_TO_RAW_CURR : -RK_AMPERE_TO_RAW_CURR), nz);
  const int32_t ta = sext16(__float2int_rz(tq.x)), tb = sext16(__float2int_rz(tq.y));
  w.cur[0] = min(max(ta, -p.raw_curr_lim), p.raw_curr_lim);
  w.cur[1] = min(max(tb, -p.raw_curr_lim), p.raw_curr_lim);
}

// One packed fast tick on the feedback s.  cs = {cos, sin}(yaw), sc = {sin, cos}(yaw).
// TRACE: also forms now_vhcl_vel_mmps (vel) -- see the header comment.
template <bool FFSAT, bool TRACE, bool KD0>
RK_DEV void fast_tick2_core(FastVeh2 &f, const rk_vdt_params_t &p, const FastConsts &fc, float2 cs, float2 sc, float nz,
                            float vel[3], float tgt[3], const Sense &s) {
  // Mvel = (rpm * RPM_TO_RADPS) * GEAR_RATIO_INV ; controller input = Mvel * GEAR_RATIO   :21-24,70-73
  const float2 mv01 = mul2(mul2(s.rw01, bc2(RK_RPM_TO_RADPS), nz), bc2(RK_GEAR_RATIO_INV), nz);
  const float2 mv23 = mul2(mul2(s.rw23, bc2(RK_RPM_TO_RADPS), nz), bc2(RK_GEAR_RATIO_INV), nz);
  const float2 now01 = mul2(mv01, bc2(RK_GEAR_RATIO), nz), now23 = mul2(mv23, bc2(RK_GEAR_RATIO), nz);
  // conv_Mdir_to_Vdir  VD_vehicle_controller.cpp:126-130
  // (sum * 0.25f) * R == sum * (0.25f * R) bit for bit: scaling by 2^-2 is exact in both places as long as
  // nothing underflows, and a sum of wheel speeds / angle steps is 0 or >= 2^-40 in magnitude (they derive
  // from int16 rpm and integer encoder steps).  The same scaling commutes with the two exact divisions.
  const float R = p.wheel_radius_mm, qR = fmul(0.25f, R);
  if(TRACE) {
    const float m0 = mv01.x, m1 = mv01.y, m2 = mv23.x, m3 = mv23.y;
    vel[0]         = fmul(fadd(fadd(fadd(m0, m1), m2), m3), qR);
    vel[1]         = fmul(fadd(fsub(fadd(-m0, m1), m2), m3), qR);
    const float sm = fadd(fadd(fsub(-m0, m1), m2), m3);
    vel[2]         = fmul(div_const(div_const(sm, p.sqrtf2, fc.rcp_s2), p.wheel_l_mm, fc.rcp_l), qR);
  }
  // Mrad = (float)((double)d * OUT_RAD_PER_RAW_ANGLE * GEAR_RATIO_INV) = fma(d, K_hi, d * K_lo)  :37-41 (rk_exact.cu);
  // the form is odd in d, so {m, -m} is the same two operations on {d, -d}
  const float2 khi = fc.khi_pm, klo = fc.klo_pm; // {K, -K}
  const float2 M0  = fma2(bc2(s.d0), khi, mul2(bc2(s.d0), klo, nz)); // {m0, -m0}
  const float2 M2  = fma2(bc2(s.d2), khi, mul2(bc2(s.d2), klo, nz)); // {m2, -m2}
  const float2 d13 = s.d13;
  const float2 M13 = fma2(d13, bc2(fc.k_hi), mul2(d13, bc2(fc.k_lo), nz)); // {m1, m3}
  // {((m0 + m1) + m2) + m3, ((-m0 + m1) - m2) + m3} * (0.25 * R) = local {dx, dy}
  const float2 l = mul2(add2(add2(add2(make_float2(M0.x, M0.y), bc2(M13.x)), make_float2(M2.x, M2.y)), bc2(M13.y)), bc2(qR), nz);
  // pos += (R(yaw) * local) * 0.001   :50-51 ; {lx*c - ly*s, lx*s + ly*c}
  const float2 a = mul2(bc2(l.x), cs, nz);
  const float2 b = mul2(bc2(l.y), sc, nz);
  f.p            = add2(f.p, mul2(__fadd2_rn(a, make_float2(-b.x, b.y)), bc2(0.001f), nz));
  const float2 txy = fast_interp2_update(f.xy, p.ts, nz);
  tgt[0] = txy.x, tgt[1] = txy.y;
  tgt[2] = fast_interp1_update(f.th, p.ts);
  // conv_Vdir_to_Mdir  :113-118 ; controller target = Mvel_tgt * GEAR_RATIO  :66-69
  const float  T  = fmul(fmul(fc.s2l, tgt[2]), 4.0f); // (not folded: a denormal-range target would round differently)
  const float2 xy = make_float2(fsub(tgt[0], tgt[1]), fadd(tgt[0], tgt[1]));
  const float2 t01 = mul2(div_const2(sub2(xy, bc2(T)), R, fc.rcp_r, nz), bc2(RK_GEAR_RATIO), nz);
  const float2 t23 = mul2(div_const2(add2(xy, bc2(T)), R, fc.rcp_r, nz), bc2(RK_GEAR_RATIO), nz);
  fast_wheel_ctrl2<1, FFSAT, KD0>(f.w01, p, fc, t01, now01, nz);
  fast_wheel_ctrl2<-1, FFSAT, KD0>(f.w23, p, fc, t23, now23, nz);
}

// The plant's encoder step rpm * 8192 / 60000 (truncating) formed in FLOAT from the float wheel speed the
// tick needs anyway: trunc(RN(rw * C)) with C = RN(8192 / 60000) equals the integer division for every int16 rw (all
// 65536 checked by tests/test_cabi_cpu.py::test_float_encoder_step_is_exact and on the device by rk_exact.cu's
// proof_small_kernel); FRND runs on the otherwise idle conversion unit, the products and the angle sums pair up as
// packed ops, and six half-rate ALU cycles per wheel (sign fix, I2FP, integer accumulate) disappear.  A negative speed
// below one count gives -0.0 where the integer path gives +0.0; the step only enters the position sums, where the sign of
// a zero term is immaterial unless the position word itself is -0.0 -- the fast kernel's chunk test keeps such a (never produced) state out.
constexpr float kDangC = 0.13653333485126495f; // RN(8192 / 60000)
template <int DIR>
RK_DEV void fast_wheel_rpm2(int32_t &rpm, int32_t cur, float &rwf) {
  rpm += ((cur * 4 - rpm) >> 4);
  rwf = (float)((DIR == 1) ? rpm : -rpm);
}
template <bool FFSAT, bool TRACE, bool KD0>
RK_DEV void fast_tick2(FastVeh2 &f, const rk_vdt_params_t &p, const FastConsts &fc, float2 cs, float2 sc, float nz,
                       float vel[3], float tgt[3]) {
  Sense s;
  fast_wheel_rpm2<1>(f.w01.rpm[0], f.w01.cur[0], s.rw01.x);
  fast_wheel_rpm2<1>(f.w01.rpm[1], f.w01.cur[1], s.rw01.y);
  fast_wheel_rpm2<-1>(f.w23.rpm[0], f.w23.cur[0], s.rw23.x);
  fast_wheel_rpm2<-1>(f.w23.rpm[1], f.w23.cur[1], s.rw23.y);
  const float2 q01 = mul2(s.rw01, bc2(kDangC), nz), q23 = mul2(s.rw23, bc2(kDangC), nz);
  s.d0 = truncf(q01.x), s.d2 = truncf(q23.x), s.d13 = make_float2(truncf(q01.y), truncf(q23.y));
  f.w01.dsf = add2(f.w01.dsf, make_float2(s.d0, s.d2)), f.w23.dsf = add2(f.w23.dsf, s.d13);
  fast_tick2_core<FFSAT, TRACE, KD0>(f, p, fc, cs, sc, nz, vel, tgt, s);
}
// the same tick fed by four recorded frames (RK_SENSOR_STREAM)
template <bool FFSAT, bool TRACE, bool KD0>
RK_DEV void fast_tick2_stream(FastVeh2 &f, StreamSense &ss, const uint64_t fr[4], const rk_vdt_params_t &p, const FastConsts &fc,
                              float2 cs, float2 sc, float nz, float vel[3], float tgt[3]) {
  Sense s;
  float d1, d3;
  fast_wheel_rx2<1>(ss, 0, f.w01.dsum[0], fr[0], s.rw01.x, s.d0);
  fast_wheel_rx2<1>(ss, 1, f.w01.dsum[1], fr[1], s.rw01.y, d1);
  fast_wheel_rx2<-1>(ss, 2, f.w23.dsum[0], fr[2], s.rw23.x, s.d2);
  fast_wheel_rx2<-1>(ss, 3, f.w23.dsum[1], fr[3], s.rw23.y, d3);
  s.d13 = make_float2(d1, d3);
  fast_tick2_core<FFSAT, TRACE, KD0>(f, p, fc, cs, sc, nz, vel, tgt, s);
}

// ---- |u * 1000| < 2^31 for every tick of a chunk that starts in state v -------------------------------
// (int16_t)(A * 1000.0f) is cvttss2si on x86 (out of range -> 0x80000000) and a saturating F2I here; the two
// agree as long as the conversion stays in range, which this bound guarantees from the chunk's constants:
//   |target_a| <= max over the profile (phase 1 closed form, then at most tm / ts + 2 increments of |a23| * ts)
//   |input|    <= GEAR_RATIO * RPM_TO_RADPS * GEAR_RATIO_INV * rpm_max
//   |u|        <= |kp| * (|tgt| + |input|) + i_limit + |kd| * y_max + ff_limit.
// Loose by design (a few percent of slack per step); written so that a NaN anywhere fails the test.
RK_DEV float interp_vel_bound(const Interp &t, float ts) {
  const float t1 = fabsf(t.dt1) + ts, tm = fabsf(t.dt1) + fabsf(t.dt2) + fabsf(t.dt3) + 2.0f * ts;
  const float v1 = fabsf(t.vel_ini) + (2.0f * fabsf(t.acl_ini) + fabsf(t.jerk_p) * t1) * t1;
  const float a23 = fabsf(t.acl_max) + fabsf(t.jerk_m) * (fabsf(t.dt3) + 2.0f * ts);
  return 1.01f * (fmaxf(fmaxf(v1, fabsf(t.vel)), fabsf(t.vel_tgt)) + a23 * (tm + 2.0f * ts));
}
template <bool STREAM>
RK_DEV bool fast_u_bounded(const Veh &v, const rk_vdt_params_t &p, const FastConsts &fc) {
  const float vx = interp_vel_bound(v.it[0], p.ts), vy = interp_vel_bound(v.it[1], p.ts), vt = interp_vel_bound(v.it[2], p.ts);
  const float tgt = 1.01f * RK_GEAR_RATIO * (vx + vy + 4.0f * fabsf(fc.s2l) * vt) * fabsf(fc.rcp_r);
  const float rpm_max = STREAM ? 32768.0f : 4.0f * (float)p.raw_curr_lim + 16.0f;
  float       now     = 1.01f * RK_GEAR_RATIO * RK_RPM_TO_RADPS * RK_GEAR_RATIO_INV * rpm_max;
  float       y0 = 0.0f, x0 = 0.0f;
#pragma unroll
  for(int k = 0; k < 4; k++) now = fmaxf(now, fabsf(v.c[k].prev_val)), y0 = fmaxf(y0, fabsf(v.c[k].lpf_y)), x0 = fmaxf(x0, fabsf(v.c[k].lpf_x));
  const float xmax = fmaxf(x0, 2.0f * now * fabsf(p.ctrl_freq));
  if(!(fabsf(fc.A1) < 0.999f)) return false;
  const float ymax = fmaxf(y0, 1.01f * 2.0f * fabsf(fc.B0) * xmax / (1.0f - fabsf(fc.A1)));
  const float u    = fabsf(p.kp) * (tgt + now) + fabsf(p.i_limit) + fabsf(p.kd) * ymax + fabsf(p.ff_limit);
  return 1.01f * RK_AMPERE_TO_RAW_CURR * u < 2.0e9f; // false for NaN
}

} // namespace rk
