// rk_imu.cu -- IMU_IF_WT901C::update()/updateData()/init() batched (src/Imu/imu_if_wt901c.cpp).
//
// One thread per IMU, q_init and the readable Data page held in registers.  When the caller wants every sample's
// output (or yaw), the K fused updates stream: per update 32 B of registers in (two 128-bit cells, the next update in
// flight) and 64 B out (four 128-bit stores) -- HBM-bound.  Without per-update output only the last sample with a
// quaternion frame decides the end state, so that one sample is read (imt_last_frame).
#include <string.h>

#include <type_traits>

#include "rk_common.cuh"
#include "rk_math.cuh"
#include "rk_stream.cuh"

namespace rk {

struct ImuData {
  float d[16]; // IMU_IF::Data in struct order (imu_if_base.hpp:12-18)
};

// IMU_IF_WT901C::updateData  imu_if_wt901c.cpp:91-129:
//   acc = s / 32768 * 16, gyro = s / 32768 * 2000, mag = s, angle = s / 32768 * 180, q = s / 32768; Y and Z negated;
//   roll = normalize_0to360(roll) - 180; q_out = the product with q_init in the rows of :123-126 (output order z, y, x, w),
//   left to right, one rounding per operation.
// On the packed snapshot (two int16 registers a word), arranged for the issue slots it takes:
//  * cvt.rn.f32.s16 straight from the register halves (no unpacking);
//  * (x / 32768) * k is ONE multiply by k * 2^-15: the division is an exact scaling, so the product is rounded once
//    either way, and 16 * 2^-15, 2000 * 2^-15, 180 * 2^-15 are exact floats;
//  * the four rows of the quaternion product run as two packed rows: a - p == a + (-p) and (-qi) * q == -(qi * q)
//    exactly, so the inner signs move into eight constant lane pairs formed once per launch from q_init; the two
//    outer negations of rows 14 and 12 stay where they are (they decide the sign of an exact zero).
RK_DEV void cvt2_s16(uint32_t w, float &lo, float &hi) {
  asm("{ .reg .b16 l, h; mov.b32 {l, h}, %2; cvt.rn.f32.s16 %0, l; cvt.rn.f32.s16 %1, h; }" : "=f"(lo), "=f"(hi) : "r"(w));
}
struct ImuQ { // lane pairs {row 14 | row 13} and {row 12 | row 15} of imu_if_wt901c.cpp:123-126, per factor q0..q3
  float2 a[4], b[4];
};
RK_DEV void imu_q_pairs(ImuQ &k, const float qi[4]) {
  k.a[0] = make_float2(qi[3], -qi[2]), k.a[1] = make_float2(qi[2], qi[3]), k.a[2] = make_float2(-qi[1], qi[0]), k.a[3] = make_float2(-qi[0], -qi[1]);
  k.b[0] = make_float2(qi[1], qi[0]), k.b[1] = make_float2(-qi[0], qi[1]), k.b[2] = make_float2(qi[3], qi[2]), k.b[3] = make_float2(-qi[2], qi[3]);
}
RK_DEV float2 imu_mul2(float s, float2 k, float nz) { return __ffma2_rn(make_float2(s, s), k, make_float2(nz, nz)); } // RN(s * k) per lane
RK_DEV void imu_update_data_w(const ImuQ &k, const uint32_t rw[8], float nz, ImuData &o) {
  float f[16];
#pragma unroll
  for(int j = 0; j < 8; j++) cvt2_s16(rw[j], f[2 * j], f[2 * j + 1]);
  const float KA = 16.0f / 32768.0f, KG = 2000.0f / 32768.0f, KE = 180.0f / 32768.0f, S = 1.0f / 32768.0f; // all exact
  o.d[0] = fmul(f[0], KA), o.d[1] = fmul(f[1], -KA), o.d[2] = fmul(f[2], -KA);
  o.d[3] = fmul(f[3], KG), o.d[4] = fmul(f[4], -KG), o.d[5] = fmul(f[5], -KG);
  o.d[6] = f[6], o.d[7] = -f[7], o.d[8] = -f[8];
  o.d[9]  = fsub(normalize_deg_0to360(fmul(f[9], KE)), 180.0f);
  o.d[10] = fmul(f[10], KE);
  o.d[11] = fmul(f[11], KE);
  float q[4];
#pragma unroll
  for(int j = 0; j < 4; j++) q[j] = fmul(f[12 + j], S);
  const float2 ra = __fadd2_rn(__fadd2_rn(__fadd2_rn(imu_mul2(q[0], k.a[0], nz), imu_mul2(q[1], k.a[1], nz)), imu_mul2(q[2], k.a[2], nz)),
                               imu_mul2(q[3], k.a[3], nz));
  const float2 rb = __fadd2_rn(__fadd2_rn(__fadd2_rn(imu_mul2(q[0], k.b[0], nz), imu_mul2(q[1], k.b[1], nz)), imu_mul2(q[2], k.b[2], nz)),
                               imu_mul2(q[3], k.b[3], nz));
  o.d[14] = -ra.x, o.d[13] = ra.y, o.d[12] = -rb.x, o.d[15] = rb.y;
}
// IMU_IF_WT901C::init  :72-75: q_init latched from q0..q3 of the snapshot (words 6 and 7), and the lane pairs rebuilt
RK_DEV void imu_latch_qinit(const uint32_t rw[8], float qi[4], ImuQ &kq) {
  cvt2_s16(rw[6], qi[0], qi[1]), cvt2_s16(rw[7], qi[2], qi[3]);
#pragma unroll
  for(int j = 0; j < 4; j++) qi[j] = fmul(qi[j], 1.0f / 32768.0f);
  imu_q_pairs(kq, qi);
}

// The state block of IMU i (RK_IS_*): q_init, the Data page, the flags word.
RK_DEV void ld_imu(const uint4 *state, int64_t n, int64_t i, float qi[4], ImuData &cur, uint32_t &flags) {
  const uint4 q = ld_plane(state, n, RK_IS_QINIT / 4, i);
  qi[0] = u2f(q.x), qi[1] = u2f(q.y), qi[2] = u2f(q.z), qi[3] = u2f(q.w);
#pragma unroll
  for(int pl = 0; pl < 4; pl++) {
    const uint4 v = ld_plane(state, n, RK_IS_DATA / 4 + pl, i);
    cur.d[4 * pl] = u2f(v.x), cur.d[4 * pl + 1] = u2f(v.y), cur.d[4 * pl + 2] = u2f(v.z), cur.d[4 * pl + 3] = u2f(v.w);
  }
  flags = ld_plane(state, n, RK_IS_FLAGS / 4, i).x;
}
RK_DEV void st_imu(uint4 *state, int64_t n, int64_t i, const float qi[4], const ImuData &cur, uint32_t flags) {
  st_plane(state, n, RK_IS_QINIT / 4, i, make_uint4(f2u(qi[0]), f2u(qi[1]), f2u(qi[2]), f2u(qi[3])));
#pragma unroll
  for(int pl = 0; pl < 4; pl++)
    st_plane(state, n, RK_IS_DATA / 4 + pl, i, make_uint4(f2u(cur.d[4 * pl]), f2u(cur.d[4 * pl + 1]), f2u(cur.d[4 * pl + 2]), f2u(cur.d[4 * pl + 3])));
  st_plane(state, n, RK_IS_FLAGS / 4, i, make_uint4(flags, 0u, 0u, 0u));
}

// The output of update u: the yaw the vehicle ISR reads each tick, mymath::deg2rad(IMT::get_status_now_yaw())
// (VD_task_main.cpp:368, imu_task_main.cpp:102-104, util_mymath.hpp:13,16), when want_yaw, and the Data page as four
// float4 planes, when want_out.
RK_DEV void imu_publish(const ImuData &cur, int u, int64_t n, int64_t i, float4 *out, bool want_out, float *yaw_rad, bool want_yaw) {
  if(want_yaw) __stcs(yaw_rad + (int64_t)u * n + i, fmul(cur.d[RK_IS_D_ANGLE + 2], RK_DEG2RAD));
  if(want_out) {
#pragma unroll
    for(int pl = 0; pl < 4; pl++)
      __stcs(out + ((int64_t)u * 4 + pl) * n + i, make_float4(cur.d[4 * pl], cur.d[4 * pl + 1], cur.d[4 * pl + 2], cur.d[4 * pl + 3]));
  }
}

// A launch without per-update output (the full tick's IMU, a boot init): nobody reads the Data page between updates, and
// each update either assigns all 16 words of the page from its own sample and q_init (quaternion frame: ::update :83-89
// clears the error bit) or leaves the page as it is and sets the error bit.  q_init changes only in the init on sample 0.
// So the end state is a closed form of the flags and ONE sample:
//   Data page = updateData(the last sample in [u0, K) with a frame), or the page from launch entry if none has one;
//   error bit = !have[K - 1] (unchanged if [u0, K) is empty);  q_init = what it was, or what the init latched;
// u0 = do_init ? 1 : 0.  One backward scan of the flags (one step unless the last sample dropped its frame) and one sample
// read or draw instead of K updates -- the same function of the same sample, so the same bits as the update loop.
template <bool GEN>
RK_DEV void imt_last_frame(int64_t i, int64_t n, int K, const int16_t *__restrict__ regs, const uint8_t *__restrict__ have_quat, int do_init,
                           float nz, const rk_stream_desc_t &sd, float qi[4], ImuData &cur, uint32_t &flags) {
  const uint32_t px = GEN ? h32_prefix(sd.seed, 20u, (uint64_t)(sd.first + i)) : 0u;
  auto sample = [&](int u, uint32_t rw[8]) { // sample u's two 128-bit cells
    uint4 c0, c1;
    if(GEN) {
      bool h;
      stream_imu_sample(px, sd.first_update + (uint32_t)u, sd.drop_every, c0, c1, h);
    } else {
      const uint4 *src = (const uint4 *)regs + (int64_t)u * 2 * n + i;
      c0 = __ldcs(src), c1 = __ldcs(src + n);
    }
    rw[0] = c0.x, rw[1] = c0.y, rw[2] = c0.z, rw[3] = c0.w, rw[4] = c1.x, rw[5] = c1.y, rw[6] = c1.z, rw[7] = c1.w;
  };
  auto have = [&](int u) -> bool { // have_quat == NULL: every sample carries a frame
    if(GEN) return stream_imu_have(px, sd.first_update + (uint32_t)u, sd.drop_every);
    return !have_quat || __ldcs(have_quat + (int64_t)u * n + i) != 0;
  };
  ImuQ     kq;
  uint32_t rw[8];
  imu_q_pairs(kq, qi);
  int u0 = 0;
  if(do_init && K > 0) { // IMU_IF_WT901C::init  :63-77: updateData against the current q_init, then latch q_init
    sample(0, rw);
    imu_update_data_w(kq, rw, nz, cur);
    imu_latch_qinit(rw, qi, kq);
    u0 = 1;
  }
  if(u0 >= K) return;
  int u = K - 1;
  while(u >= u0 && !have(u)) u--;
  if(u == K - 1) flags &= ~RK_IS_FLAG_ERROR;
  else flags |= RK_IS_FLAG_ERROR;
  if(u >= u0) {
    sample(u, rw);
    imu_update_data_w(kq, rw, nz, cur);
  }
}

// OUT / YAW: every update's page (or yaw) is stored, so every update runs; otherwise imt_last_frame.
// GEN: the register snapshots are not read from a table but drawn in registers from the stream descriptor (the same
// stream_imu_sample() the table generator runs, so the samples are those of rk_stream_imu_samples bit for bit): a planner
// that samples its sensor noise on the device never materialises 3.2 KB of snapshots per robot and launch.  Only the
// collapsed update draws, so GEN is given to imt_last_frame alone.
template <bool OUT, bool YAW, bool GEN>
RK_DEV void imt_update_body(int64_t i, uint4 *__restrict__ state, int64_t n, int K, const int16_t *__restrict__ regs,
                            const uint8_t *__restrict__ have_quat, float4 *__restrict__ out, float *__restrict__ yaw_rad, int do_init,
                            float nz, const rk_stream_desc_t &sd) {
  static_assert(!(GEN && (OUT || YAW)), "samples are drawn only by the collapsed update (imt_last_frame)");
  float    qi[4];
  ImuData  cur;
  uint32_t flags;
  ld_imu(state, n, i, qi, cur, flags);
  if constexpr(!OUT && !YAW) {
    imt_last_frame<GEN>(i, n, K, regs, have_quat, do_init, nz, sd, qi, cur, flags);
  } else {
    // the register snapshot is two 128-bit cells; the loads of update u + 1 are in flight while update u is
    // computed and stored.  Pointers advance by one sample per update.
    const uint4   *src = (const uint4 *)regs + i;
    const uint8_t *hsrc = have_quat ? have_quat + i : nullptr;
    uint4          c0 = make_uint4(0u, 0u, 0u, 0u), c1 = c0;
    bool           nhq = true;
    auto           fetch = [&]() {
      c0 = __ldcs(src), c1 = __ldcs(src + n);
      src += 2 * n;
      if(hsrc) nhq = __ldcs(hsrc) != 0, hsrc += n;
    };
    // called through a lambda: called directly, imu_publish changes how ptxas schedules this loop
    auto publish = [&](int u) { imu_publish(cur, u, n, i, out, OUT, yaw_rad, YAW); };
    if(K > 0) fetch();
    ImuQ kq;
    imu_q_pairs(kq, qi);
    int u = 0;
    if(do_init && K > 0) { // IMU_IF_WT901C::init  :63-77: updateData against the current q_init, then latch q_init
      const uint32_t rw[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
      if(K > 1) fetch();
      imu_update_data_w(kq, rw, nz, cur);
      imu_latch_qinit(rw, qi, kq);
      publish(0);
      u = 1;
    }
    for(; u < K; u++) {
      const uint32_t rw[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
      const bool     hq    = nhq;
      if(u + 1 < K) fetch();
      if(hq) { // ::update  :83-89
        flags &= ~RK_IS_FLAG_ERROR;
        imu_update_data_w(kq, rw, nz, cur);
      } else {
        flags |= RK_IS_FLAG_ERROR; // previous page stays readable
      }
      publish(u);
    }
  }
  st_imu(state, n, i, qi, cur, flags);
}
// One thread per IMU; the grid may be smaller than the batch (rk_tick_rollout runs this kernel beside the
// issue-bound vehicle rollout on a capped number of CTAs), so CTAs stride over the blocks of 256 IMUs.
// nz_src: any finite positive float; -0.0f is formed from it at run time so that ptxas cannot fold the packed
// products' "+ (-0)" into the adds that follow (see rk_vehicle_fast2.cuh).
template <bool OUT, bool YAW, bool GEN>
__global__ void __launch_bounds__(256, 4) // 64 registers: one CTA fits the slot a retiring vehicle CTA frees (rk_tick.cu)
imt_update_kernel(uint4 *__restrict__ state, int64_t n, int K, const int16_t *__restrict__ regs,
                  const uint8_t *__restrict__ have_quat, float4 *__restrict__ out, float *__restrict__ yaw_rad, int do_init, float nz_src,
                  const rk_stream_desc_t *__restrict__ desc) {
  const float            nz = fmul(-0.0f, nz_src);
  const rk_stream_desc_t sd = GEN ? *desc : rk_stream_desc_t{};
  for(int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    imt_update_body<OUT, YAW, GEN>(i, state, n, K, regs, have_quat, out, yaw_rad, do_init, nz, sd);
}

// ---------------------------------------------------------------------------------------------
// WIT serial codec (lib/wt901c/wit_c_sdk.c:77-164): the vendor parser's byte-wise state machine, one
// thread per IMU.  WitSerialDataIn does one of two things with a byte: while the window head is 0x55
// it appends (and tests the checksum when the window reaches 11 bytes), otherwise it appends and
// drops the head -- the window slides by one.  So whole runs of bytes are appended at once while the
// head is 0x55 and no frame can complete inside the run; single bytes are handled only while sliding.
// The window is a 96-bit shift register (w2:w1:w0) whose TOP cnt bytes are the parser's buffer, oldest
// byte lowest: appending k bytes is three funnel shifts by 8k, dropping the head is cnt-- and a full
// frame always sits at fixed positions (bytes 1..11).  Bytes arrive as 128-bit cells through a
// shared-memory ring the TMA unit keeps sixteen cell planes ahead (see imt_feed_bytes_kernel).
// ---------------------------------------------------------------------------------------------
struct Wit {
  uint32_t w0, w1, w2, cnt, flags;
  bool     head_ok; // cnt != 0 and the oldest byte of the window is 0x55
  uint32_t rw[8];   // the 16 tracked sReg words, two int16 per register (RK_IMT_REG_* order, even slot in the low half)
};
RK_DEV void wit_push(Wit &p, uint32_t R, uint32_t k) { // shift the low k (1..4) bytes of R in at the top
  const uint32_t s = 8u * k;
  p.w0 = __funnelshift_rc(p.w0, p.w1, s);
  p.w1 = __funnelshift_rc(p.w1, p.w2, s);
  p.w2 = __funnelshift_rc(p.w2, R, s);
}
RK_DEV bool wit_head_is_55(const Wit &p) { // byte at offset 12 - cnt of the register, cnt in 1..11
  const uint32_t off = 12u - p.cnt, w = off < 4u ? p.w0 : (off < 8u ? p.w1 : p.w2);
  return ((w >> (8u * (off & 3u))) & 0xFFu) == 0x55u;
}
RK_DEV void wit_store_reg(Wit &p, uint32_t reg, uint32_t val) { // CopeWitData's memcpy into sReg, tracked registers only
  const uint32_t slot = (reg >= 0x34u && reg <= 0x3Fu) ? reg - 0x34u : ((reg >= 0x51u && reg <= 0x54u) ? reg - 0x51u + 12u : 0xFFu);
#pragma unroll
  for(int k = 0; k < 8; k++) {
    if(slot == 2u * k) p.rw[k] = __byte_perm(p.rw[k], val, 0x3254);     // low half
    if(slot == 2u * k + 1u) p.rw[k] = __byte_perm(p.rw[k], val, 0x5410); // high half
  }
  if(reg == 0x54u) p.flags |= 1u; // q3 -> QUAT_UPDATE (SensorDataUpdata)
}
// CopeWitData :77-130 for a frame with a good checksum: which registers the four data words (d01 = d0 | d1 << 16,
// d23 = d2 | d3 << 16) land in.  The frame type differs from lane to lane and the register file is live across it, so
// the five fixed types are selects on the packed words; only WIT_REGVALUE (a dynamic register index) branches.
RK_DEV void wit_dispatch(Wit &p, uint32_t type, uint32_t d01, uint32_t d23) {
  const bool acc = type == 0x51u, gyr = type == 0x52u, ang = type == 0x53u, mag = type == 0x54u, qut = type == 0x59u;
  const uint32_t d12 = __byte_perm(d01, d23, 0x5432); // d1 | d2 << 16
  p.rw[0] = acc ? d01 : p.rw[0];                                                                   // AX AY      <- WIT_ACC (+ TEMP)
  p.rw[1] = acc ? __byte_perm(p.rw[1], d23, 0x3254) : (gyr ? __byte_perm(p.rw[1], d01, 0x5410) : p.rw[1]); // AZ | GX
  p.rw[2] = gyr ? d12 : p.rw[2];                                                                   // GY GZ      <- WIT_GYRO
  p.rw[3] = mag ? d01 : p.rw[3];                                                                   // HX HY      <- WIT_MAGNETIC
  p.rw[4] = mag ? __byte_perm(p.rw[4], d23, 0x3254) : (ang ? __byte_perm(p.rw[4], d01, 0x5410) : p.rw[4]); // HZ | Roll
  p.rw[5] = ang ? d12 : p.rw[5];                                                                   // Pitch Yaw  <- WIT_ANGLE (+ VERSION)
  p.rw[6] = qut ? d01 : p.rw[6];                                                                   // q0 q1      <- WIT_QUATER
  p.rw[7] = qut ? d23 : p.rw[7];                                                                   // q2 q3
  p.flags |= qut ? 1u : 0u;
  if(type == 0x5Fu) { // WIT_REGVALUE: four registers from s_uiReadRegIndex
    const uint32_t r = (p.flags >> 8) & 0xFFu;
    wit_store_reg(p, r, d01 & 0xFFFFu), wit_store_reg(p, r + 1, d01 >> 16), wit_store_reg(p, r + 2, d23 & 0xFFFFu), wit_store_reg(p, r + 3, d23 >> 16);
  }
  // TIME / DPORT / PRESS / GPS / VELOCITY / GSA write registers the IMU interface never reads; other types are ignored
}
RK_DEV void wit_frame(Wit &p) { // a full window: bytes 1..11 of the shift register
  const uint32_t f0 = __funnelshift_r(p.w0, p.w1, 8), f1 = __funnelshift_r(p.w1, p.w2, 8), f2 = p.w2 >> 8;
  wit_dispatch(p, (f0 >> 8) & 0xFFu, __byte_perm(f0, f1, 0x5432), __byte_perm(f1, f2, 0x5432));
}
// Healthy traffic is frames back to back.  With the window empty and 11 bytes of this update at hand, a frame that
// starts right here with a good checksum is what the byte machine would accept after appending those 11 bytes one by
// one -- nothing else can happen on the way -- so it is taken in one step; anything else goes through wit_bytes().
// f0, f1, f2: the 11 bytes, first byte in the low byte of f0.
RK_DEV bool wit_try_frame(Wit &p, uint32_t f0, uint32_t f1, uint32_t f2) {
  if((f0 & 0xFFu) != 0x55u) return false;
  const uint32_t sum = __vsadu4(f0, 0u) + __vsadu4(f1, 0u) + __vsadu4(f2 & 0xFFFFu, 0u);
  if((sum & 0xFFu) != ((f2 >> 16) & 0xFFu)) return false;
  wit_dispatch(p, (f0 >> 8) & 0xFFu, __byte_perm(f0, f1, 0x5432), __byte_perm(f1, f2, 0x5432));
  return true;
}
// `rem` (<= 4) bytes, first byte in the low byte of R: WitSerialDataIn for each  :132-164
RK_DEV void wit_bytes(Wit &p, uint32_t R, uint32_t rem) {
  while(rem) {
    if(p.cnt == 0u) p.head_ok = (R & 0xFFu) == 0x55u;
    if(p.head_ok) { // appending: nothing happens before the window is full
      const uint32_t take = min(rem, 11u - p.cnt);
      wit_push(p, R, take);
      p.cnt += take;
      R = __funnelshift_rc(R, 0u, 8u * take);
      rem -= take;
      if(p.cnt == 11u) {
        const uint32_t sum = __vsadu4(p.w0 & 0xFFFFFF00u, 0u) + __vsadu4(p.w1, 0u) + __vsadu4(p.w2 & 0x00FFFFFFu, 0u);
        if((sum & 0xFFu) == (p.w2 >> 24)) {
          wit_frame(p);
          p.cnt = 0u; // s_uiWitDataCnt = 0
        } else { // drop the head: the type byte is the new one
          p.cnt     = 10u;
          p.head_ok = ((p.w0 >> 16) & 0xFFu) == 0x55u;
        }
      }
    } else { // sliding: append one byte, drop the head (a no-op on an empty window)
      if(p.cnt) {
        wit_push(p, R, 1u);
        p.head_ok = wit_head_is_55(p);
      }
      R >>= 8;
      rem--;
    }
  }
}
// The bytes of cell A that are still to parse, byte-exact: A holds bytes [lo, lo + 16) of an update of nb bytes, B the
// next 16 when `next` (a frame may straddle into it); done counts the update's bytes parsed so far.
RK_DEV void wit_cell(Wit &p, const uint4 A, const uint4 B, uint32_t lo, uint32_t nb, bool next, uint32_t &done) {
  const uint32_t end = min(nb, lo + 16u), span = min(nb, next ? lo + 32u : lo + 16u);
  while(done < end) {
    const uint32_t off = done - lo, wi = off >> 2, sh = 8u * (off & 3u);
    const uint32_t x0 = wi == 0u ? A.x : (wi == 1u ? A.y : (wi == 2u ? A.z : A.w));
    if(p.cnt == 0u && span - done >= 11u) {
      const uint32_t x1 = wi == 0u ? A.y : (wi == 1u ? A.z : (wi == 2u ? A.w : B.x));
      const uint32_t x2 = wi == 0u ? A.z : (wi == 1u ? A.w : (wi == 2u ? B.x : B.y));
      const uint32_t x3 = wi == 0u ? A.w : (wi == 1u ? B.x : (wi == 2u ? B.y : B.z));
      if(wit_try_frame(p, __funnelshift_r(x0, x1, sh), __funnelshift_r(x1, x2, sh), __funnelshift_r(x2, x3, sh))) {
        done += 11u;
        continue;
      }
    }
    const uint32_t k = min(4u - (off & 3u), end - done); // the rest of this word, byte by byte semantics
    wit_bytes(p, x0 >> sh, k);
    done += k;
  }
}
RK_DEV void wit_load(Wit &p, const uint4 a) { // parser block plane 0: window left-aligned, zeros past the count
  p.cnt = min(a.z >> 24, 10u);                 // the window never rests full
  p.w0 = a.x, p.w1 = a.y, p.w2 = a.z & 0x00FFFFFFu, p.flags = a.w;
  p.head_ok = p.cnt && (p.w0 & 0xFFu) == 0x55u;
  for(uint32_t k = p.cnt; k < 12u; k++) { // move the cnt bytes to the top
    p.w2 = __funnelshift_l(p.w1, p.w2, 8);
    p.w1 = __funnelshift_l(p.w0, p.w1, 8);
    p.w0 <<= 8;
  }
}
RK_DEV uint4 wit_save(const Wit &p) {
  uint32_t w0 = p.w0, w1 = p.w1, w2 = p.w2;
  for(uint32_t k = p.cnt; k < 12u; k++) {
    w0 = __funnelshift_r(w0, w1, 8);
    w1 = __funnelshift_r(w1, w2, 8);
    w2 >>= 8;
  }
  return make_uint4(w0, w1, w2 | (p.cnt << 24), p.flags);
}

// ---- mbarrier + bulk async copy (TMA 1-D) primitives, sm_90+/sm_100a PTX --------------------------------
RK_DEV uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
RK_DEV void mbar_init(uint64_t *bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }
RK_DEV void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
RK_DEV void mbar_arrive(uint64_t *bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
RK_DEV void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
RK_DEV void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while(!ok);
}
// global -> shared bulk copy by the TMA unit, completion counted in bytes on `bar`
RK_DEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// The wire arrives through a ring of kWireStages shared-memory stages per CTA, one stage = the 128 consecutive cells
// of one cell plane (2 KB), filled by bulk async copies that thread 0 keeps kWireStages cells ahead: the byte
// automaton's irregular pace never exposes HBM latency and no registers are spent on prefetch.  full[s] flips when
// the bytes have landed, empty[s] when the four warps have taken their cells out of the stage.
constexpr int kWireStages = 16;

// NC4: every update brings four cells (the 55-byte WT901 burst of one 100 Hz period fits).  The update's 16 words are
// then in registers at once, and the frames that sit back to back from the start of the update -- the healthy case --
// are taken at STATIC byte offsets 0, 11, 22, 33, 44 (wit_try_frame on constant funnel shifts); whatever does not fit
// that pattern goes through the byte-exact walk of the generic path (wit_cell).
template <bool NC4>
__global__ void __launch_bounds__(128)
imt_feed_bytes_kernel(uint4 *__restrict__ state, uint4 *__restrict__ parser, int64_t n, int K, int ncells, const uint4 *__restrict__ cells,
                      const uint16_t *__restrict__ nbytes, float4 *__restrict__ out, float *__restrict__ yaw_rad, int do_init, float nz_src) {
  __shared__ __align__(128) uint4 ring[kWireStages][128];
  __shared__ __align__(8) uint64_t full_bar[kWireStages], empty_bar[kWireStages];
  const int      tid = threadIdx.x;
  const int64_t  i0 = (int64_t)blockIdx.x * 128, i = i0 + tid;
  const bool     live = i < n; // idle lanes of the last CTA still take part in the stage hand-over
  const uint32_t row_bytes = (uint32_t)min((int64_t)128, n - i0) * 16u;
  const int64_t  total = (int64_t)K * ncells;
  if(tid == 0) {
    for(int s = 0; s < kWireStages; s++) mbar_init(&full_bar[s], 1u), mbar_init(&empty_bar[s], 4u);
    mbar_fence_init();
  }
  __syncthreads();
  auto issue = [&](int64_t T) { // thread 0: cell plane T -> its stage
    const int s = (int)(T % kWireStages);
    mbar_arrive_expect_tx(&full_bar[s], row_bytes);
    bulk_g2s(&ring[s][0], cells + T * n + i0, row_bytes, &full_bar[s]);
  };
  if(tid == 0)
    for(int64_t T = 0; T < total && T < kWireStages; T++) issue(T);
  auto fetch = [&](int64_t T) -> uint4 { // this thread's cell of plane T; the stage is refilled once all four warps are through
    const int      s   = (int)(T % kWireStages);
    const uint32_t par = (uint32_t)((T / kWireStages) & 1);
    mbar_wait(&full_bar[s], par);
    const uint4 v = ring[s][tid];
    __syncwarp();
    if((tid & 31) == 0) mbar_arrive(&empty_bar[s]);
    if(tid == 0 && T + kWireStages < total) {
      mbar_wait(&empty_bar[s], par);
      issue(T + kWireStages);
    }
    return v;
  };

  float    qi[4];
  ImuData  cur;
  uint32_t flags;
  Wit      p;
  const int64_t il = live ? i : 0; // idle lanes read instance 0 and never write
  ld_imu(state, n, il, qi, cur, flags);
  {
    const uint4 a = ld_plane(parser, n, 0, il), b = ld_plane(parser, n, 1, il), c = ld_plane(parser, n, 2, il);
    wit_load(p, a);
    p.rw[0] = b.x, p.rw[1] = b.y, p.rw[2] = b.z, p.rw[3] = b.w, p.rw[4] = c.x, p.rw[5] = c.y, p.rw[6] = c.z, p.rw[7] = c.w;
  }
  ImuQ kq;
  imu_q_pairs(kq, qi);
  const float nz    = fmul(-0.0f, nz_src);
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  // two cells in registers: A is being parsed, B follows it (a frame may straddle into it)
  uint4    B = (!NC4 && total > 0) ? fetch(0) : zero4; // (generic path: cell t is in B when its update starts)
  int64_t  t = 0;
  uint32_t nb_next = (nbytes && K > 0 && live) ? (uint32_t)__ldcs(nbytes + i) : 0xFFFFFFFFu;
  for(int u = 0; u < K; u++) {
    const bool init = do_init && u == 0;
    if(init) { // WitInit: s_uiWitDataCnt = 0 ; WitReadReg(q0, 4): s_uiReadRegIndex = q0
      p.cnt   = 0u;
      p.flags = (p.flags & ~0xFF00u) | (0x51u << 8) | RK_IP_FLAG_INIT_PENDING;
    }
    const uint32_t nb = live ? min(nb_next, 16u * (uint32_t)ncells) : 0u; // bytes on the wire in this update
    if(nbytes && live && u + 1 < K) nb_next = (uint32_t)__ldcs(nbytes + (int64_t)(u + 1) * n + i); // consumed an update later
    uint32_t done = 0u; // bytes of this update already parsed
    if(NC4) {
      uint32_t w[17]; // the update's 64 bytes (+ a zero word for the shifts at the end)
#pragma unroll
      for(int c = 0; c < 4; c++) {
        const uint4 v = fetch(t++);
        w[4 * c] = v.x, w[4 * c + 1] = v.y, w[4 * c + 2] = v.z, w[4 * c + 3] = v.w;
      }
      w[16] = 0u;
#pragma unroll
      for(int f = 0; f < 5; f++) { // frame f at byte 11 f, as long as the frames before it were taken whole
        const int  wi = (11 * f) >> 2, sh = 8 * ((11 * f) & 3);
        const bool can = p.cnt == 0u && done == 11u * (uint32_t)f && nb >= 11u * (uint32_t)(f + 1);
        if(can && wit_try_frame(p, __funnelshift_r(w[wi], w[wi + 1], sh), __funnelshift_r(w[wi + 1], w[wi + 2], sh),
                                __funnelshift_r(w[wi + 2], w[wi + 3], sh)))
          done += 11u;
      }
      if(done < nb) // the rest, byte-exact: cell c = words 4c .. 4c + 3, looked up with selects (static register indices)
        for(int c = 0; c < 4; c++) {
          uint4 A, Bc;
          A.x = c == 0 ? w[0] : (c == 1 ? w[4] : (c == 2 ? w[8] : w[12])), A.y = c == 0 ? w[1] : (c == 1 ? w[5] : (c == 2 ? w[9] : w[13]));
          A.z = c == 0 ? w[2] : (c == 1 ? w[6] : (c == 2 ? w[10] : w[14])), A.w = c == 0 ? w[3] : (c == 1 ? w[7] : (c == 2 ? w[11] : w[15]));
          Bc.x = c == 0 ? w[4] : (c == 1 ? w[8] : (c == 2 ? w[12] : 0u)), Bc.y = c == 0 ? w[5] : (c == 1 ? w[9] : (c == 2 ? w[13] : 0u));
          Bc.z = c == 0 ? w[6] : (c == 1 ? w[10] : (c == 2 ? w[14] : 0u)), Bc.w = c == 0 ? w[7] : (c == 1 ? w[11] : (c == 2 ? w[15] : 0u));
          wit_cell(p, A, Bc, 16u * (uint32_t)c, nb, c + 1 < 4, done);
        }
    } else
      for(int c = 0; c < ncells; c++) {
        const uint4 A = B;
        t++;
        B = (t < total) ? fetch(t) : zero4;
        wit_cell(p, A, B, 16u * (uint32_t)c, nb, c + 1 < ncells, done);
      }
    const bool hq = (p.flags & 1u) != 0u; // isComComp :132-143
    if(hq) p.flags &= ~0xFFu;
    // init() -> getDataImmediately (:63-77,149-158) spins in isComComp() until a quaternion frame has arrived: an update
    // slot without one is still part of that wait (nothing is published, q_init is not latched); the slot that brings it
    // completes init.  The pending state lives in the parser block, so it survives slots and launches.
    const bool pending = (p.flags & RK_IP_FLAG_INIT_PENDING) != 0u;
    if(hq) {
      if(!pending) flags &= ~RK_IS_FLAG_ERROR;
      imu_update_data_w(kq, p.rw, nz, cur);
      if(pending) {
        imu_latch_qinit(p.rw, qi, kq);
        p.flags &= ~RK_IP_FLAG_INIT_PENDING;
      }
    } else if(!pending) {
      flags |= RK_IS_FLAG_ERROR;
    }
    if(live) imu_publish(cur, u, n, i, out, out != nullptr, yaw_rad, yaw_rad != nullptr);
  }
  if(!live) return;
  st_imu(state, n, i, qi, cur, flags);
  st_plane(parser, n, 0, i, wit_save(p));
  st_plane(parser, n, 1, i, make_uint4(p.rw[0], p.rw[1], p.rw[2], p.rw[3]));
  st_plane(parser, n, 2, i, make_uint4(p.rw[4], p.rw[5], p.rw[6], p.rw[7]));
}

} // namespace rk

using namespace rk;

// Calls f(std::true_type{}) or f(std::false_type{}): a run-time choice as a kernel's template argument.
template <class F>
static void with_bool(bool b, F &&f) {
  if(b) f(std::true_type{});
  else f(std::false_type{});
}

extern "C" {

size_t rk_imt_state_words(void) { return RK_IS_WORDS; }
size_t rk_imt_state_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_IS_WORDS * 4u; }

int rk_imt_update(void *d_state, int64_t n, int32_t K, const int16_t *d_regs, const uint8_t *d_have_quat, float *d_out,
                  int do_init, void *stream) {
  return rk_imt_update_yaw(d_state, n, K, d_regs, d_have_quat, d_out, nullptr, do_init, stream);
}

int rk_imt_update_yaw(void *d_state, int64_t n, int32_t K, const int16_t *d_regs, const uint8_t *d_have_quat, float *d_out,
                      float *d_yaw_rad, int do_init, void *stream) {
  return rk::imt_update_launch(d_state, n, K, d_regs, d_have_quat, d_out, d_yaw_rad, do_init, 0, stream, nullptr);
}
} // extern "C"

// max_ctas > 0: at most that many CTAs (each strides over the batch)
// d_desc != NULL (and no output page): the samples are drawn from the stream descriptor instead of read from d_regs
int rk::imt_update_launch(void *d_state, int64_t n, int32_t K, const int16_t *d_regs, const uint8_t *d_have_quat, float *d_out,
                          float *d_yaw_rad, int do_init, int max_ctas, void *stream, const void *d_desc) {
  if(n == 0 || K == 0) return RK_OK;
  const bool gen = d_desc != nullptr && !d_out && !d_yaw_rad;
  if(n < 0 || K < 0 || (!gen && !d_regs) || ((uintptr_t)d_regs & 15u) || ((uintptr_t)d_desc & 7u)) {
    set_error("rk_imt_update: bad n / K, or d_regs NULL / not 16-byte aligned");
    return RK_ERR_ARG;
  }
  if(!d_state || ((uintptr_t)d_state & 15u) || ((uintptr_t)d_out & 15u)) {
    set_error("rk_imt_update: d_state/d_out must be 16-byte aligned");
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  unsigned grid = (unsigned)((n + 255) / 256);
  if(max_ctas > 0 && grid > (unsigned)max_ctas) grid = (unsigned)max_ctas;
  const auto launch = [&](auto out, auto yaw, auto draw) {
    imt_update_kernel<out, yaw, draw><<<grid, 256, 0, (cudaStream_t)stream>>>((uint4 *)d_state, n, K, d_regs, d_have_quat, (float4 *)d_out,
                                                                            d_yaw_rad, do_init, 1.0f, (const rk_stream_desc_t *)d_desc);
  };
  if(gen) launch(std::false_type{}, std::false_type{}, std::true_type{});
  else with_bool(d_out != nullptr, [&](auto out) { with_bool(d_yaw_rad != nullptr, [&](auto yaw) { launch(out, yaw, std::false_type{}); }); });
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

extern "C" {

size_t rk_imt_parser_words(void) { return RK_IP_WORDS; }
size_t rk_imt_parser_bytes(int64_t n) { return n < 0 ? 0 : (size_t)n * RK_IP_WORDS * 4u; }

int rk_imt_feed_bytes(void *d_state, void *d_parser, int64_t n, int32_t K, int32_t ncells, const void *d_cells, const uint16_t *d_nbytes,
                      float *d_out, float *d_yaw_rad, int do_init, void *stream) {
  if(n == 0 || K == 0) return RK_OK;
  if(n < 0 || K < 0 || ncells < 0 || ncells > 4095 || (ncells > 0 && !d_cells)) {
    set_error("rk_imt_feed_bytes: bad n / K / ncells / cells");
    return RK_ERR_ARG;
  }
  if(!d_state || !d_parser || ((uintptr_t)d_state & 15u) || ((uintptr_t)d_parser & 15u) || ((uintptr_t)d_out & 15u) ||
     ((uintptr_t)d_cells & 15u) || ((uintptr_t)d_nbytes & 1u)) {
    set_error("rk_imt_feed_bytes: d_state / d_parser / d_cells / d_out must be 16-byte aligned (state and parser non-NULL)");
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  with_bool(ncells == 4, [&](auto nc4) {
    imt_feed_bytes_kernel<nc4><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        (uint4 *)d_state, (uint4 *)d_parser, n, K, ncells, (const uint4 *)d_cells, d_nbytes, (float4 *)d_out, d_yaw_rad, do_init, 1.0f);
  });
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

// The handle's blocks live in ONE mapped pinned allocation (zero-copy): the kernel reads the register snapshot and
// reads / writes the state over the bus, the host writes inputs and reads the state directly -- no cudaMemcpy anywhere;
// a getter synchronises the stream only if a launch is still in flight.
struct rk_imt {
  uint32_t    *h_mem = nullptr;  // mapped pinned: [0, RK_IS_WORDS) state, then 16 int16 registers, then the have_quat byte
  cudaStream_t st    = nullptr;
  bool         in_flight = false;
  uint32_t *state() { return h_mem; }
  int16_t  *regs() { return (int16_t *)(h_mem + RK_IS_WORDS); }
  uint8_t  *flag() { return (uint8_t *)(h_mem + RK_IS_WORDS + 8); }
};
static int imt_settle(rk_imt *h) {
  if(h->in_flight) {
    RK_CUDA(cudaStreamSynchronize(h->st));
    h->in_flight = false;
  }
  return RK_OK;
}

int rk_imt_create(rk_imt_t **out) {
  if(!out) return RK_ERR_ARG;
  *out = nullptr;
  if(int rc = require_device()) return rc;
  rk_imt     *h = new rk_imt();
  cudaError_t e = cudaHostAlloc((void **)&h->h_mem, (RK_IS_WORDS + 8 + 4) * 4, cudaHostAllocMapped);
  if(e == cudaSuccess) memset(h->h_mem, 0, (RK_IS_WORDS + 8 + 4) * 4);
  if(e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking);
  if(e != cudaSuccess) {
    int rc = cuda_fail(e, "rk_imt_create");
    rk_imt_destroy(h);
    return rc;
  }
  *out = h;
  return RK_OK;
}
void rk_imt_destroy(rk_imt_t *h) {
  if(!h) return;
  if(h->st) {
    cudaStreamSynchronize(h->st);
    cudaStreamDestroy(h->st);
  }
  if(h->h_mem) cudaFreeHost(h->h_mem);
  delete h;
}
static int imt_step(rk_imt_t *h, const int16_t regs[16], int have_quat, int do_init) {
  if(!h || !regs) return RK_ERR_ARG;
  if(int rc = imt_settle(h)) return rc; // the previous launch may still read the snapshot
  memcpy(h->regs(), regs, 32);
  *h->flag() = (uint8_t)((have_quat || do_init) ? 1 : 0); // no quaternion frame since the last call: is_error = true
  h->in_flight = true;
  return rk_imt_update(h->state(), 1, 1, h->regs(), h->flag(), nullptr, do_init, h->st);
}
int rk_imt_init(rk_imt_t *h, const int16_t regs[RK_IMT_REGS]) { return imt_step(h, regs, 1, 1); }
int rk_imt_update1(rk_imt_t *h, const int16_t regs[RK_IMT_REGS], int have_quat) { return imt_step(h, regs, have_quat, 0); }
int rk_imt_get_state(rk_imt_t *h, uint32_t words[RK_IS_WORDS]) {
  if(!h || !words) return RK_ERR_ARG;
  if(int rc = imt_settle(h)) return rc;
  memcpy(words, h->state(), RK_IS_WORDS * 4);
  return RK_OK;
}
int rk_imt_set_state(rk_imt_t *h, const uint32_t words[RK_IS_WORDS]) {
  if(!h || !words) return RK_ERR_ARG;
  if(int rc = imt_settle(h)) return rc;
  memcpy(h->state(), words, RK_IS_WORDS * 4);
  return RK_OK;
}
int rk_imt_get(rk_imt_t *h, float data[16], int *is_error) {
  uint32_t w[RK_IS_WORDS];
  if(!h || !data) return RK_ERR_ARG;
  if(int rc = rk_imt_get_state(h, w)) return rc;
  memcpy(data, &w[RK_IS_DATA], 64);
  if(is_error) *is_error = (w[RK_IS_FLAGS] & RK_IS_FLAG_ERROR) ? 1 : 0;
  return RK_OK;
}
int rk_imt_get_yaw(rk_imt_t *h, float *yaw_deg) {
  float d[16];
  if(!yaw_deg) return RK_ERR_ARG;
  if(int rc = rk_imt_get(h, d, nullptr)) return rc;
  *yaw_deg = d[RK_IS_D_ANGLE + 2];
  return RK_OK;
}
}
