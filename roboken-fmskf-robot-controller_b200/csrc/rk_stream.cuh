// rk_stream.cuh -- the counter hash of the synthetic streams (streams.py `*_v2`) and the one-sample IMU draw, shared by
// the table generators (rk_stream.cu) and the IMU update that draws its samples in registers (rk_imu.cu, GEN).
#pragma once
#include "rk_common.cuh"

namespace rk {

RK_DEV uint32_t mix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7FEB352Du;
  x ^= x >> 15;
  x *= 0x846CA68Bu;
  x ^= x >> 16;
  return x;
}
RK_DEV uint32_t h32_prefix(uint32_t seed, uint32_t stream, uint64_t inst) { // the part that does not depend on the index
  return mix32(mix32(seed ^ (stream * 0x9E3779B9u)) ^ (uint32_t)inst);
}
RK_DEV uint32_t h32_idx(uint32_t prefix, uint32_t idx) { return mix32(prefix ^ (idx * 0x85EBCA6Bu)); }
RK_DEV uint32_t sub32(uint32_t h, uint32_t k) { return mix32(h + (k + 1u) * 0x9E3779B9u); }
// k-th draw under an already mixed hash at a fraction of sub32's cost (streams.lite32): one wide multiply by an odd
// per-draw constant (FMA pipe) and one xor of the two halves -- the generators run beside rollouts that are bound by the
// half-rate ALU pipe, so the draws stay off it
RK_DEV uint32_t lite32(uint32_t h, uint32_t k) {
  const uint32_t           m = (0x85EBCA6Bu + 2u * (k + 1u) * 0x9E3779B9u) | 1u;
  const unsigned long long x = (unsigned long long)h * m;
  return (uint32_t)x ^ (uint32_t)(x >> 32);
}
RK_DEV float    u01_32(uint32_t h) { return fmul((float)(h >> 8), 1.0f / 16777216.0f); }


// Whether sample `upd` of streams.imu_samples_v2 carries a quaternion frame.  px = h32_prefix(seed, 20, robot).
RK_DEV bool stream_imu_have(uint32_t px, uint32_t upd, uint32_t drop_every) {
  return drop_every == 0u || (lite32(h32_idx(px, upd), 8u) % drop_every) != 0u;
}
// One WT901 register snapshot of streams.imu_samples_v2: the two 128-bit cells rk_imt_update consumes and the
// quaternion-frame flag.  px = h32_prefix(seed, 20, robot), upd = the sample's update index.
RK_DEV void stream_imu_sample(uint32_t px, uint32_t upd, uint32_t drop_every, uint4 &c0, uint4 &c1, bool &have) {
  const uint32_t b = h32_idx(px, upd);
  uint32_t       w[8];
#pragma unroll
  for(int k = 0; k < 6; k++) w[k] = lite32(b, (uint32_t)k); // AX..Yaw, two registers a word
  const uint32_t w6 = lite32(b, 6u), w7 = lite32(b, 7u);
  const uint32_t gu[4] = {w6 & 0xFFFFu, w6 >> 16, w7 & 0xFFFFu, w7 >> 16};
  float          g[4];
#pragma unroll
  for(int k = 0; k < 4; k++) g[k] = fsub(fmul(fadd((float)gu[k], 0.5f), 1.0f / 32768.0f), 1.0f);
  const float nrm = fsqrt(fadd(fadd(fadd(fmul(g[0], g[0]), fmul(g[1], g[1])), fmul(g[2], g[2])), fmul(g[3], g[3])));
  const float sc  = fdiv(32767.0f, nrm);
  uint32_t    q[4];
#pragma unroll
  for(int k = 0; k < 4; k++) q[k] = (uint32_t)__float2int_rn(fmul(g[k], sc)) & 0xFFFFu;
  w[6] = q[0] | (q[1] << 16), w[7] = q[2] | (q[3] << 16);
  c0 = make_uint4(w[0], w[1], w[2], w[3]), c1 = make_uint4(w[4], w[5], w[6], w[7]);
  have = stream_imu_have(px, upd, drop_every);
}
// only what the vehicle needs of a sample: the Yaw register and the flag
RK_DEV void stream_imu_yaw(uint32_t px, uint32_t upd, uint32_t drop_every, int16_t &yaw, bool &have) {
  yaw  = (int16_t)(lite32(h32_idx(px, upd), 5u) >> 16);
  have = stream_imu_have(px, upd, drop_every);
}

} // namespace rk
