// rk_plan.cu -- the two ends of a planning step around rk_plan_rollout (rk_vehicle.cu): candidate commands sampled
// around a nominal plan, and the per-robot choice among the candidates' costs (include/robotick.h, "Vehicle sampling
// planner").  Candidate j of robot r is instance r*S + j, so a robot's S candidates are contiguous in every table.
#include <limits.h>
#include <math.h>

#include "rk_stream.cuh"

#ifndef RK_PLAN_BLOCK
#define RK_PLAN_BLOCK 256
#endif

namespace rk {

constexpr uint32_t kPlanStream = 40u; // counter-hash stream of the candidate noise (streams.plan_commands_v2)

// Irwin-Hall sum of four uniforms, centred and scaled to unit variance
RK_DEV float plan_xi(uint32_t h, uint32_t a) {
  const float u0 = u01_32(lite32(h, 4u * a + 0u)), u1 = u01_32(lite32(h, 4u * a + 1u));
  const float u2 = u01_32(lite32(h, 4u * a + 2u)), u3 = u01_32(lite32(h, 4u * a + 3u));
  return fmul(fsub(fadd(fadd(fadd(u0, u1), u2), u3), 2.0f), 1.7320508f);
}

struct PlanSampleArgs {
  int64_t  first, R;
  int32_t  S, n_seg;
  uint32_t seed;
  float    sigma[3], limit_speed, limit_rot;
};

// one thread per (segment, candidate): blockIdx.y strides the segments, x runs over the R*S candidates of one segment
__global__ void __launch_bounds__(RK_PLAN_BLOCK)
plan_sample_kernel(const PlanSampleArgs a, const uint4 *__restrict__ nominal, uint4 *__restrict__ cmd) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = a.R * (int64_t)a.S;
  if(c >= n) return;
  const int64_t  r  = c / a.S;
  const uint32_t j  = (uint32_t)(c - r * a.S);
  const uint32_t px = h32_prefix(a.seed, kPlanStream, (uint64_t)(a.first + r));
  for(int s = blockIdx.y; s < a.n_seg; s += gridDim.y) {
    const uint4 nq = __ldg(nominal + (int64_t)s * a.R + r); // the S candidates of a robot share the cell
    float       v[3] = {u2f(nq.x), u2f(nq.y), u2f(nq.z)};
    if(j != 0u) {
      const uint32_t h = h32_idx(px, (uint32_t)s * (uint32_t)a.S + j);
#pragma unroll
      for(int ax = 0; ax < 3; ax++) v[ax] = fadd(v[ax], fmul(a.sigma[ax], plan_xi(h, (uint32_t)ax)));
    }
    // speed_limit_xy / speed_limit_rot (VD_task_main.cpp:127-142): a vector inside the limits passes unchanged
    const float ln = fsqrt(fadd(fmul(v[0], v[0]), fmul(v[1], v[1])));
    if(ln > a.limit_speed) v[0] = fdiv(fmul(v[0], a.limit_speed), ln), v[1] = fdiv(fmul(v[1], a.limit_speed), ln);
    v[2] = (v[2] > a.limit_rot) ? a.limit_rot : ((v[2] < -a.limit_rot) ? -a.limit_rot : v[2]);
    __stcs(cmd + (int64_t)s * n + c, make_uint4(f2u(v[0]), f2u(v[1]), f2u(v[2]), (uint32_t)RK_CMD_MOVE));
  }
}

// NaN counts as +inf; (key, j) compared lexicographically, so ties go to the lowest j
RK_DEV float plan_key(float c) { return isnan(c) ? __int_as_float(0x7F800000) : c; }
RK_DEV bool  plan_better(float k, int j, float bk, int bj) { return k < bk || (k == bk && j < bj); }
RK_DEV float warp_sum(float x) { // the same fixed butterfly in every lane: every lane ends with identical bits
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) x = fadd(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
  return x;
}
// MPPI weight of candidate cost c against the robot's minimum; 0 for a NaN cost (and for NaN from inf - inf)
RK_DEV float plan_weight(float c, float cmin, float lambda) {
  const float w = expf(-fdiv(fsub(c, cmin), lambda));
  return isnan(w) ? 0.0f : w;
}

// one warp per robot, lanes striding over the S contiguous candidates
__global__ void __launch_bounds__(RK_PLAN_BLOCK)
plan_select_kernel(const float *__restrict__ cost, const uint4 *__restrict__ cmd, int64_t R, int S, int n_seg, float lambda, int shift,
                   uint4 *__restrict__ nom, int32_t *__restrict__ best_out, float *__restrict__ best_cost_out) {
  const int64_t r    = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int     lane = threadIdx.x & 31;
  if(r >= R) return; // whole warps leave together
  const int64_t n  = R * (int64_t)S;
  const float  *cr = cost + r * S;

  float bk = __int_as_float(0x7F800000);
  int   bj = INT_MAX;
  for(int j = lane; j < S; j += 32) {
    const float k = plan_key(__ldg(cr + j));
    if(plan_better(k, j, bk, bj)) bk = k, bj = j;
  }
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) {
    const float k = __shfl_xor_sync(0xFFFFFFFFu, bk, o);
    const int   j = __shfl_xor_sync(0xFFFFFFFFu, bj, o);
    if(plan_better(k, j, bk, bj)) bk = k, bj = j;
  }
  const int best = bj; // S >= 1: some lane saw j = 0
  if(lane == 0) {
    if(best_out) best_out[r] = best;
    if(best_cost_out) best_cost_out[r] = __ldg(cr + best);
  }

  float wsum = 0.0f;
  if(lambda > 0.0f) {
    for(int j = lane; j < S; j += 32) wsum = fadd(wsum, plan_weight(__ldg(cr + j), bk, lambda));
    wsum = warp_sum(wsum);
  }
  if(!(wsum > 0.0f)) { // lambda == 0, or no finite minimum: candidate `best`, bit for bit, one lane per segment
    for(int s = lane; s < n_seg; s += 32) {
      const int ss = min(s + shift, n_seg - 1);
      nom[(int64_t)s * R + r] = __ldg(cmd + (int64_t)ss * n + r * S + best);
    }
    return;
  }
  for(int s = 0; s < n_seg; s++) {
    const int    ss = min(s + shift, n_seg - 1);
    const uint4 *cs = cmd + (int64_t)ss * n + r * S;
    float        acc[3] = {0.0f, 0.0f, 0.0f};
    for(int j = lane; j < S; j += 32) {
      const float w = plan_weight(__ldg(cr + j), bk, lambda);
      if(w == 0.0f) continue; // a zero weight contributes nothing, whatever the candidate holds
      const uint4 q = __ldg(cs + j);
      acc[0] = fadd(acc[0], fmul(w, u2f(q.x))), acc[1] = fadd(acc[1], fmul(w, u2f(q.y))), acc[2] = fadd(acc[2], fmul(w, u2f(q.z)));
    }
#pragma unroll
    for(int ax = 0; ax < 3; ax++) acc[ax] = warp_sum(acc[ax]);
    if(lane == 0)
      nom[(int64_t)s * R + r] = make_uint4(f2u(fdiv(acc[0], wsum)), f2u(fdiv(acc[1], wsum)), f2u(fdiv(acc[2], wsum)), (uint32_t)RK_CMD_MOVE);
  }
}

static bool overlap(const void *a, size_t na, const void *b, size_t nb) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return x < y + nb && y < x + na;
}

static int plan_check_rs(const char *who, int64_t R, int32_t S, int32_t n_seg) {
  if(R < 0 || S < 1 || n_seg < 1) {
    set_error("%s: need R >= 0, S >= 1 and n_seg >= 1 (R = %lld, S = %d, n_seg = %d)", who, (long long)R, S, n_seg);
    return RK_ERR_ARG;
  }
  if((uint64_t)n_seg * (uint64_t)S >= (1ull << 32)) {
    set_error("%s: n_seg * S must be < 2^32 (the hash index)", who);
    return RK_ERR_ARG;
  }
  return RK_OK;
}
static int plan_check_table(const char *who, const void *ptr, const char *name) {
  if(ptr == nullptr || ((uintptr_t)ptr & 15u) != 0) {
    set_error("%s: %s must be a non-NULL 16-byte aligned device pointer", who, name);
    return RK_ERR_ARG;
  }
  return RK_OK;
}

} // namespace rk

using namespace rk;

extern "C" {

int rk_plan_sample_commands(const rk_vdt_params_t *p, const rk_plan_sample_t *s, const rk_vdt_cmd_t *d_nominal, int64_t R, int32_t S,
                            int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream) {
  static const char *who = "rk_plan_sample_commands";
  if(!p || !s) {
    set_error("%s: NULL params/sample", who);
    return RK_ERR_ARG;
  }
  if(int rc = plan_check_rs(who, R, S, n_seg)) return rc;
  if(R == 0) return RK_OK;
  if(int rc = plan_check_table(who, d_nominal, "d_nominal")) return rc;
  if(int rc = plan_check_table(who, d_cmd, "d_cmd")) return rc;
  const int64_t n = R * (int64_t)S;
  if(overlap(d_nominal, (size_t)n_seg * R * 16u, d_cmd, (size_t)n_seg * n * 16u)) {
    set_error("%s: d_cmd must not overlap d_nominal", who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  PlanSampleArgs a;
  a.first = s->first, a.R = R, a.S = S, a.n_seg = n_seg, a.seed = s->seed;
  for(int k = 0; k < 3; k++) a.sigma[k] = s->sigma[k];
  a.limit_speed = p->limit_speed_mmps, a.limit_rot = p->limit_rot_radps;
  const dim3 grid((unsigned)((n + RK_PLAN_BLOCK - 1) / RK_PLAN_BLOCK), (unsigned)min(n_seg, 65535));
  plan_sample_kernel<<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>(a, (const uint4 *)d_nominal, (uint4 *)d_cmd);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_plan_select(const float *d_cost, const rk_vdt_cmd_t *d_cmd, int64_t R, int32_t S, int32_t n_seg, float lambda, int32_t shift,
                   rk_vdt_cmd_t *d_nominal_out, int32_t *d_best, float *d_best_cost, void *stream) {
  static const char *who = "rk_plan_select";
  if(int rc = plan_check_rs(who, R, S, n_seg)) return rc;
  if(shift < 0 || shift >= n_seg) {
    set_error("%s: need 0 <= shift < n_seg (shift = %d, n_seg = %d)", who, shift, n_seg);
    return RK_ERR_ARG;
  }
  if(!(lambda >= 0.0f) || isinf(lambda)) {
    set_error("%s: lambda must be finite and >= 0", who);
    return RK_ERR_ARG;
  }
  if(R == 0) return RK_OK;
  if(!d_cost || ((uintptr_t)d_cost & 3u)) {
    set_error("%s: d_cost must be a non-NULL float device pointer", who);
    return RK_ERR_ARG;
  }
  if(int rc = plan_check_table(who, d_cmd, "d_cmd")) return rc;
  if(int rc = plan_check_table(who, d_nominal_out, "d_nominal_out")) return rc;
  if(overlap(d_nominal_out, (size_t)n_seg * R * 16u, d_cmd, (size_t)n_seg * R * S * 16u)) {
    set_error("%s: d_nominal_out must not overlap d_cmd", who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  const unsigned warps_per_block = RK_PLAN_BLOCK / 32;
  const unsigned grid            = (unsigned)((R + warps_per_block - 1) / warps_per_block);
  plan_select_kernel<<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>(d_cost, (const uint4 *)d_cmd, R, S, n_seg, lambda, shift,
                                                                        (uint4 *)d_nominal_out, d_best, d_best_cost);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

} // extern "C"
