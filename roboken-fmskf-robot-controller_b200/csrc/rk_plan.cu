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

// one thread per (segment, candidate): blockIdx.y strides the segments, x runs over the R*S candidates of one segment.
// kSigmaTable: the noise scale of segment s, robot r is cell s*R + r of `sigma` (rk_plan_sample_commands_sigma) instead
// of a.sigma; the table comes last among the parameters so that the other instantiation's parameter offsets stay put.
template <bool kSigmaTable>
__global__ void __launch_bounds__(RK_PLAN_BLOCK)
plan_sample_kernel(const PlanSampleArgs a, const uint4 *__restrict__ nominal, uint4 *__restrict__ cmd, const float4 *__restrict__ sigma) {
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
      float          sg[3] = {a.sigma[0], a.sigma[1], a.sigma[2]};
      if constexpr(kSigmaTable) {
        const float4 t = __ldg(sigma + (int64_t)s * a.R + r); // like the nominal, one cell per robot and segment
        sg[0] = t.x, sg[1] = t.y, sg[2] = t.z;
      }
#pragma unroll
      for(int ax = 0; ax < 3; ax++) v[ax] = fadd(v[ax], fmul(sg[ax], plan_xi(h, (uint32_t)ax)));
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

// The robot's best candidate (key, j) over its S costs cr, the same in every lane; lane 0 writes best / best_cost where
// asked.  Returns j and leaves the key in bk.
RK_DEV int plan_argmin(const float *__restrict__ cr, int S, int64_t r, int lane, int32_t *__restrict__ best_out,
                       float *__restrict__ best_cost_out, float &bk) {
  bk     = __int_as_float(0x7F800000);
  int bj = INT_MAX;
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
  return best;
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

  float     bk;
  const int best = plan_argmin(cr, S, r, lane, best_out, best_cost_out, bk);

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

struct PlanRefitArgs {
  int64_t R;
  int32_t S, n_seg, k, shift;
  float   alpha, sigma_min[3];
};

// order-preserving u32 image of a finite cost; -0 is made +0 first, so that the two are one key as they are one float
RK_DEV uint32_t plan_order(float c) {
  const uint32_t u = f2u(c == 0.0f ? 0.0f : c);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// Elite bits of candidates j0 .. j0+31 (bit i: candidate j0 + i), the same in every lane: finite keys below the
// threshold key, and those at it while fewer than `take` came before (at_thr counts the ones before j0: ascending j).
RK_DEV uint32_t plan_elite_bits(const float *__restrict__ cr, int S, int j0, int lane, uint32_t thr, int take, int &at_thr) {
  const int      j     = j0 + lane;
  const float    c     = j < S ? __ldg(cr + j) : __int_as_float(0x7FC00000);
  const bool     fin   = isfinite(c);
  const uint32_t key   = plan_order(c);
  const uint32_t below = __ballot_sync(0xFFFFFFFFu, fin && key < thr);
  const uint32_t at    = __ballot_sync(0xFFFFFFFFu, fin && key == thr);
  const int      rank  = at_thr + __popc(at & ((1u << lane) - 1u));
  at_thr += __popc(at);
  return below | __ballot_sync(0xFFFFFFFFu, ((at >> lane) & 1u) && rank < take);
}

// one warp per robot, shaped like plan_select_kernel: the argmin; the key of the k_eff-th elite, fixed bit by bit from
// the top with warp-wide counts; then lanes own (segment, axis) pairs and walk the candidates 32 at a time in ascending
// j, the elites of each 32 as one ballot, reading the elite cells only.  sigma_in and sigma_out may be one table (shift == 0: each lane reads its own word first).
__global__ void __launch_bounds__(RK_PLAN_BLOCK)
plan_refit_kernel(const PlanRefitArgs a, const float *__restrict__ cost, const uint4 *__restrict__ cmd, const float4 *sigma_in,
                  uint4 *__restrict__ nom, float4 *sigma_out, int32_t *__restrict__ best_out, float *__restrict__ best_cost_out) {
  const int64_t r    = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int     lane = threadIdx.x & 31;
  if(r >= a.R) return; // whole warps leave together
  const int     S = a.S, n_seg = a.n_seg;
  const int64_t n  = a.R * (int64_t)S;
  const float  *cr = cost + r * S;

  float     bk;
  const int best = plan_argmin(cr, S, r, lane, best_out, best_cost_out, bk);
  int       fin  = 0;
  for(int j = lane; j < S; j += 32) fin += isfinite(__ldg(cr + j)) ? 1 : 0;
  const int k_eff = min(a.k, (int)__reduce_add_sync(0xFFFFFFFFu, (unsigned)fin));
  if(k_eff == 0) { // no finite cost: candidate `best` and the incoming sigma, bit for bit, one lane per segment
    for(int s = lane; s < n_seg; s += 32) {
      const int ss                    = min(s + a.shift, n_seg - 1);
      nom[(int64_t)s * a.R + r]       = __ldg(cmd + (int64_t)ss * n + r * S + best);
      sigma_out[(int64_t)s * a.R + r] = sigma_in[(int64_t)ss * a.R + r];
    }
    return;
  }

  uint32_t thr  = 0u;    // order key of the k_eff-th elite
  int      take = k_eff; // ends as that elite's rank among the candidates whose key is thr
  for(int b = 31; b >= 0; b--) {
    const uint32_t hi  = 0xFFFFFFFFu << b;
    int            cnt = 0; // finite keys equal to thr above bit b, with bit b clear
    for(int j = lane; j < S; j += 32) {
      const float c = __ldg(cr + j);
      cnt += (isfinite(c) && ((plan_order(c) ^ thr) & hi) == 0u) ? 1 : 0;
    }
    cnt = (int)__reduce_add_sync(0xFFFFFFFFu, (unsigned)cnt);
    if(take > cnt) take -= cnt, thr |= 1u << b;
  }

  const float kf = (float)k_eff, beta = fsub(1.0f, a.alpha);
  for(int p0 = 0; p0 < 3 * n_seg; p0 += 32) { // every lane takes part in the ballots; lanes past the end do not store
    const int    p = min(p0 + lane, 3 * n_seg - 1), s = p / 3, ax = p - 3 * s;
    const int    ss = min(s + a.shift, n_seg - 1);
    const float *cv = (const float *)(cmd + (int64_t)ss * n + r * S) + ax; // axis ax of candidate j is cv[4*j]
    float        sum = -0.0f; // -0 + v == v for every v: the sum starts from the first elite
    for(int j0 = 0, at = 0; j0 < S; j0 += 32)
      for(uint32_t m = plan_elite_bits(cr, S, j0, lane, thr, take, at); m != 0u; m &= m - 1u) // ascending j
        sum = fadd(sum, __ldg(cv + 4 * (int64_t)(j0 + __ffs(m) - 1)));
    const float m = fdiv(sum, kf);
    float       q = 0.0f;
    for(int j0 = 0, at = 0; j0 < S; j0 += 32)
      for(uint32_t e = plan_elite_bits(cr, S, j0, lane, thr, take, at); e != 0u; e &= e - 1u) {
        const float d = fsub(__ldg(cv + 4 * (int64_t)(j0 + __ffs(e) - 1)), m);
        q             = fadd(q, fmul(d, d));
      }
    const float sd   = fsqrt(fdiv(q, kf));
    float       mean = m, sig = sd;
    if(a.alpha > 0.0f) {
      const float sin = ((const float *)(sigma_in + (int64_t)ss * a.R + r))[ax];
      mean            = fadd(fmul(a.alpha, __ldg(cv)), fmul(beta, m));
      sig             = fadd(fmul(a.alpha, sin), fmul(beta, sd));
    }
    if(p0 + lane >= 3 * n_seg) continue;
    const float lo = ax == 0 ? a.sigma_min[0] : (ax == 1 ? a.sigma_min[1] : a.sigma_min[2]);
    float      *no = (float *)(nom + (int64_t)s * a.R + r);
    float      *so = (float *)(sigma_out + (int64_t)s * a.R + r);
    no[ax] = mean, so[ax] = fmaxf(sig, lo);
    if(ax == 0) ((uint32_t *)no)[3] = (uint32_t)RK_CMD_MOVE, so[3] = 0.0f;
  }
}

// rk_plan_peer_discs: one thread per (checkpoint, robot), x over the robots (coalesced stores), y striding the
// checkpoints.  The peer index is checked before the path is read, so nothing out of range is read.
__global__ void __launch_bounds__(RK_PLAN_BLOCK)
plan_peer_discs_kernel(const float2 *__restrict__ path, int64_t R, int n_ck, const int32_t *__restrict__ peer, int m, float radius,
                       float4 *__restrict__ obs, int M, int k0) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(r >= R) return;
  for(int c = blockIdx.y; c < n_ck; c += gridDim.y) {
    const float2 *pc = path + (int64_t)c * R;
    float4       *oc = obs + ((int64_t)c * M + k0) * R + r;
    for(int k = 0; k < m; k++) {
      const int32_t q = __ldg(peer + (int64_t)k * R + r);
      float4        d = make_float4(0.0f, 0.0f, __int_as_float(0x7FC00000), 0.0f); // contributes nothing
      if(q >= 0 && q < R && q != r) {
        const float2 x = __ldg(pc + q);
        d              = make_float4(x.x, x.y, radius, 0.0f);
      }
      oc[(int64_t)k * R] = d;
    }
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

// rk_plan_sample_commands, and with `table` rk_plan_sample_commands_sigma (d_sigma: float4 [n_seg][R])
static int plan_sample(const char *who, const rk_vdt_params_t *p, const rk_plan_sample_t *s, const rk_vdt_cmd_t *d_nominal, bool table,
                       const float *d_sigma, int64_t R, int32_t S, int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream) {
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
  if(table) {
    if(int rc = plan_check_table(who, d_sigma, "d_sigma")) return rc;
    if(overlap(d_sigma, (size_t)n_seg * R * 16u, d_cmd, (size_t)n_seg * n * 16u)) {
      set_error("%s: d_cmd must not overlap d_sigma", who);
      return RK_ERR_ARG;
    }
  }
  if(int rc = require_device()) return rc;
  PlanSampleArgs a;
  a.first = s->first, a.R = R, a.S = S, a.n_seg = n_seg, a.seed = s->seed;
  for(int k = 0; k < 3; k++) a.sigma[k] = s->sigma[k];
  a.limit_speed = p->limit_speed_mmps, a.limit_rot = p->limit_rot_radps;
  const dim3 grid((unsigned)((n + RK_PLAN_BLOCK - 1) / RK_PLAN_BLOCK), (unsigned)min(n_seg, 65535));
  if(table)
    plan_sample_kernel<true><<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>(a, (const uint4 *)d_nominal, (uint4 *)d_cmd, (const float4 *)d_sigma);
  else
    plan_sample_kernel<false><<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>(a, (const uint4 *)d_nominal, (uint4 *)d_cmd, nullptr);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

// the arguments rk_plan_select and rk_plan_refit share: sizes and shift first, then (R > 0) the tables
static int plan_check_choice(const char *who, int64_t R, int32_t S, int32_t n_seg, int32_t shift) {
  if(int rc = plan_check_rs(who, R, S, n_seg)) return rc;
  if(shift < 0 || shift >= n_seg) {
    set_error("%s: need 0 <= shift < n_seg (shift = %d, n_seg = %d)", who, shift, n_seg);
    return RK_ERR_ARG;
  }
  return RK_OK;
}
static int plan_check_choice_tables(const char *who, const float *d_cost, const rk_vdt_cmd_t *d_cmd, int64_t R, int32_t S, int32_t n_seg,
                                    const rk_vdt_cmd_t *d_nominal_out) {
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
  return RK_OK;
}

} // namespace rk

using namespace rk;

extern "C" {

int rk_plan_sample_commands(const rk_vdt_params_t *p, const rk_plan_sample_t *s, const rk_vdt_cmd_t *d_nominal, int64_t R, int32_t S,
                            int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream) {
  return plan_sample("rk_plan_sample_commands", p, s, d_nominal, false, nullptr, R, S, n_seg, d_cmd, stream);
}

int rk_plan_sample_commands_sigma(const rk_vdt_params_t *p, const rk_plan_sample_t *s, const rk_vdt_cmd_t *d_nominal, const float *d_sigma,
                                  int64_t R, int32_t S, int32_t n_seg, rk_vdt_cmd_t *d_cmd, void *stream) {
  return plan_sample("rk_plan_sample_commands_sigma", p, s, d_nominal, true, d_sigma, R, S, n_seg, d_cmd, stream);
}

int rk_plan_select(const float *d_cost, const rk_vdt_cmd_t *d_cmd, int64_t R, int32_t S, int32_t n_seg, float lambda, int32_t shift,
                   rk_vdt_cmd_t *d_nominal_out, int32_t *d_best, float *d_best_cost, void *stream) {
  static const char *who = "rk_plan_select";
  if(int rc = plan_check_choice(who, R, S, n_seg, shift)) return rc;
  if(!(lambda >= 0.0f) || isinf(lambda)) {
    set_error("%s: lambda must be finite and >= 0", who);
    return RK_ERR_ARG;
  }
  if(R == 0) return RK_OK;
  if(int rc = plan_check_choice_tables(who, d_cost, d_cmd, R, S, n_seg, d_nominal_out)) return rc;
  if(int rc = require_device()) return rc;
  const unsigned warps_per_block = RK_PLAN_BLOCK / 32;
  const unsigned grid            = (unsigned)((R + warps_per_block - 1) / warps_per_block);
  plan_select_kernel<<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>(d_cost, (const uint4 *)d_cmd, R, S, n_seg, lambda, shift,
                                                                        (uint4 *)d_nominal_out, d_best, d_best_cost);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_plan_refit(const float *d_cost, const rk_vdt_cmd_t *d_cmd, const float *d_sigma_in, int64_t R, int32_t S, int32_t n_seg,
                  const rk_plan_refit_t *rf, int32_t shift, rk_vdt_cmd_t *d_nominal_out, float *d_sigma_out, int32_t *d_best,
                  float *d_best_cost, void *stream) {
  static const char *who = "rk_plan_refit";
  if(int rc = plan_check_choice(who, R, S, n_seg, shift)) return rc;
  if(!rf) {
    set_error("%s: NULL refit", who);
    return RK_ERR_ARG;
  }
  if(rf->elite < 1 || rf->elite > S) {
    set_error("%s: need 1 <= elite <= S (elite = %d, S = %d)", who, rf->elite, S);
    return RK_ERR_ARG;
  }
  if(!(rf->alpha >= 0.0f && rf->alpha <= 1.0f)) {
    set_error("%s: alpha must be in [0, 1]", who);
    return RK_ERR_ARG;
  }
  for(int k = 0; k < 3; k++)
    if(!(rf->sigma_min[k] >= 0.0f) || isinf(rf->sigma_min[k])) {
      set_error("%s: sigma_min[%d] must be finite and >= 0", who, k);
      return RK_ERR_ARG;
    }
  if(R == 0) return RK_OK;
  if(int rc = plan_check_choice_tables(who, d_cost, d_cmd, R, S, n_seg, d_nominal_out)) return rc;
  if(int rc = plan_check_table(who, d_sigma_in, "d_sigma_in")) return rc;
  if(int rc = plan_check_table(who, d_sigma_out, "d_sigma_out")) return rc;
  const size_t nsig = (size_t)n_seg * R * 16u;
  if(overlap(d_sigma_out, nsig, d_sigma_in, nsig) && !(shift == 0 && d_sigma_out == d_sigma_in)) {
    set_error("%s: d_sigma_out must not overlap d_sigma_in, unless shift == 0 and they are the same table", who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  PlanRefitArgs a;
  a.R = R, a.S = S, a.n_seg = n_seg, a.k = rf->elite, a.shift = shift, a.alpha = rf->alpha;
  for(int k = 0; k < 3; k++) a.sigma_min[k] = rf->sigma_min[k];
  const unsigned warps_per_block = RK_PLAN_BLOCK / 32;
  const unsigned grid            = (unsigned)((R + warps_per_block - 1) / warps_per_block);
  plan_refit_kernel<<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>(a, d_cost, (const uint4 *)d_cmd, (const float4 *)d_sigma_in,
                                                                       (uint4 *)d_nominal_out, (float4 *)d_sigma_out, d_best, d_best_cost);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

int rk_plan_peer_discs(const float *d_path, int64_t R, int32_t n_ck, const int32_t *d_peer, int32_t m, float radius, float *d_obs, int32_t M,
                       int32_t k0, void *stream) {
  static const char *who = "rk_plan_peer_discs";
  if(R < 0 || n_ck < 0 || m < 0) {
    set_error("%s: need R, n_ck and m >= 0 (R = %lld, n_ck = %d, m = %d)", who, (long long)R, n_ck, m);
    return RK_ERR_ARG;
  }
  if(k0 < 0 || (int64_t)k0 + m > M) {
    set_error("%s: need 0 <= k0 and k0 + m <= M (k0 = %d, m = %d, M = %d)", who, k0, m, M);
    return RK_ERR_ARG;
  }
  if(!(radius >= 0.0f) || isinf(radius)) {
    set_error("%s: radius must be finite and >= 0", who);
    return RK_ERR_ARG;
  }
  if(R == 0 || n_ck == 0 || m == 0) return RK_OK;
  if(!d_path || ((uintptr_t)d_path & 7u) || !d_peer || ((uintptr_t)d_peer & 3u)) {
    set_error("%s: d_path (8-byte aligned float2) and d_peer (int32) must be non-NULL device pointers", who);
    return RK_ERR_ARG;
  }
  if(int rc = plan_check_table(who, d_obs, "d_obs")) return rc;
  if(overlap(d_obs, (size_t)n_ck * M * R * 16u, d_path, (size_t)n_ck * R * 8u)) {
    set_error("%s: d_obs must not overlap d_path", who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  const dim3 grid((unsigned)((R + RK_PLAN_BLOCK - 1) / RK_PLAN_BLOCK), (unsigned)min(n_ck, 65535));
  plan_peer_discs_kernel<<<grid, RK_PLAN_BLOCK, 0, (cudaStream_t)stream>>>((const float2 *)d_path, R, n_ck, d_peer, m, radius,
                                                                            (float4 *)d_obs, M, k0);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

} // extern "C"
