// rk_plan.cu -- the two ends of a planning step around rk_plan_rollout (rk_vehicle.cu): candidate commands sampled
// around a nominal plan, and the per-robot choice among the candidates' costs (include/robotick.h, "Vehicle sampling
// planner"); and the planner kernels outside the rollout: peer discs, cost-to-go fields and map inflation.  Candidate j of robot r is
// instance r*S + j, so a robot's S candidates are contiguous in every table.
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

// rk_plan_cost_to_go: one CTA per 32 x 32 tile of a field window, tiles numbered field-major then row-major.  Each
// thread owns column tx of rows ty, ty + 8, ty + 16, ty + 24 of its tile.
constexpr int kCtgTile = 32, kCtgHalo = kCtgTile + 2, kCtgThreads = 256, kCtgRows = kCtgThreads / kCtgTile;
constexpr int kCtgMaxBatch = 64; // rounds per batch at most (the batch doubles from 4)

struct CtgArgs {
  const float   *cells; // the map, [n_maps][height][width]
  int32_t        n_maps, width, height;
  float          x0, y0, inv_res, outside;
  float          step_a, step_d, k_cost, lethal;
  const float2  *goal;      // [n_fields]
  const int32_t *field_map; // [n_fields]; NULL: map 0
  const int2    *offset;    // [n_fields]; NULL: (0, 0)
  int32_t        fw, fh, tiles_x, tiles_y;
  float         *field; // [n_fields][fh][fw]
};

struct CtgTile {
  int  f, x0, y0; // the field, and the window cell of the tile's cell (0, 0)
  int  k;         // the field's map
  int2 o;         // the field's offset
};
RK_DEV CtgTile ctg_tile(const CtgArgs &a, int t) {
  const int per = a.tiles_x * a.tiles_y, f = t / per, q = t - f * per, ty = q / a.tiles_x;
  CtgTile c;
  c.f = f, c.x0 = (q - ty * a.tiles_x) * kCtgTile, c.y0 = ty * kCtgTile;
  c.k = a.field_map != nullptr ? __ldg(a.field_map + f) : 0;
  c.o = a.offset != nullptr ? __ldg(a.offset + f) : make_int2(0, 0);
  return c;
}
// The cost c of window cell (ix, iy) (in the window, of a field whose map index is in range and |offset| <= 2^24)
RK_DEV float ctg_cost(const CtgArgs &a, const CtgTile &c, int ix, int iy) {
  const int mx = c.o.x + ix, my = c.o.y + iy;
  return (mx >= 0 && mx < a.width && my >= 0 && my < a.height) ? __ldg(a.cells + (c.k * a.height + my) * a.width + mx) : a.outside;
}

// D = +inf over the tile's cells, 0 at the goal cell; dirty[t] = the goal lies in tile t
__global__ void __launch_bounds__(kCtgThreads) plan_ctg_init_kernel(const CtgArgs a, uint32_t *__restrict__ dirty) {
  const CtgTile c = ctg_tile(a, blockIdx.x);
  int           gx = -1, gy = -1;
  if((uint32_t)c.k < (uint32_t)a.n_maps) {
    const float2 g = __ldg(a.goal + c.f);
    plan_window_cell(fmul(fsub(g.x, a.x0), a.inv_res), fmul(fsub(g.y, a.y0), a.inv_res), c.o, a.fw, a.fh, gx, gy);
  }
  float *D = a.field + (int64_t)c.f * a.fh * a.fw;
  for(int q = threadIdx.x; q < kCtgTile * kCtgTile; q += kCtgThreads) {
    const int ix = c.x0 + (q & (kCtgTile - 1)), iy = c.y0 + q / kCtgTile;
    if(ix < a.fw && iy < a.fh) D[iy * a.fw + ix] = (ix == gx && iy == gy) ? 0.0f : __int_as_float(0x7F800000);
  }
  if(threadIdx.x == 0) dirty[blockIdx.x] = (gx >= c.x0 && gx < c.x0 + kCtgTile && gy >= c.y0 && gy < c.y0 + kCtgTile) ? 1u : 0u;
}

// One round: a tile runs if it or one of its 8 neighbours changed in the previous round (dirty_in).  It loads D with a
// 1-cell halo into shared memory, relaxes its cells in place until a sweep changes nothing, writes back the cells that
// decreased, and reports in dirty_out (every tile writes its flag, so the buffer needs no clearing) and *count.
// Other tiles may write the halo's cells during the round: a read sees the old or the new value, both upper bounds that
// some path attains, and a tile that changed runs its neighbours again in the next round.
__global__ void __launch_bounds__(kCtgThreads)
plan_ctg_relax_kernel(const CtgArgs a, const uint32_t *__restrict__ dirty_in, uint32_t *__restrict__ dirty_out, int32_t *__restrict__ count) {
  __shared__ float   sD[kCtgHalo][kCtgHalo];
  __shared__ uint8_t sOk[kCtgHalo][kCtgHalo]; // in the window and not blocked
  const int          t  = blockIdx.x;
  const int          per = a.tiles_x * a.tiles_y, tq = t % per, tyi = tq / a.tiles_x, txi = tq - tyi * a.tiles_x;
  bool               go = false;
  if(threadIdx.x < 9) {
    const int ny = tyi + (int)threadIdx.x / 3 - 1, nx = txi + (int)threadIdx.x % 3 - 1;
    go = ny >= 0 && ny < a.tiles_y && nx >= 0 && nx < a.tiles_x && dirty_in[t - tq + ny * a.tiles_x + nx] != 0u;
  }
  if(!__syncthreads_or(go)) {
    if(threadIdx.x == 0) dirty_out[t] = 0u;
    return;
  }
  const CtgTile c = ctg_tile(a, t);
  float        *D = a.field + (int64_t)c.f * a.fh * a.fw;
  for(int q = threadIdx.x; q < kCtgHalo * kCtgHalo; q += kCtgThreads) {
    const int hy = q / kCtgHalo, hx = q - hy * kCtgHalo, ix = c.x0 + hx - 1, iy = c.y0 + hy - 1;
    float     d  = __int_as_float(0x7F800000);
    bool      ok = false;
    if(ix >= 0 && ix < a.fw && iy >= 0 && iy < a.fh) d = D[iy * a.fw + ix], ok = !(ctg_cost(a, c, ix, iy) >= a.lethal);
    sD[hy][hx] = d, sOk[hy][hx] = ok;
  }
  __syncthreads();
  const int tx = threadIdx.x & (kCtgTile - 1), ty = threadIdx.x / kCtgTile, x = tx + 1;
  float     wa[4], wd[4], d0[4];
  uint32_t  diag = 0u; // bits 4j .. 4j+3: the diagonal edges into row j's cell that may be taken (-,-), (+,-), (-,+), (+,+)
  bool      mine[4];
#pragma unroll
  for(int j = 0; j < 4; j++) {
    const int y = ty + kCtgRows * j + 1;
    mine[j]     = sOk[y][x] != 0;
    d0[j]       = sD[y][x];
    wa[j] = wd[j] = 0.0f;
    if(mine[j]) {
      const float cq = ctg_cost(a, c, c.x0 + tx, c.y0 + y - 1);
      const float tq = cq > 0.0f ? fadd(1.0f, fmul(a.k_cost, cq)) : 1.0f;
      wa[j] = fmul(a.step_a, tq), wd[j] = fmul(a.step_d, tq);
      const bool l = sOk[y][x - 1], r = sOk[y][x + 1], dn = sOk[y - 1][x], up = sOk[y + 1][x];
      diag |= ((l && dn ? 1u : 0u) | (r && dn ? 2u : 0u) | (l && up ? 4u : 0u) | (r && up ? 8u : 0u)) << (4 * j);
    }
  }
  const float inf = __int_as_float(0x7F800000);
  volatile float(*s)[kCtgHalo] = sD;
  for(;;) {
    bool ch = false;
#pragma unroll
    for(int j = 0; j < 4; j++) {
      if(!mine[j]) continue;
      const int      y = ty + kCtgRows * j + 1;
      const uint32_t b = diag >> (4 * j);
      // fl(a + w) is monotone in a: the least of the candidates D(p) + w is the least D(p) plus w
      const float ma = fminf(fminf(s[y][x - 1], s[y][x + 1]), fminf(s[y - 1][x], s[y + 1][x]));
      const float md = fminf(fminf((b & 1u) ? s[y - 1][x - 1] : inf, (b & 2u) ? s[y - 1][x + 1] : inf),
                             fminf((b & 4u) ? s[y + 1][x - 1] : inf, (b & 8u) ? s[y + 1][x + 1] : inf));
      const float nd = fminf(fadd(ma, wa[j]), fadd(md, wd[j]));
      if(nd < s[y][x]) s[y][x] = nd, ch = true;
    }
    if(!__syncthreads_or(ch)) break;
  }
  bool changed = false;
#pragma unroll
  for(int j = 0; j < 4; j++) {
    const int   y = ty + kCtgRows * j + 1;
    const float d = sD[y][x];
    if(mine[j] && d < d0[j]) D[(c.y0 + y - 1) * a.fw + c.x0 + tx] = d, changed = true;
  }
  changed = __syncthreads_or(changed);
  if(threadIdx.x == 0) {
    dirty_out[t] = changed ? 1u : 0u;
    if(changed) atomicAdd(count, 1);
  }
}

// rk_plan_inflate: an exact squared Euclidean distance transform truncated at rmax = floor(sqrt(n_table - 1)) cells, which
// keeps every d2 < n_table exact, in two passes.  The column pass writes g = min(vertical distance to the nearest
// obstacle of the column, rmax + 1) to the work space; the row pass takes min over |dx| <= rmax of dx^2 + g(x + dx)^2 and
// applies the table.  A capped g gives d2 >= (rmax + 1)^2 >= n_table, which the table treats as no obstacle.
constexpr int kInflThreads = 128, kInflChunk = 64, kInflMaxR = 255; // kInflChunk: the bits of one mask word

struct InflateArgs {
  const float *cells; // [n_maps][height][width]
  const float *table; // [n_table]
  float       *dst;   // [n_maps][height][width]
  int32_t      n_maps, width, height, rmax, n_table;
  float        lethal;
  bool         edge; // the cells off the grid are obstacles
};

// One thread per (map, chunk of 64 rows, column), x fastest.  Bit i of the mask is row y0 + i; the rows above and below
// the chunk are searched only as far as rmax from its ends, and the off-grid rows -1 and H count when edge is set.
__global__ void __launch_bounds__(kInflThreads) plan_inflate_cols_kernel(const InflateArgs a, int chunks, uint16_t *__restrict__ g) {
  const int64_t t = (int64_t)blockIdx.x * kInflThreads + threadIdx.x;
  const int     W = a.width, H = a.height, R = a.rmax, lim = R + 1;
  if(t >= (int64_t)a.n_maps * chunks * W) return;
  const int64_t q = t / W;
  const int     x = (int)(t - q * W), ch = (int)(q % chunks), k = (int)(q / chunks);
  const int     y0 = ch * kInflChunk, n = min(kInflChunk, H - y0);
  const float  *col = a.cells + (int64_t)k * H * W + x;
  uint64_t      m = 0;
#pragma unroll 8
  for(int i = 0; i < n; i++) m |= (__ldg(col + (int64_t)(y0 + i) * W) >= a.lethal ? 1ull : 0ull) << i;
  int above = y0 - lim; // the nearest obstacle row before the chunk, or a row far enough to cap
  for(int y = y0 - 1; y >= y0 - R; y--) {
    if(y < 0) {
      if(a.edge) above = -1;
      break;
    }
    if(__ldg(col + (int64_t)y * W) >= a.lethal) {
      above = y;
      break;
    }
  }
  const int y1 = y0 + n;
  int       below = y1 - 1 + lim; // the nearest obstacle row after the chunk, or a row far enough to cap
  for(int y = y1; y <= y1 - 1 + R; y++) {
    if(y >= H) {
      if(a.edge) below = H;
      break;
    }
    if(__ldg(col + (int64_t)y * W) >= a.lethal) {
      below = y;
      break;
    }
  }
  uint16_t *gc = g + (int64_t)k * H * W + x;
  for(int i = 0; i < n; i++) {
    const int      y = y0 + i;
    const uint64_t lo = m & (~0ull >> (63 - i)), hi = m >> i;
    const int      up = lo ? __clzll((long long)lo) - (63 - i) : y - above;
    const int      dn = hi ? __ffsll((long long)hi) - 1 : below - y;
    gc[(int64_t)y * W] = (uint16_t)min(min(up, dn), lim);
  }
}

// One CTA per (map, row, segment of 128 columns): g^2 of the segment and rmax columns on each side in shared memory
// ((rmax + 1)^2 off the grid: the off-grid columns are the axial terms below).  Each thread walks dx outward and stops
// once dx^2 alone reaches its best.
__global__ void __launch_bounds__(kInflThreads) plan_inflate_rows_kernel(const InflateArgs a, int segs, const uint16_t *__restrict__ g) {
  __shared__ int sg[kInflThreads + 2 * kInflMaxR];
  const int64_t  row = blockIdx.x / segs; // k*H + y
  const int      W = a.width, R = a.rmax, x0 = (int)(blockIdx.x - row * segs) * kInflThreads, lim2 = (R + 1) * (R + 1);
  const uint16_t *gr = g + row * W;
  for(int i = threadIdx.x; i < kInflThreads + 2 * R; i += kInflThreads) {
    const int x = x0 - R + i;
    int       v = lim2;
    if(x >= 0 && x < W) {
      const int d = gr[x];
      v           = d * d;
    }
    sg[i] = v;
  }
  __syncthreads();
  const int x = x0 + (int)threadIdx.x;
  if(x >= W) return;
  const int *s    = sg + R + threadIdx.x; // s[dx]: g^2 at column x + dx
  int        best = s[0];
  for(int dx = 1; dx <= R && dx * dx < best; dx++) best = min(best, dx * dx + min(s[-dx], s[dx]));
  if(a.edge) {
    if(x + 1 <= R) best = min(best, (x + 1) * (x + 1));
    if(W - x <= R) best = min(best, (W - x) * (W - x));
  }
  const int64_t i = row * W + x;
  const float   c = __ldg(a.cells + i);
  float         o = c;
  if(best < a.n_table) {
    const float v = __ldg(a.table + best);
    o             = (v > c || isnan(c)) ? v : c;
  }
  a.dst[i] = o;
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

// Tiles of a cost-to-go build; 0 for sizes rk_plan_cost_to_go rejects
static int64_t ctg_tiles(int32_t n_fields, int32_t fw, int32_t fh) {
  if(n_fields < 1 || fw < 1 || fh < 1 || fw > (1 << 24) || fh > (1 << 24) || (int64_t)n_fields * fh * fw > INT_MAX) return 0;
  return (int64_t)n_fields * ((fw + kCtgTile - 1) / kCtgTile) * ((fh + kCtgTile - 1) / kCtgTile);
}

// Cells of an inflation (the map-grid size rule); 0 for sizes rk_plan_inflate rejects
static int64_t infl_cells(int32_t n_maps, int32_t width, int32_t height) {
  if(n_maps < 1 || width < 1 || height < 1 || width > (1 << 24) || height > (1 << 24) || (int64_t)n_maps * height * width > INT_MAX) return 0;
  return (int64_t)n_maps * height * width;
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

size_t rk_plan_cost_to_go_work_bytes(int32_t n_fields, int32_t fw, int32_t fh) {
  const int64_t T = ctg_tiles(n_fields, fw, fh);
  return T == 0 ? 0 : (size_t)(kCtgMaxBatch + 2 * T) * sizeof(uint32_t);
}

int rk_plan_cost_to_go(const rk_plan_map_t *map, const rk_plan_ctg_t *spec, const float *d_goal, const int32_t *d_field_map,
                       const int32_t *d_offset, int32_t n_fields, int32_t fw, int32_t fh, float *d_field, void *d_work, int32_t *rounds_out,
                       void *stream) {
  static const char *who = "rk_plan_cost_to_go";
  if(!map || !spec) {
    set_error("%s: NULL map/spec", who);
    return RK_ERR_ARG;
  }
  if(int rc = plan_check_map_grid(who, map)) return rc;
  if(int rc = plan_check_map_tables(who, map)) return rc;
  if(!isfinite(spec->step_axial) || !(spec->step_axial > 0.0f) || !isfinite(spec->step_diag) || !(spec->step_diag > 0.0f)) {
    set_error("%s: step_axial and step_diag must be finite and > 0", who);
    return RK_ERR_ARG;
  }
  if(!(spec->k_cost >= 0.0f) || isinf(spec->k_cost)) {
    set_error("%s: k_cost must be finite and >= 0", who);
    return RK_ERR_ARG;
  }
  if(!(spec->lethal > 0.0f)) {
    set_error("%s: lethal must be > 0 (+inf allowed, NaN not)", who);
    return RK_ERR_ARG;
  }
  const int64_t T = ctg_tiles(n_fields, fw, fh);
  if(T == 0) {
    set_error("%s: need n_fields, fw, fh >= 1, fw, fh <= 2^24 and n_fields * fh * fw < 2^31 (n_fields = %d, fw = %d, fh = %d)", who,
              n_fields, fw, fh);
    return RK_ERR_ARG;
  }
  if(!d_goal || ((uintptr_t)d_goal & 7u) || ((uintptr_t)d_field_map & 3u) || ((uintptr_t)d_offset & 7u) || !d_field ||
     ((uintptr_t)d_field & 3u) || !d_work || ((uintptr_t)d_work & 3u)) {
    set_error("%s: d_goal (float2) and d_offset (int2, may be NULL) must be 8-byte aligned, d_field_map (int32, may be NULL), "
              "d_field (float) and d_work 4-byte aligned, and d_goal, d_field and d_work non-NULL",
              who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  CtgArgs a;
  a.cells = map->d_cells, a.n_maps = map->n_maps, a.width = map->width, a.height = map->height;
  a.x0 = map->x0, a.y0 = map->y0, a.inv_res = map->inv_res, a.outside = map->outside;
  a.step_a = spec->step_axial, a.step_d = spec->step_diag, a.k_cost = spec->k_cost, a.lethal = spec->lethal;
  a.goal = (const float2 *)d_goal, a.field_map = d_field_map, a.offset = (const int2 *)d_offset;
  a.fw = fw, a.fh = fh, a.tiles_x = (fw + kCtgTile - 1) / kCtgTile, a.tiles_y = (fh + kCtgTile - 1) / kCtgTile;
  a.field = d_field;
  int32_t     *count = (int32_t *)d_work;
  uint32_t    *dirty[2] = {(uint32_t *)d_work + kCtgMaxBatch, (uint32_t *)d_work + kCtgMaxBatch + T};
  cudaStream_t st = (cudaStream_t)stream;
  plan_ctg_init_kernel<<<(unsigned)T, kCtgThreads, 0, st>>>(a, dirty[0]);
  RK_CUDA(cudaGetLastError());
  int32_t rounds = 0, host[kCtgMaxBatch];
  for(int batch = 4, cur = 0;; batch = min(2 * batch, kCtgMaxBatch)) {
    RK_CUDA(cudaMemsetAsync(count, 0, batch * sizeof(int32_t), st));
    for(int b = 0; b < batch; b++, cur ^= 1) plan_ctg_relax_kernel<<<(unsigned)T, kCtgThreads, 0, st>>>(a, dirty[cur], dirty[cur ^ 1], count + b);
    RK_CUDA(cudaGetLastError());
    RK_CUDA(cudaMemcpyAsync(host, count, batch * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RK_CUDA(cudaStreamSynchronize(st));
    int b = 0;
    while(b < batch && host[b] != 0) b++;
    rounds += b;
    if(b < batch) break; // a round changed nothing: every later one is empty
  }
  if(rounds_out) *rounds_out = rounds;
  return RK_OK;
}

size_t rk_plan_inflate_work_bytes(int32_t n_maps, int32_t width, int32_t height) {
  const int64_t n = infl_cells(n_maps, width, height);
  return n == 0 ? 0 : ((size_t)n * sizeof(uint16_t) + 3u) & ~(size_t)3u;
}

int rk_plan_inflate(const rk_plan_map_t *map, const rk_plan_inflate_t *spec, float *d_dst, void *d_work, void *stream) {
  static const char *who = "rk_plan_inflate";
  if(!map || !spec) {
    set_error("%s: NULL map/spec", who);
    return RK_ERR_ARG;
  }
  if(int rc = plan_check_map_grid(who, map)) return rc;
  if(int rc = plan_check_map_tables(who, map)) return rc;
  if(spec->n_table < 1 || spec->n_table > 65536) {
    set_error("%s: need 1 <= n_table <= 65536 (n_table = %d)", who, spec->n_table);
    return RK_ERR_ARG;
  }
  if(!(spec->lethal > 0.0f)) {
    set_error("%s: lethal must be > 0 (+inf allowed, NaN not)", who);
    return RK_ERR_ARG;
  }
  if(!spec->d_table || ((uintptr_t)spec->d_table & 3u) || !d_dst || ((uintptr_t)d_dst & 3u) || !d_work || ((uintptr_t)d_work & 3u)) {
    set_error("%s: d_table, d_dst and d_work must be non-NULL 4-byte aligned device pointers", who);
    return RK_ERR_ARG;
  }
  const int64_t n       = infl_cells(map->n_maps, map->width, map->height);
  const size_t  n_cells = (size_t)n * 4u, n_work = rk_plan_inflate_work_bytes(map->n_maps, map->width, map->height);
  const size_t  n_tab   = (size_t)spec->n_table * 4u;
  if(overlap(d_dst, n_cells, map->d_cells, n_cells) || overlap(d_dst, n_cells, d_work, n_work) || overlap(d_dst, n_cells, spec->d_table, n_tab) ||
     overlap(d_work, n_work, map->d_cells, n_cells) || overlap(d_work, n_work, spec->d_table, n_tab)) {
    set_error("%s: d_dst and d_work must not overlap each other, the cells or the table", who);
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  int r = (int)sqrt((double)(spec->n_table - 1)); // rmax = floor(sqrt(n_table - 1)), made exact in integers
  while(r * r > spec->n_table - 1) r--;
  while((r + 1) * (r + 1) <= spec->n_table - 1) r++;
  InflateArgs a;
  a.cells = map->d_cells, a.table = spec->d_table, a.dst = d_dst;
  a.n_maps = map->n_maps, a.width = map->width, a.height = map->height, a.rmax = r, a.n_table = spec->n_table;
  a.lethal = spec->lethal, a.edge = map->outside >= spec->lethal;
  const int          chunks = (map->height + kInflChunk - 1) / kInflChunk, segs = (map->width + kInflThreads - 1) / kInflThreads;
  const int64_t      col_threads = (int64_t)map->n_maps * chunks * map->width;
  const cudaStream_t st = (cudaStream_t)stream;
  uint16_t          *g = (uint16_t *)d_work;
  plan_inflate_cols_kernel<<<(unsigned)((col_threads + kInflThreads - 1) / kInflThreads), kInflThreads, 0, st>>>(a, chunks, g);
  plan_inflate_rows_kernel<<<(unsigned)((int64_t)map->n_maps * map->height * segs), kInflThreads, 0, st>>>(a, segs, g);
  RK_CUDA(cudaGetLastError());
  return RK_OK;
}

} // extern "C"
