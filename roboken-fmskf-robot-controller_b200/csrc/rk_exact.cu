// rk_exact.cu -- exhaustive on-device proofs that gate the fast path (rk_vehicle_fast.cuh).
//
// Run once per parameter set (a few milliseconds on a B200) by rk_vdt_rollout() before the
// fast kernel is first used; results are cached.  If any proof fails for the given constants
// the library silently uses the transcription kernel -- results are identical either way.
//   1. div_const(x, c, RN(1/c)) == x / c bit for bit, for every finite float x (2^32 cases),
//      c = wheel radius; for c = SQRTF2 and WHEEL_L_MM the sequence must be exact for
//      x == 0 and |x| >= 2^-40 (their operand is a sum of wheel speeds derived from int16 rpm,
//      which is 0 or >= 2^-34 in magnitude).
//   2. fma(d, K_hi, d*K_lo) == (float)((double)d * OUT_RAD_PER_RAW_ANGLE * GEAR_RATIO_INV)
//      for every integer |d| <= 2^17 (the closed-loop plant needs |d| < 4096, recorded frames |d| <= 40960).
//   3. plant_dang(r) == r * 8192 / 60000 (C truncation) for every int16 r.
#include <mutex>
#include <string.h>

#include "rk_vehicle_fast2.cuh"

namespace rk {

struct ProofOut {
  unsigned int div_fail_any;     // failures anywhere (finite x)
  unsigned int div_fail_outside; // failures with x == +-0 or |x| >= 2^-40
  unsigned int mrad_fail, dang_fail;
  unsigned int div_fail_mid;     // failures with x == +-0 or 2^-40 <= |x| <= 2^64 (small divisors overflow / underflow beyond)
};

__global__ void proof_div_kernel(float c, ProofOut *out) {
  const float    rcp = fdiv(1.0f, c);
  unsigned int   any = 0, outside = 0, mid = 0;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for(uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; b < 0x100000000ull; b += stride) {
    const unsigned int u = (unsigned int)b, au = u & 0x7fffffffu;
    if(au >= 0x7f800000u) continue; // NaN / Inf are outside the fast path's domain
    const float x = u2f(u);
    if(f2u(div_const(x, c, rcp)) != f2u(fdiv(x, c))) {
      any++;
      if(au == 0u || au >= 0x2b800000u /* 2^-40 */) outside++;
      if(au == 0u || (au >= 0x2b800000u && au <= 0x5f800000u /* 2^64 */)) mid++;
    }
  }
  if(any) atomicAdd(&out->div_fail_any, any);
  if(outside) atomicAdd(&out->div_fail_outside, outside);
  if(mid) atomicAdd(&out->div_fail_mid, mid);
}

__global__ void proof_small_kernel(ProofOut *out) {
  const int  i = blockIdx.x * blockDim.x + threadIdx.x;
  const double K    = (double)RK_OUT_RAD_PER_RAW_ANGLE * (double)RK_GEAR_RATIO_INV;
  const float  k_hi = __double2float_rn(K);
  const float  k_lo = __double2float_rn(K - (double)k_hi);
  if(i <= 2 * 131072) { // |d| <= 2^17: every step rx_callback's int16 unwrap can produce, plant or recorded frames
    const int   d   = i - 131072;
    const float ref = __double2float_rn(__dmul_rn(__dmul_rn((double)d, (double)RK_OUT_RAD_PER_RAW_ANGLE), (double)RK_GEAR_RATIO_INV));
    const float df  = (float)d;
    if(f2u(ref) != f2u(__fmaf_rn(df, k_hi, fmul(df, k_lo)))) atomicAdd(&out->mrad_fail, 1u);
  }
  if(i < 65536) {
    const int r = i - 32768;
    if(plant_dang(r) != r * 8192 / 60000) atomicAdd(&out->dang_fail, 1u);
    // the same step formed in float by the packed tick (the float encoder step in fast_tick2, rk_vehicle_fast2.cuh): trunc(RN(r * C))
    if(truncf(fmul((float)r, kDangC)) != (float)(r * 8192 / 60000)) atomicAdd(&out->dang_fail, 1u);
  }
}

// Proof results are cached per (device, radius, sqrt2, L): alternating parameter sets or several GPUs in one process
// prove each combination once.  The proofs run on a private non-blocking stream (never the legacy default stream), so
// a first use inside rk_vdt_rollout synchronises with that stream only; rk_vdt_prepare() runs them ahead of time
// (required before a rollout is captured into a CUDA graph: the proof allocates and synchronises).
struct ProofEntry {
  int   device;
  float r, s2, l;
  bool  ok;
};
static ProofEntry g_proofs[32];
static int        g_n_proofs = 0;
static std::mutex g_proof_mu;

// true iff the fast path may be used with these divisors on the current device
bool fast_path_proven(const rk_vdt_params_t &p) {
  std::lock_guard<std::mutex> lk(g_proof_mu);
  int dev = -1;
  if(cudaGetDevice(&dev) != cudaSuccess) return false;
  for(int k = 0; k < g_n_proofs; k++) {
    const ProofEntry &e = g_proofs[k];
    if(e.device == dev && e.r == p.wheel_radius_mm && e.s2 == p.sqrtf2 && e.l == p.wheel_l_mm) return e.ok;
  }
  ProofEntry ne = {dev, p.wheel_radius_mm, p.sqrtf2, p.wheel_l_mm, false};
  auto       remember = [&](bool ok) {
    ne.ok = ok;
    if(g_n_proofs < 32) g_proofs[g_n_proofs++] = ne;
    else g_proofs[31] = ne; // a 33rd combination: the last slot is recycled
    return ok;
  };
  if(!(p.wheel_radius_mm > 0.0f) || !(p.sqrtf2 > 0.0f) || !(p.wheel_l_mm > 0.0f)) return remember(false);
  cudaStream_t st = nullptr;
  if(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  ProofOut *d_out = nullptr, h[4];
  if(cudaMalloc((void **)&d_out, 4 * sizeof(ProofOut)) != cudaSuccess) {
    cudaGetLastError();
    cudaStreamDestroy(st);
    return false;
  }
  for(int k = 0; k < 4; k++) h[k] = ProofOut{0u, 0u, 0u, 0u, 0u};
  cudaMemcpyAsync(d_out, h, sizeof(h), cudaMemcpyHostToDevice, st);
  const float cs[3] = {p.wheel_radius_mm, p.sqrtf2, p.wheel_l_mm};
  for(int k = 0; k < 3; k++) proof_div_kernel<<<148 * 16, 256, 0, st>>>(cs[k], d_out + k);
  proof_small_kernel<<<1025, 256, 0, st>>>(d_out + 3);
  cudaError_t e = cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, st);
  if(e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d_out);
  cudaStreamDestroy(st);
  if(e != cudaSuccess) {
    cudaGetLastError();
    return false; // not cached: a transient failure must not disable the fast path for good
  }
  bool ok = true;
  ok &= (h[0].div_fail_any == 0u);                                   // radius: every finite float
  for(int k = 1; k < 3; k++) ok &= (h[k].div_fail_outside == 0u);    // sqrt2, L: 0 and |x| >= 2^-40
  ok &= (h[3].mrad_fail == 0u) && (h[3].dang_fail == 0u);
  return remember(ok);
}

// Exhaustive check of div_const(x, c, RN(1/c)) == x / c (bit for bit) over every finite float x on
// the current device (one pass, ~4 ms, cached per (device, c)):  2 = exact for every x,
// 1 = exact for x == +-0 and |x| >= 2^-40 (the tiny-quotient range underflows), 0 = not usable.
// Used by kernels that divide by a launch constant every tick (e.g. the MG joint's velocity
// limit, AD_joint_mg_servo.cpp:140).
int div_const_exact(float c) {
  static std::mutex mu;
  static struct { int dev; uint32_t bits; int ok; } cache[16];
  static int n_cache = 0;
  if(!(c > 0.0f) || !(c < 3.0e38f)) return 0;
  int dev = -1;
  if(cudaGetDevice(&dev) != cudaSuccess) return 0;
  uint32_t bits;
  memcpy(&bits, &c, 4);
  std::lock_guard<std::mutex> lk(mu);
  for(int k = 0; k < n_cache; k++)
    if(cache[k].dev == dev && cache[k].bits == bits) return cache[k].ok;
  ProofOut *d_out = nullptr, h = ProofOut{0u, 0u, 0u, 0u, 0u};
  if(cudaMalloc((void **)&d_out, sizeof(ProofOut)) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  cudaStream_t st = nullptr;
  if(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    cudaFree(d_out);
    return 0;
  }
  cudaMemcpyAsync(d_out, &h, sizeof(h), cudaMemcpyHostToDevice, st);
  proof_div_kernel<<<148 * 16, 256, 0, st>>>(c, d_out);
  cudaError_t e = cudaMemcpyAsync(&h, d_out, sizeof(h), cudaMemcpyDeviceToHost, st);
  if(e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaStreamDestroy(st);
  cudaFree(d_out);
  if(e != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  const int ok = (h.div_fail_any == 0u) ? 2 : (h.div_fail_mid == 0u) ? 1 : 0; // 1: exact for 0 and 2^-40 <= |x| <= 2^64
  if(n_cache < 16) cache[n_cache].dev = dev, cache[n_cache].bits = bits, cache[n_cache].ok = ok, n_cache++;
  return ok;
}

} // namespace rk

extern "C" {
/* Test / diagnostics hook: runs (or returns the cached result of) the fast-path proofs for
 * the given parameters on the current device.  1 = proven, 0 = not proven (transcription
 * kernel is used), <0 = error. */
int rk_vdt_prepare(const rk_vdt_params_t *p) {
  if(!p) return RK_ERR_ARG;
  if(int rc = rk::require_device()) return rc;
  (void)rk::fast_path_proven(*p);
  return RK_OK;
}
int rk_vdt_fast_path_proven(const rk_vdt_params_t *p) {
  if(!p) return -RK_ERR_ARG;
  if(rk::require_device() != RK_OK) return -RK_ERR_CUDA;
  return rk::fast_path_proven(*p) ? 1 : 0;
}
}
