// rk_common.cuh -- shared device/host helpers for librobotick_b200.so (sm_100a only).
//
// Bit-exactness discipline (SURVEY.md section 0, finding 5): the firmware's float results
// feed integer outputs ((int16_t)(A*1000) and phase switches), so every float operation on
// the data path is an explicit round-to-nearest intrinsic (__fadd_rn/__fmul_rn/__fdiv_rn/
// __fsqrt_rn).  Those are never contracted into FMAs by nvcc regardless of -fmad; the
// library is additionally compiled with -fmad=false.  __fmaf_rn appears only inside
// exhaustively verified replacement sequences (see rk_exact.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/robotick.h"

#define RK_DEV __device__ __forceinline__

namespace rk {

RK_DEV float fadd(float a, float b) { return __fadd_rn(a, b); }
RK_DEV float fsub(float a, float b) { return __fsub_rn(a, b); }
RK_DEV float fmul(float a, float b) { return __fmul_rn(a, b); }
RK_DEV float fdiv(float a, float b) { return __fdiv_rn(a, b); }
RK_DEV float fsqrt(float a) { return __fsqrt_rn(a); }

RK_DEV int32_t sext16(int32_t v) { return (int32_t)(int16_t)v; }
RK_DEV uint32_t pack16(int32_t lo, int32_t hi) { return ((uint32_t)lo & 0xFFFFu) | ((uint32_t)hi << 16); }
RK_DEV int32_t lo16(uint32_t w) { return (int32_t)(int16_t)(w & 0xFFFFu); }
RK_DEV int32_t hi16(uint32_t w) { return ((int32_t)w) >> 16; }

// (int32_t)(float) as the x86 build of the firmware source performs it: cvttss2si, which
// returns INT_MIN for NaN / out of range (F2I.TRUNC saturates instead).
RK_DEV int32_t f2i_x86(float f) {
  const int32_t r = __float2int_rz(f);
  return (fabsf(f) < 2147483648.0f) ? r : (int32_t)0x80000000u;
}
// (int16_t)(float), likewise: cvttss2si to 32 bits, keep the low 16 (C++ leaves out-of-range
// undefined; SURVEY.md Appendix C) -- so a value beyond +-2^31 becomes 0, not -1.
RK_DEV int32_t f2s16(float f) { return sext16(f2i_x86(f)); }

// ---- 128-bit plane access ------------------------------------------------------------
// plane pl of an n-instance block, instance i.  Streaming: each cell is touched once per
// launch, so bypass L1 allocation.
RK_DEV uint4 ld_plane(const uint4 *blk, int64_t n, int pl, int64_t i) {
  return __ldcs(blk + (int64_t)pl * n + i);
}
RK_DEV void st_plane(uint4 *blk, int64_t n, int pl, int64_t i, uint4 v) { __stcs(blk + (int64_t)pl * n + i, v); }

RK_DEV float u2f(uint32_t u) { return __uint_as_float(u); }
RK_DEV uint32_t f2u(float f) { return __float_as_uint(f); }

// The cost-to-go window cell under grid coordinates (u, v) (rk_plan_cost_to_go's goal cell and rk_plan_rollout_field's
// lookup): a window of w x h cells whose cell (0, 0) is grid cell o.  False when (u, v) is off the window, NaN, or the
// window's edges |o| or |o + size| exceed 2^24, where (float) would no longer be exact.
RK_DEV bool plan_window_cell(float u, float v, int2 o, int32_t w, int32_t h, int &ix, int &iy) {
  if(!(o.x >= -(1 << 24) && o.x <= (1 << 24) - w && o.y >= -(1 << 24) && o.y <= (1 << 24) - h)) return false;
  if(!(u >= (float)o.x && u < (float)(o.x + w) && v >= (float)o.y && v < (float)(o.y + h))) return false;
  ix = (int)floorf(u) - o.x, iy = (int)floorf(v) - o.y;
  return true;
}

} // namespace rk

// ---- host-side error plumbing --------------------------------------------------------
namespace rk {
void        set_error(const char *fmt, ...);
int         cuda_fail(cudaError_t e, const char *what);
int         require_device();
// rk_imt_update_yaw / rk_adt_update with a cap on the grid (rk_tick.cu runs them beside the vehicle rollout)
int imt_update_launch(void *d_state, int64_t n, int32_t K, const int16_t *d_regs, const uint8_t *d_have_quat, float *d_out,
                      float *d_yaw_rad, int do_init, int max_ctas, void *stream, const void *d_desc = nullptr);
int adt_update_launch(const rk_adt_params_t *p, void *d_state, const void *d_cmdtab, int64_t n, int32_t K, uint32_t *d_trace,
                      int max_ctas, void *stream);
// rk_plan_rollout_map's checks of an rk_plan_map_t, shared with rk_plan_cost_to_go: the grid (sizes, origin, resolution,
// outside; not w_map) and the tables
int plan_check_map_grid(const char *who, const rk_plan_map_t *map);
int plan_check_map_tables(const char *who, const rk_plan_map_t *map);
} // namespace rk

#define RK_CUDA(call)                                        \
  do {                                                       \
    cudaError_t _e = (call);                                 \
    if(_e != cudaSuccess) return rk::cuda_fail(_e, #call);   \
  } while(0)
