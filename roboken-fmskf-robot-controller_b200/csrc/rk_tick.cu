// rk_tick.cu -- the full controller tick (vehicle + IMU + arm) as one asynchronous call.
//
// The firmware's three tasks share exactly one value: the vehicle ISR reads
// deg2rad(IMT::get_status_now_yaw()) before each VEHICLE_CTRL::update() (VD_task_main.cpp:368).
// A monolithic one-thread-per-robot kernel would carry 53 planes of state (848 B) per thread
// and run the issue-bound vehicle tick at a fraction of its occupancy, so the three sub-systems
// stay three kernels -- but none of them waits for another (round 2):
//   * the vehicle rollout forms the yaw itself from the IMU's register snapshots (the Yaw register of
//     sample y scaled as updateData() does, held over updates without a quaternion frame;
//     rk_vdt_rollout_t::d_imu_regs), so the IMU kernel is no longer its predecessor.  The one word it
//     needs from the IMU block -- Data.angle[2] at launch, held if update 0 carries no quaternion frame --
//     is snapshot into the caller's scratch before anything else runs;
//   * the IMU update (one frame per robot: nothing reads the IMU block inside the launch, so only the last
//     sample with a quaternion frame is read -- rk_imu.cu, imt_last_frame) and the arm tick (a few real ticks
//     per segment -- rk_arm.cu, loop_jump) run on a high-priority side stream.  The vehicle kernel fills the
//     register file with four 128-thread CTAs per SM; whenever one of its CTAs retires, a pending
//     high-priority CTA takes the slot, so the two small kernels execute inside the vehicle rollout's shadow
//     instead of after it.  Their grids are uncapped by default: each side CTA then finishes its 128 or 256
//     robots and gives the slot back, where a capped grid of one CTA per SM holds a vehicle slot for the
//     whole latency-bound stride over the batch (RK_OPT_TICK_SIDE_CTAS caps them; DESIGN.md 3.5).
#include <mutex>

#include "rk_common.cuh"

namespace rk {
struct TickStreams {
  cudaStream_t side = nullptr;
  cudaEvent_t  fork = nullptr, join = nullptr;
  int          sm_count = 0;
  // diagnostics (rk_tick_debug_timeline): timestamps of the last call's kernels, recorded only while enabled
  cudaEvent_t tl[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};
static bool g_tick_timeline = false;
static std::mutex  g_tick_mu; // held across the whole fork / launch / join sequence: the event pair is per device
static TickStreams g_tick[64];
static int         g_tick_side_ctas_per_sm = 0; // rk_set_option(RK_OPT_TICK_SIDE_CTAS, 0..8): 0 = uncapped grids

int tick_set_side_ctas(int v) {
  if(v < 0 || v > 8) return RK_ERR_ARG;
  g_tick_side_ctas_per_sm = v;
  return RK_OK;
}

static int tick_streams(TickStreams **out) {
  int dev = 0;
  RK_CUDA(cudaGetDevice(&dev));
  if(dev < 0 || dev >= 64) {
    set_error("rk_tick_rollout: device index %d out of range", dev);
    return RK_ERR_ARG;
  }
  TickStreams &t = g_tick[dev];
  if(!t.side) {
    int lo = 0, hi = 0; // numerically lower = higher priority
    RK_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    RK_CUDA(cudaStreamCreateWithPriority(&t.side, cudaStreamNonBlocking, hi));
    RK_CUDA(cudaEventCreateWithFlags(&t.fork, cudaEventDisableTiming));
    RK_CUDA(cudaEventCreateWithFlags(&t.join, cudaEventDisableTiming));
    RK_CUDA(cudaDeviceGetAttribute(&t.sm_count, cudaDevAttrMultiProcessorCount, dev));
  }
  *out = &t;
  return RK_OK;
}

// Data.angle[2] (degrees) of every IMU block -> yaw0[i]
__global__ void tick_yaw0_kernel(const uint4 *__restrict__ imt_state, int64_t n, float *__restrict__ yaw0) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  constexpr int W = RK_IS_DATA + RK_IS_D_ANGLE + 2;
  const uint4   q = imt_state[(int64_t)(W / 4) * n + i];
  yaw0[i]         = u2f(W % 4 == 0 ? q.x : W % 4 == 1 ? q.y : W % 4 == 2 ? q.z : q.w);
}
} // namespace rk

using namespace rk;

extern "C" int rk_tick_rollout(const rk_vdt_params_t *vp, const rk_adt_params_t *ap, void *d_vdt_state, void *d_imt_state,
                               void *d_adt_state, const void *d_adt_cmdtab, int64_t n, const rk_tick_rollout_t *a, void *stream) {
  if(!vp || !ap || !a) {
    set_error("rk_tick_rollout: NULL params/args");
    return RK_ERR_ARG;
  }
  if(n == 0 || a->steps == 0) return RK_OK;
  if(n < 0 || a->steps < 0 || a->slow_period <= 0 || (!a->d_regs && !(a->d_imu_desc && a->d_yaw_reg)) || !a->d_yaw || !d_imt_state ||
     ((uintptr_t)d_imt_state & 15u)) {
    set_error("rk_tick_rollout: bad n / steps / slow_period, or d_regs (or d_imu_desc + d_yaw_reg) / d_yaw / d_imt_state NULL or misaligned");
    return RK_ERR_ARG;
  }
  if(int rc = require_device()) return rc;
  std::lock_guard<std::mutex> lk(g_tick_mu);
  TickStreams                *ts = nullptr;
  if(int rc = tick_streams(&ts)) return rc;
  cudaStream_t  st     = (cudaStream_t)stream;
  const int32_t n_slow = (a->steps + a->slow_period - 1) / a->slow_period;
  const int     cap    = g_tick_side_ctas_per_sm * ts->sm_count;

  auto mark = [&](int k, cudaStream_t s) { // diagnostics only
    if(!g_tick_timeline) return;
    if(!ts->tl[k]) cudaEventCreate(&ts->tl[k]);
    cudaEventRecord(ts->tl[k], s);
  };
  mark(0, st);
  // what the vehicle holds if IMU update 0 carries no quaternion frame; taken before the IMU kernel can store
  tick_yaw0_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const uint4 *)d_imt_state, n, a->d_yaw);
  RK_CUDA(cudaGetLastError());

  // IMU: n_slow updates, arm: n_slow ticks -- on the side stream, forked from / joined to the caller's stream
  RK_CUDA(cudaEventRecord(ts->fork, st));
  RK_CUDA(cudaStreamWaitEvent(ts->side, ts->fork, 0));
  mark(1, ts->side);
  // d_imu_desc: the IMU update draws its samples in registers (the vehicle reads the Yaw column the generator wrote)
  int rc = imt_update_launch(d_imt_state, n, n_slow, a->d_regs, a->d_have_quat, nullptr, nullptr, 0, cap, ts->side,
                             (a->d_imu_desc && a->d_yaw_reg) ? (const void *)a->d_imu_desc : nullptr);
  mark(2, ts->side);
  if(rc == RK_OK) rc = adt_update_launch(ap, d_adt_state, d_adt_cmdtab, n, n_slow, a->d_adt_trace, cap, ts->side);
  mark(3, ts->side);
  const cudaError_t ej = cudaEventRecord(ts->join, ts->side); // whatever was enqueued on the side stream is joined below
  if(rc == RK_OK && ej == cudaSuccess) {
    rk_vdt_rollout_t v = {};
    v.steps = a->steps, v.sensor_mode = RK_SENSOR_PLANT;
    v.d_cmd = a->d_cmd, v.n_seg = a->n_seg, v.seg_len = a->seg_len;
    if(a->d_yaw_reg) v.d_yaw_reg = a->d_yaw_reg; // the Yaw column in 2 bytes per sample (same hold semantics)
    else v.d_imu_regs = a->d_regs;
    v.d_imu_have_quat = a->d_have_quat, v.d_imu_yaw0_deg = a->d_yaw;
    v.n_yaw = n_slow, v.yaw_period = a->slow_period;
    v.d_trace = a->d_vdt_trace, v.d_goal = a->d_goal, v.d_cost = a->d_cost;
    v.reset_state = a->reset_vehicle;
    mark(4, st);
    rc = rk_vdt_rollout(vp, d_vdt_state, n, &v, st);
    mark(5, st);
  }
  if(ej == cudaSuccess) {
    const cudaError_t ew = cudaStreamWaitEvent(st, ts->join, 0);
    if(ew != cudaSuccess && rc == RK_OK) rc = cuda_fail(ew, "cudaStreamWaitEvent(join)");
  } else if(rc == RK_OK) {
    rc = cuda_fail(ej, "cudaEventRecord(join)");
  }
  return rc;
}

/* Diagnostics: enable = 1 makes the following rk_tick_rollout calls record timestamps; with out != NULL the call
 * synchronises the device and returns, for the LAST rk_tick_rollout on the current device, milliseconds relative to
 * its entry: [0] side stream starts, [1] IMU kernel done, [2] arm kernel done, [3] vehicle rollout starts,
 * [4] vehicle rollout done. */
extern "C" int rk_tick_debug_timeline(int enable, float out[5]) {
  if(int rc = require_device()) return rc;
  std::lock_guard<std::mutex> lk(g_tick_mu);
  g_tick_timeline = enable != 0;
  if(!out) return RK_OK;
  TickStreams *ts = nullptr;
  if(int rc = tick_streams(&ts)) return rc;
  RK_CUDA(cudaDeviceSynchronize());
  for(int k = 0; k < 5; k++) {
    out[k] = -1.0f;
    if(ts->tl[0] && ts->tl[k + 1]) cudaEventElapsedTime(&out[k], ts->tl[0], ts->tl[k + 1]);
  }
  cudaGetLastError();
  return RK_OK;
}
