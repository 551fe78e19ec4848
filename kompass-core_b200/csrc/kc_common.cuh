// kc_common.cuh — shared helpers for the sm_100a kernels and their host launchers.
//
// Numerics contract (DESIGN.md §Numerics): the whole library is compiled with -fmad=false, so
// every float/double multiply and add rounds separately exactly like the reference's baseline
// x86-64 build; division and sqrt are IEEE round-to-nearest (nvcc default -prec-div/-prec-sqrt).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cfloat>
#include <cstdarg>
#include <cstdio>
#include <string>

#include "../../include/kompass_b200.h"

namespace kc {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char *fmt, ...);
int32_t cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define KC_CUDA(expr)                                                     \
  do {                                                                    \
    cudaError_t _e = (expr);                                              \
    if (_e != cudaSuccess) return kc::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define KC_REQUIRE(cond, code, ...) \
  do {                              \
    if (!(cond)) {                  \
      kc::set_error(__VA_ARGS__);   \
      return (code);                \
    }                               \
  } while (0)

#define KC_TRY(expr)              \
  do {                            \
    int32_t _rc = (expr);         \
    if (_rc != KC_OK) return _rc; \
  } while (0)

// Grow-only device / pinned buffers (never shrunk, like the reference's device buffers,
// ref: src/utils/cost_evaluator_gpu.cpp:245-271).
template <typename T>
struct DevBuf {
  T *ptr = nullptr;
  size_t cap = 0;
  int32_t reserve(size_t n) {
    if (n <= cap) return KC_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = n + n / 4 + 64;
    cudaError_t e = cudaMalloc(&ptr, want * sizeof(T));
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("cudaMalloc of %zu bytes failed: %s", want * sizeof(T), cudaGetErrorString(e));
      return e == cudaErrorMemoryAllocation ? KC_ERR_OOM : KC_ERR_CUDA;
    }
    cap = want;
    return KC_OK;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

template <typename T>
struct PinnedBuf {
  T *ptr = nullptr;
  size_t cap = 0;
  int32_t reserve(size_t n) {
    if (n <= cap) return KC_OK;
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = n + n / 4 + 64;
    cudaError_t e = cudaHostAlloc(&ptr, want * sizeof(T), cudaHostAllocDefault);
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("cudaHostAlloc of %zu bytes failed: %s", want * sizeof(T), cudaGetErrorString(e));
      return KC_ERR_OOM;
    }
    cap = want;
    return KC_OK;
  }
  void release() {
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

int32_t ensure_device();  // selects the device (LOCAL_RANK aware) once per process; KC_ERR_CUDA if none
int sm_count();
int device_index();  // the CUDA device this process's handles live on

// ---- batched launch set of independent robots (kc_planner.cu) --------------------------------
// Used by kc_planner_batch_cloud (every robot on the planner's own path and horizon) and by the
// fleet controller (kc_dwa.cu: every robot with its own path, horizon, tracked segment and sensor).

// TrajectorySampler::updateHorizon (trajectory_sampler.cpp:316-326): clamps `horizon` to
// [2 time_step, base_horizon] in place and returns the points per trajectory it gives.
int32_t horizon_points(double time_step, double base_horizon, double &horizon);

struct BatchPath {  // a robot's reference path: host X / Y (segment length and step), device X / Y / acc
  const float *hX = nullptr, *hY = nullptr;
  const float *dX = nullptr, *dY = nullptr, *dAcc = nullptr;
  int32_t n = 0;
  float total_length = 0.0f;
};
struct BatchRobot {
  const double *vel = nullptr, *pose = nullptr;  // [3] each
  int32_t P = 0;                                 // points per trajectory (<= the planner's base horizon)
  BatchPath path;
  int32_t seg_start = 0, seg_count = 0;  // tracked segment (Path::getPart range)
  int64_t offset = 0;                    // sensor slice: `count` points / beams from `offset`
  int32_t count = 0;
};
struct BatchSensor {  // one sensor kind for every robot of a call
  bool cloud = true;
  const float *xyz = nullptr;                      // clouds: [n x 3], world frame
  const double *ranges = nullptr, *angles = nullptr;  // scans: beam arrays
};
// One control cycle for R robots, chunk after chunk of launch sets. results [R] always; cycles [R]
// (may be NULL) also receives every robot's winner record (rows point into the planner's host
// copy, valid until its next call).
int32_t planner_batch(kc_planner *p, int32_t R, const BatchRobot *robots, const BatchSensor &sensor,
                      kc_batch_result *results, kc_cycle_result *cycles);

#ifdef __CUDACC__
// ---- warp helpers ----------------------------------------------------------------------------
constexpr unsigned FULL = 0xffffffffu;

// Device-scope acquire/release fence for the "last CTA finishes the job" pattern. __threadfence()
// is membar.gl = fence.sc.gpu (MEMBAR.SC + L1 invalidate), far heavier than the ordering the ticket
// protocol needs when every CTA of a grid executes it.
__device__ __forceinline__ void fence_acq_rel() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// Programmatic dependent launch (consecutive kernels of one stream launched with
// cudaLaunchAttributeProgrammaticStreamSerialization): the producer lets the next grid be staged
// early, the consumer runs its prologue (anything that reads no producer output) and then waits for
// the producer grid to have completed with its writes visible. Both are no-ops in a plain launch.
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ double shfl_d(double v, int src) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_sync(FULL, lo, src);
  hi = __shfl_sync(FULL, hi, src);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_xor_d(double v, int m) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_xor_sync(FULL, lo, m);
  hi = __shfl_xor_sync(FULL, hi, m);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v = fmin(v, shfl_xor_d(v, m));
  return v;
}
// (value, index) lexicographic min: lower value, ties -> lower index
__device__ __forceinline__ void warp_argmin_f(float &v, int &i) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    float ov = __shfl_xor_sync(FULL, v, m);
    int oi = __shfl_xor_sync(FULL, i, m);
    if (ov < v || (ov == v && oi < i)) {
      v = ov;
      i = oi;
    }
  }
}
#endif

}  // namespace kc
