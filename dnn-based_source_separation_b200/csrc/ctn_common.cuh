// Shared device/host helpers for the Conv-TasNet sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ctn_b200.h"

#define CTN_TILE_T 128  // activation pitch granularity (frames)

// launch counter (thread local) -- bench.py reports it as gpu_launches
extern thread_local int g_ctn_launches;
extern thread_local long long g_ctn_total_launches;
extern thread_local int g_ctn_depth;
extern thread_local int g_ctn_last_launches;
#define CTN_COUNT_LAUNCH() (++g_ctn_total_launches, ++g_ctn_launches)
// every extern "C" entry opens one; the outermost scope resets / publishes the launch count and makes the device that owns
// `devptr` (any device pointer argument of the call) current for the duration of the call: kernels, memsets and function
// attributes always go to the tensors' GPU, whatever the caller's current device is (restored on exit)
struct LaunchScope {
  int prev_dev = -1;
  explicit LaunchScope(const void* devptr = nullptr) {
    if (g_ctn_depth++ == 0) {
      g_ctn_launches = 0;
      if (devptr) {
        cudaPointerAttributes at;
        int cur = 0;
        if (cudaPointerGetAttributes(&at, devptr) == cudaSuccess && at.type == cudaMemoryTypeDevice &&
            cudaGetDevice(&cur) == cudaSuccess && cur != at.device) {
          prev_dev = cur;
          cudaSetDevice(at.device);
        }
        cudaGetLastError();  // a host pointer is not an error here
      }
    }
  }
  ~LaunchScope() {
    if (--g_ctn_depth == 0) {
      g_ctn_last_launches = g_ctn_launches;
      if (prev_dev >= 0) cudaSetDevice(prev_dev);
    }
  }
};
#define CTN_MAX_DEVICES 64
static inline int ctn_current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return (d >= 0 && d < CTN_MAX_DEVICES) ? d : 0;
}
// SM count of the current device (persistent grids are sized by it), queried once per device ordinal
inline int ctn_num_sms() {
  static int sms[CTN_MAX_DEVICES] = {};
  const int dev = ctn_current_device();
  if (sms[dev] <= 0) {
    cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
    if (sms[dev] <= 0) sms[dev] = 148;
  }
  return sms[dev];
}

#define CTN_RETURN_IF_CUDA_ERR()                      \
  do {                                                \
    cudaError_t _e = cudaGetLastError();              \
    if (_e != cudaSuccess) return (int)_e;            \
  } while (0)

#define CTN_TRY(expr)                                 \
  do {                                                \
    int _s = (expr);                                  \
    if (_s != 0) return _s;                           \
  } while (0)

static inline int ctn_round_up(int v, int m) { return (v + m - 1) / m * m; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of (a, b) accumulated in double, result valid in thread 0.  red must hold 2*32 doubles.
__device__ __forceinline__ void block_sum2_d(double& a, double& b, double* red) {
  a = warp_sum_d(a);
  b = warp_sum_d(b);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) { red[wid] = a; red[32 + wid] = b; }
  __syncthreads();
  if (wid == 0) {
    a = lane < nw ? red[lane] : 0.0;
    b = lane < nw ? red[32 + lane] : 0.0;
    a = warp_sum_d(a);
    b = warp_sum_d(b);
  }
}

// (mean, rstd) of a gLN group from its (sum, sumsq) in double; n = C*frames.  GroupNorm: biased variance,
// eps inside the sqrt (src/modules/norm.py:18).
__device__ __forceinline__ float2 gln_mean_rstd(const double* __restrict__ st, double n, float eps) {
  const double mean = st[0] / n;
  double var = st[1] / n - mean * mean;
  var = var > 0.0 ? var : 0.0;
  return make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
}

__device__ __forceinline__ float prelu_f(float v, float a) { return v >= 0.f ? v : a * v; }

// ---- optional stage timing (ctn_profile_enable / ctn_profile_read) -------------------------------------------
void ctn_prof_begin(int stage, cudaStream_t st);
void ctn_prof_end(int stage, cudaStream_t st);
struct StageTimer {
  int stage; cudaStream_t st;
  StageTimer(int s, cudaStream_t stream) : stage(s), st(stream) { ctn_prof_begin(stage, st); }
  ~StageTimer() { ctn_prof_end(stage, st); }
};
