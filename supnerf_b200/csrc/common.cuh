// Shared helpers for the supnerf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <stdint.h>
#include <stdio.h>

namespace snb {

void set_error(const char* fmt, ...);

#define SNB_CHECK_CUDA(expr)                                                               \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      snb::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

#define SNB_REQUIRE(cond, ...)         \
  do {                                 \
    if (!(cond)) {                     \
      snb::set_error(__VA_ARGS__);     \
      return 2;                        \
    }                                  \
  } while (0)

extern std::atomic<unsigned long long> g_launches;  // kernels launched by this library (all host threads), for bench.py's gpu_launches
#define SNB_LAUNCH_CHECK()            \
  do {                                \
    snb::g_launches.fetch_add(1, std::memory_order_relaxed); \
    SNB_CHECK_CUDA(cudaGetLastError()); \
  } while (0)

int sm_count();  // cached per device; <=0 on failure

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// gridDim.x of a grid-stride launch over n items, per_block items per block: ceil(n / per_block) blocks, at least one, at most
// ceil(per_sm * SMs / n_objs) -- an equal share of per_sm blocks per SM for each of the n_objs objects a launch spreads over
// gridDim.y.  <= 0 when there is no device.
static inline int grid_1d(int64_t n, int64_t per_block, int per_sm, int n_objs = 1) {
  const int sms = sm_count();
  if (sms <= 0) return sms;
  const int64_t blocks = ceil_div(n > 0 ? n : 1, per_block), cap = ceil_div((int64_t)per_sm * sms, n_objs);
  return (int)(blocks < cap ? blocks : cap);
}

}  // namespace snb
