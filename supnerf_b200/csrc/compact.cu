// Miss-ray compaction for the fused box render (bf16 modes).
//
// A ray that misses the object's box gets near = far = -1 (renderer.py:103-110), so its S samples are ONE point, the decoder's
// S outputs are identical and only the last sample carries weight (SURVEY.md §3.1, §8d "accounting rule for miss rays": a
// kernel may run one decoder row per miss ray as long as throughput accounting uses the rows it really executed).  With the
// reference's roi (a square around the projected box) 30-60 % of the rays hit: the decoder is >90 % of the step, so this is a
// ~2x cut in work.  Everything stays on the device -- the host never learns the counts:
//   plan     hit mask (N) -> order[] (hit rays first, then miss rays), pos[] (rank inside its class), counts {n_hit, n_miss,
//            rows, rows padded to the 128-row tile} ; one block, N <= a few 10^5
//   gather   dense xyz / viewdir (N,S,3) -> compact rows: hit rays S rows each, then one row per miss ray, then padding
//   expand   compact sigma / rgb -> dense (N,S): miss rays replicated, so the unmodified compositing kernels run on them
//   reduce   dense d sigma / d rgb -> compact: miss rays summed over their S samples (the decoder row is shared)
// The box sampler's backward reads d xyz / d viewdir in compact row order (sampler.cu, sample_box_bwd_compact): a miss ray's row is
// credited to its last sample -- the backward only uses sum_k g_x_k (origin) and sum_k z_k g_x_k with z_k = -1 for every k
// (direction) on miss rays, both independent of which k holds it.
// Exact: same per-row decoder arithmetic; gradients differ from the dense path only by fp32 summation order.
#include "common.cuh"
#include "compact.h"

namespace snb {

// one block: the rays ranked hit-first, then the row counts
__global__ void __launch_bounds__(1024) compact_plan_kernel(const uint8_t* __restrict__ hit, int64_t n_rays, int S,
                                                           int32_t* __restrict__ order, int32_t* __restrict__ pos,
                                                           int64_t* __restrict__ counts) {
  const int n_hit = rank_hits_first(hit, n_rays, order, pos);
  if (threadIdx.x == 0) {
    const int64_t n_miss = n_rays - n_hit;
    const int64_t rows = (int64_t)n_hit * S + n_miss;
    counts[0] = n_hit; counts[1] = n_miss; counts[2] = rows; counts[3] = (rows + 127) / 128 * 128;
  }
}

__global__ void __launch_bounds__(256) compact_gather_kernel(const float* __restrict__ xyz, const float* __restrict__ vrep,
                                                            const int32_t* __restrict__ order, const int64_t* __restrict__ counts,
                                                            int S, float* __restrict__ xyz_c, float* __restrict__ vrep_c) {
  const int64_t n_hit = counts[0], rows = counts[2], rows_pad = counts[3];
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows_pad; r += (int64_t)gridDim.x * blockDim.x) {
    int64_t src;
    if (r < n_hit * S) src = (int64_t)order[r / S] * S + (r % S);
    else if (r < rows) src = (int64_t)order[n_hit + (r - n_hit * S)] * S + (S - 1);   // a miss ray's samples are one point (to an ulp of z): take the last, the only one with weight
    else src = 0;                                                           // padding up to the tile: results ignored
#pragma unroll
    for (int a = 0; a < 3; ++a) { xyz_c[3 * r + a] = __ldg(xyz + 3 * src + a); vrep_c[3 * r + a] = __ldg(vrep + 3 * src + a); }
  }
}

__device__ __forceinline__ int64_t compact_row(bool h, int p, int k, int64_t n_hit, int S) {
  return h ? (int64_t)p * S + k : n_hit * S + p;
}

__global__ void __launch_bounds__(256) compact_expand_kernel(const float* __restrict__ sigma_c, const float* __restrict__ rgb_c,
                                                            const uint8_t* __restrict__ hit, const int32_t* __restrict__ pos,
                                                            const int64_t* __restrict__ counts, int64_t n_rays, int S,
                                                            float* __restrict__ sigma, float* __restrict__ rgb) {
  const int64_t n_hit = counts[0], total = n_rays * S;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t ray = i / S;
    const int64_t r = compact_row(hit[ray] != 0, pos[ray], (int)(i % S), n_hit, S);
    sigma[i] = __ldg(sigma_c + r);
    rgb[3 * i] = __ldg(rgb_c + 3 * r); rgb[3 * i + 1] = __ldg(rgb_c + 3 * r + 1); rgb[3 * i + 2] = __ldg(rgb_c + 3 * r + 2);
  }
}

// one warp per compact row group: hit rows copy, miss rows sum over the ray's S dense samples
__global__ void __launch_bounds__(256) compact_reduce_kernel(const float* __restrict__ g_sigma, const float* __restrict__ g_rgb,
                                                            const int32_t* __restrict__ order, const int64_t* __restrict__ counts,
                                                            int S, float* __restrict__ g_sigma_c, float* __restrict__ g_rgb_c) {
  const int64_t n_hit = counts[0], rows = counts[2], rows_pad = counts[3];
  const int64_t hit_rows = n_hit * S;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r = gt; r < hit_rows; r += nt) {                      // hit rows: plain copy
    const int64_t src = (int64_t)order[r / S] * S + (r % S);
    g_sigma_c[r] = __ldg(g_sigma + src);
    g_rgb_c[3 * r] = __ldg(g_rgb + 3 * src); g_rgb_c[3 * r + 1] = __ldg(g_rgb + 3 * src + 1); g_rgb_c[3 * r + 2] = __ldg(g_rgb + 3 * src + 2);
  }
  const int lane = threadIdx.x & 31;
  const int64_t gw = gt >> 5, nw = nt >> 5;
  for (int64_t m = gw; m < rows_pad - hit_rows; m += nw) {           // miss rows (and the zero padding)
    const int64_t r = hit_rows + m;
    float a = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f;
    if (r < rows) {
      const int64_t src = (int64_t)order[n_hit + m] * S;
      for (int k = lane; k < S; k += 32) {
        a += __ldg(g_sigma + src + k);
        b0 += __ldg(g_rgb + 3 * (src + k)); b1 += __ldg(g_rgb + 3 * (src + k) + 1); b2 += __ldg(g_rgb + 3 * (src + k) + 2);
      }
      a = warp_sum(a); b0 = warp_sum(b0); b1 = warp_sum(b1); b2 = warp_sum(b2);
    }
    if (lane == 0) { g_sigma_c[r] = a; g_rgb_c[3 * r] = b0; g_rgb_c[3 * r + 1] = b1; g_rgb_c[3 * r + 2] = b2; }
  }
}

int compact_plan(const uint8_t* hit, int64_t n_rays, int S, int32_t* order, int32_t* pos, int64_t* counts, cudaStream_t st) {
  SNB_REQUIRE(n_rays < (int64_t)1 << 30, "compact_plan: too many rays");
  compact_plan_kernel<<<1, 1024, 0, st>>>(hit, n_rays, S, order, pos, counts);
  SNB_LAUNCH_CHECK();
  return 0;
}
int compact_gather(const float* xyz, const float* vrep, const int32_t* order, const int64_t* counts, int64_t n_rays, int S,
                   float* xyz_c, float* vrep_c, cudaStream_t st) {
  const int g = grid_1d(n_rays * S, 256, 8);
  SNB_REQUIRE(g > 0, "compact_gather: no CUDA device");
  compact_gather_kernel<<<g, 256, 0, st>>>(xyz, vrep, order, counts, S, xyz_c, vrep_c);
  SNB_LAUNCH_CHECK();
  return 0;
}
int compact_expand(const float* sigma_c, const float* rgb_c, const uint8_t* hit, const int32_t* pos, const int64_t* counts,
                   int64_t n_rays, int S, float* sigma, float* rgb, cudaStream_t st) {
  const int g = grid_1d(n_rays * S, 256, 8);
  SNB_REQUIRE(g > 0, "compact_expand: no CUDA device");
  compact_expand_kernel<<<g, 256, 0, st>>>(sigma_c, rgb_c, hit, pos, counts, n_rays, S, sigma, rgb);
  SNB_LAUNCH_CHECK();
  return 0;
}
int compact_reduce(const float* g_sigma, const float* g_rgb, const int32_t* order, const int64_t* counts, int64_t n_rays, int S,
                   float* g_sigma_c, float* g_rgb_c, cudaStream_t st) {
  const int g = grid_1d(n_rays * S, 256, 8);
  SNB_REQUIRE(g > 0, "compact_reduce: no CUDA device");
  compact_reduce_kernel<<<g, 256, 0, st>>>(g_sigma, g_rgb, order, counts, S, g_sigma_c, g_rgb_c);
  SNB_LAUNCH_CHECK();
  return 0;
}
}  // namespace snb
