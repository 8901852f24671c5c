// Miss-ray compaction helpers (compact.cu), the hit-first ranking they share with the batched render (render_batch.cu) and the box
// sampler's backward in compact row order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace snb {

// The n rays of `hit` ranked hit-first by ONE block of 1024 threads: order[] = the hit rays, then the miss rays, each class in
// ascending index; pos[i] = ray i's rank inside its class.  Returns the number of hit rays, in every thread.
// Pre-pass: total number of hits (so the miss rays can be placed behind them).  Then super-chunks of 16 384 rays: warp w owns 512
// consecutive rays as 16 coalesced 32-byte rows held in registers (16 independent loads = one memory latency), ballots give the
// in-row ranks, a 32-entry shared-memory scan the warp offsets, a running carry the rest.
__device__ __forceinline__ int rank_hits_first(const uint8_t* __restrict__ hit, int64_t n, int32_t* __restrict__ order,
                                               int32_t* __restrict__ pos) {
  __shared__ int warp_tot[32];
  __shared__ int total_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt = (1u << lane) - 1u;
  int local = 0;
  for (int64_t i0 = 0; i0 < n; i0 += 8 * 1024) {
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int64_t i = i0 + (int64_t)k * 1024 + tid; local += (i < n && hit[i]) ? 1 : 0; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if (lane == 0) warp_tot[warp] = local;
  __syncthreads();
  if (tid == 0) { int t = 0; for (int w = 0; w < 32; ++w) t += warp_tot[w]; total_s = t; }
  __syncthreads();
  const int n_hit = total_s;
  int carry = 0;   // hits in earlier super-chunks (identical in every thread)
  for (int64_t sc = 0; sc < n; sc += 16384) {
    const int64_t wbase = sc + (int64_t)warp * 512;
    unsigned m[16];
    int wcnt = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const int64_t i = wbase + k * 32 + lane;
      m[k] = __ballot_sync(0xffffffffu, i < n && hit[i]);
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) wcnt += __popc(m[k]);
    __syncthreads();                       // warp_tot is free again
    if (lane == 0) warp_tot[warp] = wcnt;
    __syncthreads();
    int before = carry, chunk_tot = 0;
    for (int w = 0; w < 32; ++w) { const int t = warp_tot[w]; if (w < warp) before += t; chunk_tot += t; }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const int64_t i = wbase + k * 32 + lane;
      const int h = (m[k] >> lane) & 1u;
      const int hits_before = before + __popc(m[k] & lt);      // hit rays with a smaller index
      if (i < n) {
        const int p = h ? hits_before : (int)(i - hits_before);   // rank inside its class
        pos[i] = p;
        order[h ? p : n_hit + p] = (int32_t)i;
      }
      before += __popc(m[k]);
    }
    carry += chunk_tot;
  }
  return n_hit;
}

int compact_plan(const uint8_t* hit, int64_t n_rays, int S, int32_t* order, int32_t* pos, int64_t* counts, cudaStream_t st);
int compact_gather(const float* xyz, const float* vrep, const int32_t* order, const int64_t* counts, int64_t n_rays, int S,
                   float* xyz_c, float* vrep_c, cudaStream_t st);
int compact_expand(const float* sigma_c, const float* rgb_c, const uint8_t* hit, const int32_t* pos, const int64_t* counts,
                   int64_t n_rays, int S, float* sigma, float* rgb, cudaStream_t st);
int compact_reduce(const float* g_sigma, const float* g_rgb, const int32_t* order, const int64_t* counts, int64_t n_rays, int S,
                   float* g_sigma_c, float* g_rgb_c, cudaStream_t st);

// sampler.cu: box-sampler backward reading the decoder's input gradients in compact row order (no scatter to dense)
int sample_box_bwd_compact(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter, int64_t n_rays,
                           int32_t n_samples, float half_diag, const float* h, const float* g_xyz_c, const float* g_vrep_c,
                           const float* g_z_vals, const int32_t* pos, const int64_t* counts, float* g_rays_o, float* g_viewdir,
                           cudaStream_t st);

}  // namespace snb
