// Miss-ray compaction helpers (compact.cu) and the box sampler's backward in compact row order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace snb {

int compact_plan(const uint8_t* hit, int64_t n_rays, int S, int32_t* order, int32_t* pos, int64_t* counts, cudaStream_t st);
int compact_gather(const float* xyz, const float* vrep, const int32_t* order, const int64_t* counts, int64_t n_rays, int S,
                   float* xyz_c, float* vrep_c, cudaStream_t st);
int compact_expand(const float* sigma_c, const float* rgb_c, const uint8_t* hit, const int32_t* pos, const int64_t* counts,
                   int64_t n_rays, int S, float* sigma, float* rgb, cudaStream_t st);
int compact_reduce(const float* g_sigma, const float* g_rgb, const int32_t* order, const int64_t* counts, int64_t n_rays, int S,
                   float* g_sigma_c, float* g_rgb_c, cudaStream_t st);
int compact_scatter(const float* g_xyz_c, const float* g_vrep_c, const uint8_t* hit, const int32_t* pos, const int64_t* counts,
                    int64_t n_rays, int S, float* g_xyz, float* g_vrep, cudaStream_t st);

// sampler.cu: box-sampler backward reading the decoder's input gradients in compact row order (no scatter to dense)
int sample_box_bwd_compact(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter, int64_t n_rays,
                           int32_t n_samples, float half_diag, const float* h, const float* g_xyz_c, const float* g_vrep_c,
                           const float* g_z_vals, const int32_t* pos, const int64_t* counts, float* g_rays_o, float* g_viewdir,
                           cudaStream_t st);

}  // namespace snb
