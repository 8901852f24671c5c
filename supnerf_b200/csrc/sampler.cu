// K1 / K1b — ray generation, ray/AABB slab test, stratified depth sampling (box stack of
// renderer.py) and the spherical-shell sampler (utils.py stack), forward and backward to the rays /
// the camera pose.  One warp per ray, lanes across samples, so the (N,S,3) tensors are written and
// read as contiguous 12*S-byte rows.  Arithmetic that decides integers (the hit mask) or that the
// reference evaluates as separate fp32 ops uses explicit round-to-nearest intrinsics so nvcc cannot
// contract it into FMAs.
#include "common.cuh"
#include "sampler.cuh"
#include "../../include/supnerf_b200.h"
#include <math.h>

namespace snb {

__global__ void __launch_bounds__(256) get_rays_fwd_kernel(const float* __restrict__ px, const float* __restrict__ py,
                                                          int64_t n, const float* __restrict__ K,
                                                          const float* __restrict__ c2w, float* __restrict__ rays_o,
                                                          float* __restrict__ viewdir) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float d[3];
    pixel_dir(K, c2w, px[i], py[i], d);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      viewdir[3 * i + a] = d[a];
      rays_o[3 * i + a] = __ldg(c2w + 4 * a + 3);
    }
  }
}

// g_c2w[i][j<3] += sum_rays g_r[i] p[j],  g_c2w[i][3] += sum_rays g_o[i];  g_r = (g_d - d (g_d.d)) / |r|
__global__ void __launch_bounds__(256) get_rays_bwd_kernel(const float* __restrict__ px, const float* __restrict__ py,
                                                          int64_t n, const float* __restrict__ K,
                                                          const float* __restrict__ c2w,
                                                          const float* __restrict__ g_o, const float* __restrict__ g_d,
                                                          float* __restrict__ g_c2w) {
  float acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gd[3] = {g_d[3 * i], g_d[3 * i + 1], g_d[3 * i + 2]};
    float p[3], gr[3];
    dir_grad_to_pose(K, c2w, px[i], py[i], gd, p, gr);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      acc[4 * a + 0] += gr[a] * p[0];
      acc[4 * a + 1] += gr[a] * p[1];
      acc[4 * a + 2] += gr[a] * p[2];
      acc[4 * a + 3] += g_o[3 * i + a];
    }
  }
  __shared__ float red[8][12];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    float v = warp_sum(acc[i]);
    if (lane == 0) red[w][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    float v = 0.f;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) v += red[k][threadIdx.x];
    atomicAdd(g_c2w + threadIdx.x, v);
  }
}

__global__ void __launch_bounds__(256) sample_box_fwd_kernel(
    const float* __restrict__ rays_o, const float* __restrict__ viewdir, const float* __restrict__ z_steps,
    const float* __restrict__ jitter, int64_t n_rays, int S, float half_diag, float hx, float hy, float hz,
    float* __restrict__ xyz, float* __restrict__ vrep, float* __restrict__ z_vals, uint8_t* __restrict__ hit) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float half[3] = {hx, hy, hz};
  const float fstep = (float)(1.0 / (double)S);  // python float 1.0/S, rounded to fp32 when it scales the fp32 draw
  for (int64_t ray = warp; ray < n_rays; ray += nwarps) {
    float o[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      o[a] = __fdiv_rn(__ldg(rays_o + 3 * ray + a), half_diag);  // rays_o / (obj_diag / 2), renderer.py:102
      d[a] = __ldg(viewdir + 3 * ray + a);
    }
    const Slab sl = slab_test(o, d, half);
    const float near = sl.hit ? sl.t_near : -1.f, far = sl.hit ? sl.t_far : -1.f;
    if (lane == 0) hit[ray] = sl.hit ? 1 : 0;
    for (int k = lane; k < S; k += 32) {
      const float zs = __fadd_rn(__ldg(z_steps + k), __fmul_rn(__ldg(jitter + ray * S + k), fstep));
      const float zc = __fadd_rn(__fmul_rn(near, __fsub_rn(1.f, zs)), __fmul_rn(far, zs));
      float x[3], q = 0.f;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        x[a] = __fadd_rn(o[a], __fmul_rn(zc, d[a]));
        const float m = __fmul_rn(__fsub_rn(x[a], o[a]), half_diag);
        q = __fadd_rn(q, __fmul_rn(m, m));
      }
      const int64_t idx = ray * S + k;
      xyz[3 * idx] = x[0]; xyz[3 * idx + 1] = x[1]; xyz[3 * idx + 2] = x[2];
      if (vrep) { vrep[3 * idx] = d[0]; vrep[3 * idx + 1] = d[1]; vrep[3 * idx + 2] = d[2]; }
      z_vals[idx] = sqrtf(q);
    }
  }
}

__global__ void __launch_bounds__(256) ray_box_fwd_kernel(const float* __restrict__ ro, const float* __restrict__ rd,
                                                         const float* __restrict__ amin, const float* __restrict__ amax,
                                                         int64_t n, float* __restrict__ t_near, float* __restrict__ t_far,
                                                         uint8_t* __restrict__ hit) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float o[3], d[3], lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      o[a] = ro[3 * i + a]; d[a] = rd[3 * i + a];
      lo[a] = amin ? amin[3 * i + a] : -1.f; hi[a] = amax ? amax[3 * i + a] : 1.f;
    }
    const Slab sl = slab_test2(o, d, lo, hi);
    t_near[i] = sl.t_near; t_far[i] = sl.t_far; hit[i] = sl.hit ? 1 : 0;
  }
}

__global__ void __launch_bounds__(256) ray_box_bwd_kernel(const float* __restrict__ ro, const float* __restrict__ rd,
                                                         const float* __restrict__ amin, const float* __restrict__ amax,
                                                         int64_t n, const float* __restrict__ g_near,
                                                         const float* __restrict__ g_far, float* __restrict__ g_o,
                                                         float* __restrict__ g_d, float* __restrict__ g_min,
                                                         float* __restrict__ g_max) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float o[3], d[3], lo[3], hi[3], go[3], gd[3], glo[3], ghi[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      o[a] = ro[3 * i + a]; d[a] = rd[3 * i + a];
      lo[a] = amin ? amin[3 * i + a] : -1.f; hi[a] = amax ? amax[3 * i + a] : 1.f;
    }
    const Slab sl = slab_test2(o, d, lo, hi);
    slab_backward(sl, o, lo, hi, g_near[i], g_far[i], go, gd, glo, ghi);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      g_o[3 * i + a] = go[a]; g_d[3 * i + a] = gd[a];
      if (g_min) g_min[3 * i + a] = glo[a];
      if (g_max) g_max[3 * i + a] = ghi[a];
    }
  }
}

__global__ void __launch_bounds__(256) sample_box_bwd_kernel(
    const float* __restrict__ rays_o, const float* __restrict__ viewdir, const float* __restrict__ z_steps,
    const float* __restrict__ jitter, int64_t n_rays, int S, float half_diag, float hx, float hy, float hz,
    const float* __restrict__ g_xyz, const float* __restrict__ g_vrep, const float* __restrict__ g_zv,
    float* __restrict__ g_rays_o, float* __restrict__ g_viewdir,
    const int32_t* __restrict__ cpos, const int64_t* __restrict__ ccounts,   // non-NULL: g_xyz / g_vrep are in compact.cu's row order
    int detach_bounds) {   // renderer.render_rays_v3: the slab test ran on detached copies of the rays (renderer.py:425-432)
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float half[3] = {hx, hy, hz};
  const float fstep = (float)(1.0 / (double)S);
  for (int64_t ray = warp; ray < n_rays; ray += nwarps) {
    float o[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      o[a] = __fdiv_rn(__ldg(rays_o + 3 * ray + a), half_diag);
      d[a] = __ldg(viewdir + 3 * ray + a);
    }
    const Slab sl = slab_test(o, d, half);
    const float near = sl.hit ? sl.t_near : -1.f, far = sl.hit ? sl.t_far : -1.f;
    const float dn = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    float g[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // d o (3), d d (3), d |z|, d near, d far
    for (int k = lane; k < S; k += 32) {
      const int64_t idx = ray * S + k;
      // compacted gradients: S rows per hit ray; a miss ray's single row stands for all its samples and is credited to the last one
      int64_t gidx = idx;
      if (cpos != nullptr) gidx = sl.hit ? (int64_t)cpos[ray] * S + k : (k == S - 1 ? ccounts[0] * S + cpos[ray] : -1);
      fold_sample_grad((g_xyz && gidx >= 0) ? g_xyz + 3 * gidx : nullptr, (g_vrep && gidx >= 0) ? g_vrep + 3 * gidx : nullptr,
                       g_zv ? g_zv + idx : nullptr, __ldg(z_steps + k), __ldg(jitter + idx), fstep, near, far, d, dn, half_diag, g);
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) g[i] = warp_sum(g[i]);
    float gon[3] = {g[0], g[1], g[2]}, gd[3] = {g[3], g[4], g[5]};
    const float gzabs = g[6], gnear = g[7], gfar = g[8];
    if (lane == 0) {
      if (dn > 0.f) {
#pragma unroll
        for (int a = 0; a < 3; ++a) gd[a] += gzabs * half_diag * d[a] / dn;
      }
      if (sl.hit && !detach_bounds) {
        const float lo[3] = {-half[0], -half[1], -half[2]};
        float go2[3], gd2[3], glo[3], ghi[3];
        slab_backward(sl, o, lo, half, gnear, gfar, go2, gd2, glo, ghi);
#pragma unroll
        for (int a = 0; a < 3; ++a) { gon[a] += go2[a]; gd[a] += gd2[a]; }
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        g_rays_o[3 * ray + a] = gon[a] / half_diag;
        g_viewdir[3 * ray + a] = gd[a];
      }
    }
  }
}

__global__ void __launch_bounds__(256) sample_shell_fwd_kernel(
    const float* __restrict__ rays_o, const float* __restrict__ viewdir, const float* __restrict__ z, int64_t n_rays,
    int S, float obj_diag, int swap, float* __restrict__ xyz, float* __restrict__ vrep) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t ray = warp; ray < n_rays; ray += nwarps) {
    float o[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { o[a] = __ldg(rays_o + 3 * ray + a); d[a] = __ldg(viewdir + 3 * ray + a); }
    for (int k = lane; k < S; k += 32) {
      const float zk = __ldg(z + k);
      float x[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) x[a] = __fdiv_rn(__fadd_rn(o[a], __fmul_rn(d[a], zk)), obj_diag);
      const int64_t idx = ray * S + k;
      if (swap) {
        xyz[3 * idx] = -x[1]; xyz[3 * idx + 1] = x[0]; xyz[3 * idx + 2] = x[2];
        if (vrep) { vrep[3 * idx] = -d[1]; vrep[3 * idx + 1] = d[0]; vrep[3 * idx + 2] = d[2]; }
      } else {
        xyz[3 * idx] = x[0]; xyz[3 * idx + 1] = x[1]; xyz[3 * idx + 2] = x[2];
        if (vrep) { vrep[3 * idx] = d[0]; vrep[3 * idx + 1] = d[1]; vrep[3 * idx + 2] = d[2]; }
      }
    }
  }
}

__global__ void __launch_bounds__(256) sample_shell_bwd_kernel(
    const float* __restrict__ z, int64_t n_rays, int S, float obj_diag, int swap,
    const float* __restrict__ g_xyz, const float* __restrict__ g_vrep, float* __restrict__ g_rays_o,
    float* __restrict__ g_viewdir) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t ray = warp; ray < n_rays; ray += nwarps) {
    float go[3] = {0.f, 0.f, 0.f}, gd[3] = {0.f, 0.f, 0.f};
    for (int k = lane; k < S; k += 32) {
      const int64_t idx = ray * S + k;
      const float zk = __ldg(z + k);
      float gx[3] = {0.f, 0.f, 0.f}, gv[3] = {0.f, 0.f, 0.f};
      if (g_xyz) { gx[0] = __ldg(g_xyz + 3 * idx); gx[1] = __ldg(g_xyz + 3 * idx + 1); gx[2] = __ldg(g_xyz + 3 * idx + 2); }
      if (g_vrep) { gv[0] = __ldg(g_vrep + 3 * idx); gv[1] = __ldg(g_vrep + 3 * idx + 1); gv[2] = __ldg(g_vrep + 3 * idx + 2); }
      if (swap) {  // out = (-in_y, in_x, in_z)
        float t0 = gx[1], t1 = -gx[0]; gx[0] = t0; gx[1] = t1;
        t0 = gv[1]; t1 = -gv[0]; gv[0] = t0; gv[1] = t1;
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float g = gx[a] / obj_diag;
        go[a] += g; gd[a] += g * zk + gv[a];
      }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) { go[a] = warp_sum(go[a]); gd[a] = warp_sum(gd[a]); }
    if (lane == 0) {
#pragma unroll
      for (int a = 0; a < 3; ++a) { g_rays_o[3 * ray + a] = go[a]; g_viewdir[3 * ray + a] = gd[a]; }
    }
  }
}

}  // namespace snb

using namespace snb;

extern "C" int snb_get_rays_fwd(const float* px, const float* py, int64_t n_rays, const float* K, const float* c2w,
                                float* rays_o, float* viewdir, void* stream) {
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 256, 8);
  SNB_REQUIRE(grid > 0, "get_rays_fwd: no CUDA device");
  get_rays_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(px, py, n_rays, K, c2w, rays_o, viewdir);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_get_rays_bwd(const float* px, const float* py, int64_t n_rays, const float* K, const float* c2w,
                                const float* g_rays_o, const float* g_viewdir, float* g_c2w, void* stream) {
  if (n_rays == 0) return 0;
  const int grid = grid_1d(n_rays, 256 * 4, 1);
  SNB_REQUIRE(grid > 0, "get_rays_bwd: no CUDA device");
  get_rays_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(px, py, n_rays, K, c2w, g_rays_o, g_viewdir, g_c2w);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_ray_box_fwd(const float* ray_o, const float* ray_d, const float* aabb_min, const float* aabb_max,
                               int64_t n_rays, float* t_near, float* t_far, uint8_t* hit, void* stream) {
  SNB_REQUIRE((aabb_min == nullptr) == (aabb_max == nullptr), "ray_box_fwd: give both aabb corners or neither");
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 256, 8);
  SNB_REQUIRE(grid > 0, "ray_box_fwd: no CUDA device");
  ray_box_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ray_o, ray_d, aabb_min, aabb_max, n_rays, t_near, t_far, hit);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_ray_box_bwd(const float* ray_o, const float* ray_d, const float* aabb_min, const float* aabb_max,
                               int64_t n_rays, const float* g_near, const float* g_far, float* g_ray_o, float* g_ray_d,
                               float* g_aabb_min, float* g_aabb_max, void* stream) {
  SNB_REQUIRE((aabb_min == nullptr) == (aabb_max == nullptr), "ray_box_bwd: give both aabb corners or neither");
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 256, 8);
  SNB_REQUIRE(grid > 0, "ray_box_bwd: no CUDA device");
  ray_box_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ray_o, ray_d, aabb_min, aabb_max, n_rays, g_near, g_far,
                                                             g_ray_o, g_ray_d, g_aabb_min, g_aabb_max);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_sample_box_fwd(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter,
                                  int64_t n_rays, int32_t n_samples, float half_diag, const float* h,
                                  float* xyz, float* viewdir_rep, float* z_vals, uint8_t* hit, void* stream) {
  SNB_REQUIRE(n_samples >= 1 && h != nullptr, "sample_box_fwd: bad arguments");
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 8, 8);
  SNB_REQUIRE(grid > 0, "sample_box_fwd: no CUDA device");
  sample_box_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rays_o, viewdir, z_steps, jitter, n_rays, n_samples,
                                                                half_diag, h[0], h[1], h[2], xyz, viewdir_rep, z_vals, hit);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_sample_box_bwd(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter,
                                  int64_t n_rays, int32_t n_samples, float half_diag, const float* h,
                                  const float* g_xyz, const float* g_viewdir_rep, const float* g_z_vals,
                                  float* g_rays_o, float* g_viewdir, int32_t detach_bounds, void* stream) {
  SNB_REQUIRE(n_samples >= 1 && h != nullptr, "sample_box_bwd: bad arguments");
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 8, 8);
  SNB_REQUIRE(grid > 0, "sample_box_bwd: no CUDA device");
  sample_box_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rays_o, viewdir, z_steps, jitter, n_rays, n_samples,
                                                                half_diag, h[0], h[1], h[2], g_xyz, g_viewdir_rep, g_z_vals,
                                                                g_rays_o, g_viewdir, nullptr, nullptr, detach_bounds != 0);
  SNB_LAUNCH_CHECK();
  return 0;
}

// internal (fused render with miss-ray compaction): g_xyz / g_viewdir_rep hold the decoder's input gradients in compact.cu's row
// order (pos / counts from compact_plan); g_z_vals stays dense.  Replaces a scatter to dense + snb_sample_box_bwd.
namespace snb {
int sample_box_bwd_compact(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter, int64_t n_rays,
                           int32_t n_samples, float half_diag, const float* h, const float* g_xyz_c, const float* g_vrep_c,
                           const float* g_z_vals, const int32_t* pos, const int64_t* counts, float* g_rays_o, float* g_viewdir,
                           cudaStream_t st) {
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 8, 8);
  SNB_REQUIRE(grid > 0, "sample_box_bwd: no CUDA device");
  sample_box_bwd_kernel<<<grid, 256, 0, st>>>(rays_o, viewdir, z_steps, jitter, n_rays, n_samples, half_diag, h[0], h[1], h[2],
                                              g_xyz_c, g_vrep_c, g_z_vals, g_rays_o, g_viewdir, pos, counts, 0);
  SNB_LAUNCH_CHECK();
  return 0;
}
}  // namespace snb

extern "C" int snb_sample_shell_fwd(const float* rays_o, const float* viewdir, const float* z, int64_t n_rays,
                                    int32_t n_samples, float obj_diag, int32_t shapenet_swap,
                                    float* xyz, float* viewdir_rep, void* stream) {
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 8, 8);
  SNB_REQUIRE(grid > 0, "sample_shell_fwd: no CUDA device");
  sample_shell_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rays_o, viewdir, z, n_rays, n_samples, obj_diag,
                                                                  shapenet_swap, xyz, viewdir_rep);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_sample_shell_bwd(const float* z, int64_t n_rays, int32_t n_samples, float obj_diag, int32_t shapenet_swap,
                                    const float* g_xyz, const float* g_viewdir_rep,
                                    float* g_rays_o, float* g_viewdir, void* stream) {
  if (n_rays == 0) return 0;
  int grid = grid_1d(n_rays, 8, 8);
  SNB_REQUIRE(grid > 0, "sample_shell_bwd: no CUDA device");
  sample_shell_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(z, n_rays, n_samples, obj_diag, shapenet_swap, g_xyz,
                                                                  g_viewdir_rep, g_rays_o, g_viewdir);
  SNB_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// The per-ray stratified sampler on its own (renderer.py:27-41 = utils.sample_from_rays_v2, utils.py:170-184):
//   z[r][k] = near_r (1 - zs) + far_r zs,   zs = z_steps[k] + jitter[r][k] * (1 / S)        (rays (N, 8): near, far in columns 6, 7)
// Backward: g_near = sum_k g (1 - zs), g_far = sum_k g zs.  Inside prepare_sampled_rays the same arithmetic is fused into the box sampler.
// ---------------------------------------------------------------------------------------------------------------------
namespace snb {
__global__ void __launch_bounds__(256) stratified_z_fwd_kernel(const float* __restrict__ rays, int ld, const float* __restrict__ z_steps,
                                                             const float* __restrict__ jitter, int64_t n_rays, int S, float* __restrict__ z) {
  const float fstep = (float)(1.0 / (double)S);
  const int64_t total = n_rays * S;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / S;
    const int k = (int)(i - r * S);
    const float near = __ldg(rays + r * ld + ld - 2), far = __ldg(rays + r * ld + ld - 1);
    const float zs = __fadd_rn(__ldg(z_steps + k), __fmul_rn(__ldg(jitter + i), fstep));
    z[i] = __fadd_rn(__fmul_rn(near, __fsub_rn(1.f, zs)), __fmul_rn(far, zs));
  }
}
__global__ void __launch_bounds__(256) stratified_z_bwd_kernel(const float* __restrict__ z_steps, const float* __restrict__ jitter,
                                                             int64_t n_rays, int S, const float* __restrict__ g_z,
                                                             float* __restrict__ g_near, float* __restrict__ g_far) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float fstep = (float)(1.0 / (double)S);
  for (int64_t r = warp; r < n_rays; r += nwarps) {
    float a = 0.f, b = 0.f;
    for (int k = lane; k < S; k += 32) {
      const float zs = __fadd_rn(__ldg(z_steps + k), __fmul_rn(__ldg(jitter + r * S + k), fstep));
      const float g = __ldg(g_z + r * S + k);
      a += g * (1.f - zs);
      b += g * zs;
    }
    a = warp_sum(a); b = warp_sum(b);
    if (lane == 0) { g_near[r] = a; g_far[r] = b; }
  }
}
}  // namespace snb

extern "C" int snb_stratified_z_fwd(const float* rays, int32_t row_floats, const float* z_steps, const float* jitter, int64_t n_rays,
                                    int32_t n_samples, float* z, void* stream) {
  SNB_REQUIRE(n_rays >= 0 && n_samples >= 1 && row_floats >= 2, "stratified_z_fwd: bad arguments");
  if (n_rays == 0) return 0;
  SNB_REQUIRE(rays && z_steps && jitter && z, "stratified_z_fwd: null pointer");
  const int grid = grid_1d(n_rays * n_samples, 256, 16);
  SNB_REQUIRE(grid > 0, "stratified_z_fwd: no CUDA device");
  stratified_z_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rays, row_floats, z_steps, jitter, n_rays, n_samples, z);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_stratified_z_bwd(const float* z_steps, const float* jitter, int64_t n_rays, int32_t n_samples, const float* g_z,
                                    float* g_near, float* g_far, void* stream) {
  SNB_REQUIRE(n_rays >= 0 && n_samples >= 1, "stratified_z_bwd: bad arguments");
  if (n_rays == 0) return 0;
  SNB_REQUIRE(z_steps && jitter && g_z && g_near && g_far, "stratified_z_bwd: null pointer");
  int grid = grid_1d(n_rays, 8, 8);
  SNB_REQUIRE(grid > 0, "stratified_z_bwd: no CUDA device");
  stratified_z_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(z_steps, jitter, n_rays, n_samples, g_z, g_near, g_far);
  SNB_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Counter-based stratified jitter: u[r][k] = Philox4x32-10(counter = (ray id, k / 4), key = seed)[k % 4] in [0, 1).
// The reference draws the (N, S) jitter with ONE torch.rand_like on the device generator (renderer.py:39-40), whose stream
// cannot be sliced: a rank that renders a shard of the rays would have to draw all N x S numbers (33.5 M at config C4) to
// stay consistent with the other ranks.  A counter-based draw is a pure function of (seed, ray id, sample index): every rank
// fills ONLY its rows and the union over the ranks equals the one-GPU draw bit for bit.  (Not the reference's random stream:
// the tests that pin results to the reference feed the recorded jitter instead.)
// ---------------------------------------------------------------------------------------------------------------------
namespace snb {
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}

__global__ void __launch_bounds__(256) jitter_fill_kernel(uint64_t seed, const int64_t* __restrict__ ray_ids, int64_t n_rays, int n_samples,
                                                        float* __restrict__ out) {
  const int quads = (n_samples + 3) / 4;
  const int64_t total = n_rays * quads;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / quads;
    const int q = (int)(i - r * quads);
    const uint64_t id = ray_ids ? (uint64_t)ray_ids[r] : (uint64_t)r;
    const uint4 x = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)q, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float u[4] = {(float)(x.x >> 8) * 5.9604644775390625e-8f, (float)(x.y >> 8) * 5.9604644775390625e-8f,
                        (float)(x.z >> 8) * 5.9604644775390625e-8f, (float)(x.w >> 8) * 5.9604644775390625e-8f};
    float* dst = out + r * n_samples + 4 * q;
    if ((n_samples & 3) == 0) *reinterpret_cast<float4*>(dst) = make_float4(u[0], u[1], u[2], u[3]);
    else
      for (int j = 0; j < 4 && 4 * q + j < n_samples; ++j) dst[j] = u[j];
  }
}
}  // namespace snb

extern "C" int snb_jitter_fill(uint64_t seed, const int64_t* ray_ids, int64_t n_rays, int32_t n_samples, float* out, void* stream) {
  if (n_rays == 0) return 0;
  SNB_REQUIRE(n_rays > 0 && n_samples >= 1 && out, "jitter_fill: bad arguments");
  SNB_REQUIRE((n_samples & 3) != 0 || ((uintptr_t)out & 15) == 0, "jitter_fill: out must be 16-byte aligned");
  const int64_t total = n_rays * ((n_samples + 3) / 4);
  const int grid = grid_1d(total, 256, 16);
  SNB_REQUIRE(grid > 0, "jitter_fill: no CUDA device");
  jitter_fill_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(seed, ray_ids, n_rays, n_samples, out);
  SNB_LAUNCH_CHECK();
  return 0;
}
