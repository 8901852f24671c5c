// Device helpers of the ray / box-sampler kernels (sampler.cu), shared with the batched render (render_batch.cu): each is the one
// copy of its arithmetic, so the per-object and the batched paths compute the same bits.
#pragma once
#include "common.cuh"
#include <math.h>

namespace snb {

// torch.minimum/maximum propagate NaN (utils.py:308-312).
__device__ __forceinline__ float nan_min(float a, float b) { return (a != a || b != b) ? NAN : fminf(a, b); }
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a || b != b) ? NAN : fmaxf(a, b); }

struct Slab {
  float t_near, t_far;
  bool hit;
  float tmin[3], tmax[3], inv[3];
};

// utils.py:303-319 in the reference's op order: reciprocal; (aabb - o) * inv; min/max; two compares.
__device__ __forceinline__ Slab slab_test2(const float o[3], const float d[3], const float lo[3], const float hi[3]) {
  Slab r;
  float t0[3], t1[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    r.inv[a] = __frcp_rn(d[a]);
    r.tmin[a] = __fmul_rn(__fsub_rn(lo[a], o[a]), r.inv[a]);
    r.tmax[a] = __fmul_rn(__fsub_rn(hi[a], o[a]), r.inv[a]);
    t0[a] = nan_min(r.tmin[a], r.tmax[a]);
    t1[a] = nan_max(r.tmin[a], r.tmax[a]);
  }
  r.t_near = nan_max(nan_max(t0[0], t0[1]), t0[2]);
  r.t_far = nan_min(nan_min(t1[0], t1[1]), t1[2]);
  bool inside = r.t_far > r.t_near;
  float m = inside ? 1.f : 0.f;
  r.hit = inside && (__fmul_rn(r.t_far, m) > 0.f);
  return r;
}

__device__ __forceinline__ Slab slab_test(const float o[3], const float d[3], const float half[3]) {
  const float lo[3] = {-half[0], -half[1], -half[2]};
  return slab_test2(o, d, lo, half);
}

// torch.maximum / torch.minimum backward: the selected operand gets the gradient, ties split it.
__device__ __forceinline__ void pick_max(float a, float b, float g, float& ga, float& gb) {
  if (a == b) { ga = 0.5f * g; gb = 0.5f * g; }
  else if (a > b) { ga = g; gb = 0.f; }
  else { ga = 0.f; gb = g; }
}
__device__ __forceinline__ void pick_min(float a, float b, float g, float& ga, float& gb) {
  if (a == b) { ga = 0.5f * g; gb = 0.5f * g; }
  else if (a < b) { ga = g; gb = 0.f; }
  else { ga = 0.f; gb = g; }
}

// gradients of (t_near, t_far) w.r.t. origin, direction and the two box corners, per axis
__device__ __forceinline__ void slab_backward(const Slab& sl, const float o[3], const float lo[3], const float hi[3],
                                              float gnear, float gfar, float go[3], float gd[3], float glo[3], float ghi[3]) {
  float t0[3], t1[3], g0[3], g1[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) { t0[a] = nan_min(sl.tmin[a], sl.tmax[a]); t1[a] = nan_max(sl.tmin[a], sl.tmax[a]); }
  float gxy, gz_;
  pick_max(nan_max(t0[0], t0[1]), t0[2], gnear, gxy, gz_);
  g0[2] = gz_;
  pick_max(t0[0], t0[1], gxy, g0[0], g0[1]);
  pick_min(nan_min(t1[0], t1[1]), t1[2], gfar, gxy, gz_);
  g1[2] = gz_;
  pick_min(t1[0], t1[1], gxy, g1[0], g1[1]);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float gmin_a, gmax_a, ga, gb;
    pick_min(sl.tmin[a], sl.tmax[a], g0[a], gmin_a, gmax_a);  // t0 = min(tmin, tmax)
    pick_max(sl.tmin[a], sl.tmax[a], g1[a], ga, gb);          // t1 = max(tmin, tmax)
    gmin_a += ga; gmax_a += gb;
    // tmin = (lo - o) * inv ; tmax = (hi - o) * inv ; inv = 1/d
    go[a] = -(gmin_a + gmax_a) * sl.inv[a];
    glo[a] = gmin_a * sl.inv[a];
    ghi[a] = gmax_a * sl.inv[a];
    const float ginv = gmin_a * (lo[a] - o[a]) + gmax_a * (hi[a] - o[a]);
    gd[a] = -ginv * sl.inv[a] * sl.inv[a];
  }
}

// utils.get_rays for one pixel: dirs = ((px - cx) / fx, (py - cy) / fy, 1); rays_d = sum(dirs * R, -1); viewdir = rays_d / |rays_d|,
// as separate round-to-nearest fp32 ops.  K (3,3) and c2w (3,4) row-major; the caller forms the origin.
__device__ __forceinline__ void pixel_dir(const float* __restrict__ K, const float* __restrict__ c2w, float px, float py, float d[3]) {
  const float cx = __ldg(K + 2), cy = __ldg(K + 5), fx = __ldg(K), fy = __ldg(K + 4);
  const float p0 = __fdiv_rn(__fsub_rn(px, cx), fx), p1 = __fdiv_rn(__fsub_rn(py, cy), fy), p2 = 1.f;
  float r[3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
    r[a] = __fadd_rn(__fadd_rn(__fmul_rn(p0, __ldg(c2w + 4 * a)), __fmul_rn(p1, __ldg(c2w + 4 * a + 1))), __fmul_rn(p2, __ldg(c2w + 4 * a + 2)));
  const float nrm = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(r[0], r[0]), __fmul_rn(r[1], r[1])), __fmul_rn(r[2], r[2])));
#pragma unroll
  for (int a = 0; a < 3; ++a) d[a] = __fdiv_rn(r[a], nrm);
}

// Backward of the box sampler for one sample k of a ray (o, d, near, far):
//   zs = z_steps[k] + jitter[k] / S;  z = near (1 - zs) + far zs;  xyz = o + z d;  z_vals = |z d| * half_diag
// g_x, g_v, g_z point at the sample's d xyz (3), d viewdir (3) and d z_vals, or are NULL where those are zero.  Adds the sample's
// share to g = {d o (3), d d (3, without the |z d| term), d |z| (the |z d| term's factor), d near, d far}; dn = |d|.
__device__ __forceinline__ void fold_sample_grad(const float* __restrict__ g_x, const float* __restrict__ g_v, const float* __restrict__ g_z,
                                                 float z_step, float jit, float fstep, float near, float far, const float d[3], float dn,
                                                 float half_diag, float g[9]) {
  const float zs = __fadd_rn(z_step, __fmul_rn(jit, fstep));
  const float zc = __fadd_rn(__fmul_rn(near, __fsub_rn(1.f, zs)), __fmul_rn(far, zs));
  float gx[3] = {0.f, 0.f, 0.f};
  if (g_x != nullptr) { gx[0] = __ldg(g_x); gx[1] = __ldg(g_x + 1); gx[2] = __ldg(g_x + 2); }
  float gz = gx[0] * d[0] + gx[1] * d[1] + gx[2] * d[2];
#pragma unroll
  for (int a = 0; a < 3; ++a) { g[a] += gx[a]; g[3 + a] += zc * gx[a]; }
  if (g_v != nullptr) { g[3] += __ldg(g_v); g[4] += __ldg(g_v + 1); g[5] += __ldg(g_v + 2); }
  if (g_z != nullptr) {
    const float gv = __ldg(g_z);
    const float sgn = (zc > 0.f) ? 1.f : ((zc < 0.f) ? -1.f : 0.f);
    gz += gv * sgn * dn * half_diag;
    g[6] += gv * fabsf(zc);
  }
  g[7] += gz * (1.f - zs);
  g[8] += gz * zs;
}

// Backward of get_rays' direction for one pixel: r = R p, p = ((px - cx) / fx, (py - cy) / fy, 1), d = r / |r|.
// g_r = (g_d - d (g_d . d)) / |r|; the pose gets d c2w[a][j < 3] = g_r[a] p[j], which the caller accumulates in its own precision.
__device__ __forceinline__ void dir_grad_to_pose(const float* __restrict__ K, const float* __restrict__ c2w, float px, float py,
                                                 const float g_d[3], float pp[3], float g_r[3]) {
  const float cx = __ldg(K + 2), cy = __ldg(K + 5), fx = __ldg(K), fy = __ldg(K + 4);
  pp[0] = (px - cx) / fx; pp[1] = (py - cy) / fy; pp[2] = 1.f;
  float r[3], d[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) r[a] = pp[0] * __ldg(c2w + 4 * a) + pp[1] * __ldg(c2w + 4 * a + 1) + pp[2] * __ldg(c2w + 4 * a + 2);
  const float inv = 1.f / sqrtf(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
#pragma unroll
  for (int a = 0; a < 3; ++a) d[a] = r[a] * inv;
  const float dot = g_d[0] * d[0] + g_d[1] * d[1] + g_d[2] * d[2];
#pragma unroll
  for (int a = 0; a < 3; ++a) g_r[a] = (g_d[a] - d[a] * dot) * inv;
}

}  // namespace snb
