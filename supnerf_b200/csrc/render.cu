// Fused render entry points: one C call enqueues the whole box-render of one object (rays -> slab test + stratified
// samples -> decoder -> compositing) on the caller's stream, and one call its backward.  Replaces the body of
// NeRFRenderer.render_rays between the target resize and the return (renderer.py:125-165) and its autograd backward.
// Every intermediate lives in ONE caller-provided workspace (no allocation, no synchronisation here), so a refine
// iteration costs two host calls per object instead of ~50 autograd-node launches.
#include "common.cuh"
#include "compact.h"
#include "decoder.h"
#include <stdlib.h>

using namespace snb;

namespace {

inline size_t al(size_t bytes) { return (bytes + 255) & ~size_t(255); }
// rows handed to the decoder as the host-side maximum: with compaction the real count is on the device and always a multiple
// of the 128-row tile, so any ray / sample count works; without it the bf16 decoder needs N * S to be a multiple of 128 itself
inline int64_t decoder_rows(snb_handle h, const snb_render_desc& d);

// Miss-ray compaction (compact.cu) applies to the box render on the tensor-core decoders: they take the device-side row count (the
// FFMA back end runs dense rows); SNB_NO_COMPACT=1 disables it.
bool use_compaction(snb_handle h, const snb_render_desc& d) {
  static const bool off = [] { const char* e = getenv("SNB_NO_COMPACT"); return e && atoi(e) != 0; }();
  if (off || d.mode != SNB_RENDER_BOX || d.n_rays <= 0) return false;
  Backend be;
  return select_backend(h, d.precision, &be) == nullptr && be != Backend::Ffma;
}

// forward workspace (kept for the backward): rays_o, viewdir (N,3) | xyz, vrep (M,3) | z_vals (M) | sigma (M) | rgb (M,3) | mlp ws
// | compaction: hit (N) u8, order, pos (N) i32, counts (4) i64, xyz_c, vrep_c (M+128,3), sigma_c (M+128), rgb_c (M+128,3)
struct FwdLayout {
  size_t rays_o, viewdir, xyz, vrep, z, sigma, rgb, mlp, total;
  size_t hit, order, pos, counts, xyz_c, vrep_c, sigma_c, rgb_c;
  FwdLayout(snb_handle h, const snb_render_desc& d) {
    const size_t N = (size_t)d.n_rays, M = N * (size_t)d.n_samples;
    size_t o = 0;
    hit = o; o += al(N);
    order = o; o += al(N * 4);
    pos = o; o += al(N * 4);
    counts = o; o += al(64);
    if (use_compaction(h, d)) {
      xyz_c = o; o += al((M + 128) * 12);
      vrep_c = o; o += al((M + 128) * 12);
      sigma_c = o; o += al((M + 128) * 4);
      rgb_c = o; o += al((M + 128) * 12);
    } else { xyz_c = vrep_c = sigma_c = rgb_c = 0; }
    rays_o = o; o += al(N * 12);
    viewdir = o; o += al(N * 12);
    xyz = o; o += al(M * 12);
    vrep = o; o += al(M * 12);
    z = o; o += al(M * 4);
    sigma = o; o += al(M * 4);
    rgb = o; o += al(M * 12);
    mlp = o; o += al(snb_mlp_workspace_bytes(h, decoder_rows(h, d), 1, d.precision));
    total = o;
  }
};

// backward scratch: g_sigma (M) | g_rgbs (M,3) | g_z (M) | g_xyz, g_vrep (M,3) | g_rays_o, g_viewdir (N,3) | mlp scratch
struct BwdLayout {
  size_t g_sigma, g_rgbs, g_z, g_xyz, g_vrep, g_rays_o, g_viewdir, mlp, total;
  size_t g_sigma_c, g_rgb_c, g_xyz_c, g_vrep_c;
  BwdLayout(snb_handle h, const snb_render_desc& d) {
    const size_t N = (size_t)d.n_rays, M = N * (size_t)d.n_samples;
    size_t o = 0;
    if (use_compaction(h, d)) {
      g_sigma_c = o; o += al((M + 128) * 4);
      g_rgb_c = o; o += al((M + 128) * 12);
      g_xyz_c = o; o += al((M + 128) * 12);
      g_vrep_c = o; o += al((M + 128) * 12);
    } else { g_sigma_c = g_rgb_c = g_xyz_c = g_vrep_c = 0; }
    g_sigma = o; o += al(M * 4);
    g_rgbs = o; o += al(M * 12);
    g_z = o; o += al(M * 4);
    g_xyz = o; o += al(M * 12);
    g_vrep = o; o += al(M * 12);
    g_rays_o = o; o += al(N * 12);
    g_viewdir = o; o += al(N * 12);
    mlp = o; o += al(snb_mlp_bwd_scratch_bytes(h, decoder_rows(h, d), 1, d.precision));
    total = o;
  }
};

inline int64_t decoder_rows(snb_handle h, const snb_render_desc& d) {
  const int64_t M = (int64_t)d.n_rays * d.n_samples;
  return use_compaction(h, d) ? (M + 127) / 128 * 128 : M;
}

int check_desc(snb_handle h, const snb_render_desc* d, const char* who) {
  SNB_REQUIRE(h != nullptr && d != nullptr, "%s: null handle or descriptor", who);
  SNB_REQUIRE(d->n_rays >= 0 && d->n_samples >= 1, "%s: bad sizes", who);
  SNB_REQUIRE(d->precision == SNB_PREC_FP32 || d->precision == SNB_PREC_BF16 || d->precision == SNB_PREC_BF16_TRAIN ||
              d->precision == SNB_PREC_FP32_TC, "%s: unknown precision %d", who, d->precision);
  SNB_REQUIRE(d->mode == SNB_RENDER_BOX || d->mode == SNB_RENDER_SHELL, "%s: unknown mode %d", who, d->mode);
  return 0;
}

inline float* F(void* base, size_t off) { return reinterpret_cast<float*>(static_cast<uint8_t*>(base) + off); }
inline const float* F(const void* base, size_t off) { return reinterpret_cast<const float*>(static_cast<const uint8_t*>(base) + off); }

}  // namespace

extern "C" size_t snb_render_workspace_bytes(snb_handle h, const snb_render_desc* d) {
  if (!h || !d || d->n_rays < 0 || d->n_samples < 1) return 0;
  return FwdLayout(h, *d).total + 256;
}

extern "C" size_t snb_render_bwd_scratch_bytes(snb_handle h, const snb_render_desc* d) {
  if (!h || !d || d->n_rays < 0 || d->n_samples < 1) return 0;
  return BwdLayout(h, *d).total + 256;
}

extern "C" int snb_render_fwd(snb_handle h, const snb_render_desc* d, const float* px, const float* py, const float* K,
                              const float* c2w, const float* z_steps, const float* jitter, const float* shape_latent,
                              const float* texture_latent, float* out_rgb, float* out_depth, float* out_acc, uint8_t* out_hit,
                              void* workspace, void* stream) {
  if (check_desc(h, d, "render_fwd")) return 2;
  if (d->n_rays == 0) return 0;
  const bool shell = d->mode == SNB_RENDER_SHELL;
  SNB_REQUIRE(px && py && K && c2w && z_steps && (jitter || shell) && shape_latent && texture_latent && out_rgb && out_depth &&
              out_acc && (out_hit || shell) && workspace, "render_fwd: null pointer");
  SNB_REQUIRE(((uintptr_t)workspace & 255) == 0, "render_fwd: workspace must be 256-byte aligned");
  const FwdLayout L(h, *d);
  const int64_t N = d->n_rays, M = N * d->n_samples;
  void* ws = workspace;
  if (snb_get_rays_fwd(px, py, N, K, c2w, F(ws, L.rays_o), F(ws, L.viewdir), stream)) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* wsb = static_cast<uint8_t*>(ws);
  if (shell) {   // utils.py stack: one shared z vector, no slab test
    if (snb_sample_shell_fwd(F(ws, L.rays_o), F(ws, L.viewdir), z_steps, N, d->n_samples, d->obj_diag, d->shapenet_swap,
                             F(ws, L.xyz), F(ws, L.vrep), stream)) return 1;
  } else {
    if (snb_sample_box_fwd(F(ws, L.rays_o), F(ws, L.viewdir), z_steps, jitter, N, d->n_samples, d->half_diag, d->aabb_half,
                           F(ws, L.xyz), F(ws, L.vrep), F(ws, L.z), wsb + L.hit, stream)) return 1;
    SNB_CHECK_CUDA(cudaMemcpyAsync(out_hit, wsb + L.hit, (size_t)N, cudaMemcpyDeviceToDevice, st));
  }
  if (use_compaction(h, *d)) {
    // decoder on the compacted rows only: S rows per hit ray + ONE row per miss ray (their S samples are one point)
    int32_t* order = reinterpret_cast<int32_t*>(wsb + L.order);
    int32_t* pos = reinterpret_cast<int32_t*>(wsb + L.pos);
    int64_t* counts = reinterpret_cast<int64_t*>(wsb + L.counts);
    if (compact_plan(wsb + L.hit, N, d->n_samples, order, pos, counts, st)) return 1;
    if (compact_gather(F(ws, L.xyz), F(ws, L.vrep), order, counts, N, d->n_samples, F(ws, L.xyz_c), F(ws, L.vrep_c), st)) return 1;
    if (decoder_forward(h, d->precision, F(ws, L.xyz_c), F(ws, L.vrep_c), decoder_rows(h, *d), 1, shape_latent, texture_latent,
                        F(ws, L.sigma_c), F(ws, L.rgb_c), wsb + L.mlp, st, {counts + 3})) return 1;
    if (compact_expand(F(ws, L.sigma_c), F(ws, L.rgb_c), wsb + L.hit, pos, counts, N, d->n_samples, F(ws, L.sigma), F(ws, L.rgb), st))
      return 1;
  } else if (snb_mlp_fwd(h, d->precision, F(ws, L.xyz), F(ws, L.vrep), M, 1, shape_latent, texture_latent, F(ws, L.sigma),
                         F(ws, L.rgb), wsb + L.mlp, stream)) return 1;
  return snb_composite_fwd(F(ws, L.sigma), F(ws, L.rgb), shell ? z_steps : F(ws, L.z), shell ? N : 1, N, d->n_samples, d->flags,
                           out_rgb, out_depth, out_acc, stream);
}

extern "C" int snb_render_bwd(snb_handle h, const snb_render_desc* d, const float* px, const float* py, const float* K,
                              const float* c2w, const float* z_steps, const float* jitter, const float* shape_latent,
                              const float* texture_latent, const void* workspace, const float* g_rgb, const float* g_depth,
                              const float* g_acc, void* scratch, float* g_c2w, float* g_shape_latent, float* g_texture_latent,
                              float* const* g_weights, void* stream) {
  if (check_desc(h, d, "render_bwd")) return 2;
  SNB_REQUIRE(g_shape_latent && g_texture_latent, "render_bwd: latent gradient outputs are required");
  cudaStream_t st = (cudaStream_t)stream;
  if (g_c2w) SNB_CHECK_CUDA(cudaMemsetAsync(g_c2w, 0, 12 * sizeof(float), st));
  if (d->n_rays == 0) return decoder_zero_grads(h, 1, g_shape_latent, g_texture_latent, g_weights, st);   // nothing rendered
  const bool shell = d->mode == SNB_RENDER_SHELL;
  SNB_REQUIRE(px && py && K && c2w && z_steps && (jitter || shell) && shape_latent && texture_latent && workspace && g_rgb &&
              g_depth && g_acc && scratch, "render_bwd: null pointer");
  SNB_REQUIRE((((uintptr_t)workspace | (uintptr_t)scratch) & 255) == 0, "render_bwd: workspace/scratch must be 256-byte aligned");
  const FwdLayout L(h, *d);
  const BwdLayout G(h, *d);
  const int64_t N = d->n_rays, M = N * d->n_samples;
  const void* ws = workspace;
  void* sc = scratch;
  const bool pose = g_c2w != nullptr;
  // shell mode: z is built from detached python floats (utils.py:468-469), it carries no gradient
  if (snb_composite_bwd(F(ws, L.sigma), F(ws, L.rgb), shell ? z_steps : F(ws, L.z), shell ? N : 1, N, d->n_samples, d->flags, g_rgb,
                        g_depth, g_acc, F(sc, G.g_sigma), F(sc, G.g_rgbs), (pose && !shell) ? F(sc, G.g_z) : nullptr, stream)) return 1;
  if (use_compaction(h, *d)) {
    const uint8_t* wsb = static_cast<const uint8_t*>(ws);
    const int32_t* order = reinterpret_cast<const int32_t*>(wsb + L.order);
    const int32_t* pos = reinterpret_cast<const int32_t*>(wsb + L.pos);
    const int64_t* counts = reinterpret_cast<const int64_t*>(wsb + L.counts);
    if (compact_reduce(F(sc, G.g_sigma), F(sc, G.g_rgbs), order, counts, N, d->n_samples, F(sc, G.g_sigma_c), F(sc, G.g_rgb_c), st)) return 1;
    if (decoder_backward(h, d->precision, F(ws, L.xyz_c), F(ws, L.vrep_c), decoder_rows(h, *d), 1, shape_latent, texture_latent,
                         F(ws, L.sigma_c), F(sc, G.g_sigma_c), F(sc, G.g_rgb_c), wsb + L.mlp, static_cast<uint8_t*>(sc) + G.mlp,
                         pose ? F(sc, G.g_xyz_c) : nullptr, pose ? F(sc, G.g_vrep_c) : nullptr, g_shape_latent, g_texture_latent, g_weights,
                         st, {counts + 3})) return 1;
    if (!pose) return 0;
    if (sample_box_bwd_compact(F(ws, L.rays_o), F(ws, L.viewdir), z_steps, jitter, N, d->n_samples, d->half_diag, d->aabb_half,
                               F(sc, G.g_xyz_c), F(sc, G.g_vrep_c), F(sc, G.g_z), pos, counts, F(sc, G.g_rays_o), F(sc, G.g_viewdir), st))
      return 1;
    return snb_get_rays_bwd(px, py, N, K, c2w, F(sc, G.g_rays_o), F(sc, G.g_viewdir), g_c2w, stream);
  } else if (snb_mlp_bwd(h, d->precision, F(ws, L.xyz), F(ws, L.vrep), M, 1, shape_latent, texture_latent, F(ws, L.sigma),
                  F(sc, G.g_sigma), F(sc, G.g_rgbs), static_cast<const uint8_t*>(ws) + L.mlp, static_cast<uint8_t*>(sc) + G.mlp,
                  pose ? F(sc, G.g_xyz) : nullptr, pose ? F(sc, G.g_vrep) : nullptr, g_shape_latent, g_texture_latent, g_weights,
                  stream)) return 1;
  if (!pose) return 0;
  if (shell) {
    if (snb_sample_shell_bwd(z_steps, N, d->n_samples, d->obj_diag, d->shapenet_swap, F(sc, G.g_xyz), F(sc, G.g_vrep),
                             F(sc, G.g_rays_o), F(sc, G.g_viewdir), stream)) return 1;
  } else if (snb_sample_box_bwd(F(ws, L.rays_o), F(ws, L.viewdir), z_steps, jitter, N, d->n_samples, d->half_diag, d->aabb_half,
                                F(sc, G.g_xyz), F(sc, G.g_vrep), F(sc, G.g_z), F(sc, G.g_rays_o), F(sc, G.g_viewdir), 0, stream)) return 1;
  return snb_get_rays_bwd(px, py, N, K, c2w, F(sc, G.g_rays_o), F(sc, G.g_viewdir), g_c2w, stream);
}
