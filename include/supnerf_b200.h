/* supnerf_b200 — C ABI of the B200-native SUP-NeRF object-centric render hot path.
 *
 * The reference (abhi1kumar/SUP-NeRF) has no FFI: its boundary is the Python call API of
 * src/renderer.py, src/utils.py:94-672 and src/model_{codenerf,autorf,supnerf}.py.  These entry
 * points are what a ctypes binding for that path binds (INTEGRATION.md shows the stub); each one
 * cites the reference function it replaces.  Conventions:
 *   - every pointer is a DEVICE pointer to fp32 row-major data unless stated; borrowed for the call;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no call synchronises;
 *   - return 0 on success, non-zero on error; snb_last_error() gives the message (thread-local);
 *   - no global mutable state besides the per-handle weight tables; one handle per (device, model).
 * There is NO CPU fallback: without a CUDA device every compute call returns an error.
 */
#ifndef SUPNERF_B200_H
#define SUPNERF_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SNB_ABI_VERSION 2

/* flags for the compositing kernels */
#define SNB_WHITE_BKGD 1 /* renderer.py:60-63 */
#define SNB_SIGMA_RELU 2 /* renderer.py:52; cleared only for utils.volume_rendering (utils.py:191) */

/* decoder families */
#define SNB_ARCH_CODENERF 0 /* CodeNeRF / AutoRFMix / SUPNeRF decoder: model_codenerf.py:39-63 */
#define SNB_ARCH_AUTORF 1   /* AutoRF decoder: model_autorf.py:156-186 */

/* MLP arithmetic */
#define SNB_PREC_FP32 0 /* SIMT FFMA, fp32 everywhere: the 1e-5 parity mode */
#define SNB_PREC_BF16 1 /* tcgen05 bf16 x bf16 -> fp32 TMEM accumulators: the 2e-2 throughput mode (weights frozen) */
#define SNB_PREC_BF16_TRAIN 2 /* the same arithmetic; the forward/backward additionally keep every layer's operand tiles in the
                                 workspace / scratch so that snb_mlp_bwd can produce all weight gradients on the tensor core */
#define SNB_PREC_FP32_TC 3 /* the 1e-5 parity mode on the tensor cores (weights frozen; CodeNeRF family, W = 128 or 256): every MMA operand
                              is held as two fp16 parts (x = hi + lo) and every product issued as three tcgen05 MMAs into fp32 TMEM
                              accumulators; biases, latent layers, heads and reductions stay fp32 FFMA.  Errors against the fp64
                              oracle on par with SNB_PREC_FP32; valid for |weight| < 255 and |activation| < 65504 (beyond: inf / NaN).
                              Row constraints as SNB_PREC_BF16 (rows per object a multiple of 128).  Workspace / scratch sizes as
                              SNB_PREC_BF16; needs snb_pack_weights. */

typedef struct snb_handle_s* snb_handle;

typedef struct {
  int32_t arch;           /* SNB_ARCH_* */
  int32_t shape_blocks;   /* ctor arg of the same name */
  int32_t texture_blocks; /* ctor arg of the same name */
  int32_t W;              /* hidden width (CodeNeRF: W; AutoRFMix/SUPNeRF/AutoRF: latent_dim) */
  int32_t latent_dim;
  int32_t num_xyz_freq;   /* 10 */
  int32_t num_dir_freq;   /* 4 */
} snb_arch;

int snb_abi_version(void);
const char* snb_last_error(void);
/* Number of kernels this library has launched in this process (bench.py reports it as gpu_launches). */
uint64_t snb_launch_count(void);
/* Number of SMs etc. of the current device; fails without a GPU. */
int snb_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K3 / K3b: alpha compositing -------------------------------------------------------------
 * Replaces NeRFRenderer.volume_render (renderer.py:43-65), volume_rendering3 (renderer.py:355-379),
 * utils.volume_rendering2 (utils.py:202-217), utils.volume_rendering_batch (utils.py:220-233) and
 * utils.volume_rendering (utils.py:187-199).
 * sigma (N,S); rgb (N,S,3); z: row r(i) = i / rays_per_zrow, i.e. rays_per_zrow = 1 for per-ray
 * z_vals (N,S), = N for one shared vector (S,), = n for (B,S) against (B,n,S).
 * out_rgb (N,3), out_depth (N), out_acc (N) (transmittance before the last sample). */
int snb_composite_fwd(const float* sigma, const float* rgb, const float* z, int64_t rays_per_zrow,
                      int64_t n_rays, int32_t n_samples, int32_t flags,
                      float* out_rgb, float* out_depth, float* out_acc, void* stream);
/* Backward of the above (autograd of renderer.py:50-65).  g_z is per ray (N,S) whatever the z
 * layout (the caller reduces it for shared rows); g_z may be NULL. */
int snb_composite_bwd(const float* sigma, const float* rgb, const float* z, int64_t rays_per_zrow,
                      int64_t n_rays, int32_t n_samples, int32_t flags,
                      const float* g_rgb, const float* g_depth, const float* g_acc,
                      float* g_sigma, float* g_rgbs, float* g_z, void* stream);

/* ---- K1 / K1b: ray generation, slab test, stratified sampling ----------------------------------
 * snb_get_rays: utils.get_rays / get_rays_specified (utils.py:107-151).  px,py (N) pixel coords
 * (fp32, as produced by torch.linspace); K (3,3) and c2w (3,4) on the device.
 * Backward gives g_c2w (12 floats, ACCUMULATED with atomics: zero it first). */
int snb_get_rays_fwd(const float* px, const float* py, int64_t n_rays, const float* K, const float* c2w,
                     float* rays_o, float* viewdir, void* stream);
int snb_get_rays_bwd(const float* px, const float* py, int64_t n_rays, const float* K, const float* c2w,
                     const float* g_rays_o, const float* g_viewdir, float* g_c2w, void* stream);
/* snb_ray_box: the slab test alone — utils.ray_box_intersection_tensor (utils.py:283-327) and its
 * numpy twin ray_box_intersection (utils.py:236-280).  aabb_min/aabb_max are per-ray (N,3) or both
 * NULL for the unit box.  Outputs are UNCOMPACTED: t_near (N), t_far (N), hit (N) uint8; the
 * reference's `t_near[hit]` compaction is the caller's.  Backward: gradients of the uncompacted
 * t_near/t_far to ray_o, ray_d (and, if non-NULL, aabb_min/aabb_max), ties split as torch does. */
int snb_ray_box_fwd(const float* ray_o, const float* ray_d, const float* aabb_min, const float* aabb_max,
                    int64_t n_rays, float* t_near, float* t_far, uint8_t* hit, void* stream);
int snb_ray_box_bwd(const float* ray_o, const float* ray_d, const float* aabb_min, const float* aabb_max,
                    int64_t n_rays, const float* g_near, const float* g_far,
                    float* g_ray_o, float* g_ray_d, float* g_aabb_min, float* g_aabb_max, void* stream);
/* snb_sample_box: NeRFRenderer.prepare_sampled_rays (renderer.py:91-115) incl. the slab test
 * ray_box_intersection_tensor (utils.py:283-327) and sample_from_ray (renderer.py:27-41).
 * half_diag = diag/2 and aabb_half = (l,w,h)/diag are the reference's host-rounded float32s.
 * z_steps (S) = torch.linspace(0, 1-1/S, S) (renderer.py:38, kept as an input so its fp32 rounding
 * is the reference's); jitter (N,S) = the torch.rand_like draw (renderer.py:40).  Outputs: xyz (N,S,3), viewdir_rep (N,S,3, nullable),
 * z_vals (N,S), hit (N) uint8 — bit-exact with the reference's bool mask. */
int snb_sample_box_fwd(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter,
                       int64_t n_rays, int32_t n_samples, float half_diag, const float* aabb_half_host3,
                       float* xyz, float* viewdir_rep, float* z_vals, uint8_t* hit, void* stream);
int snb_sample_box_bwd(const float* rays_o, const float* viewdir, const float* z_steps, const float* jitter,
                       int64_t n_rays, int32_t n_samples, float half_diag, const float* aabb_half_host3,
                       const float* g_xyz, const float* g_viewdir_rep, const float* g_z_vals,
                       float* g_rays_o, float* g_viewdir, int32_t detach_bounds, void* stream);
/* snb_sample_shell: utils.sample_from_rays (utils.py:154-167) + `xyz /= obj_diag` (utils.py:472) +
 * the shapenet axis swap (utils.py:491-495).  z (S) is the shared sample vector (built on the host
 * exactly as the reference does).  inv_scale = 1 for a plain sample_from_rays. */
/* The per-ray stratified sampler on its own (renderer.py:27-41 = utils.sample_from_rays_v2, utils.py:170-184): rays (N, row_floats)
 * with near / far in the last two columns, z_steps (S), jitter (N,S) -> z (N,S) = near (1 - zs) + far zs, zs = z_steps + jitter / S.
 * Backward: g_z (N,S) -> g_near (N), g_far (N).  snb_sample_box_bwd's detach_bounds != 0: near / far carry no gradient (the slab
 * test ran on detached rays: renderer.render_rays_v3, renderer.py:425-432). */
int snb_stratified_z_fwd(const float* rays, int32_t row_floats, const float* z_steps, const float* jitter, int64_t n_rays,
                         int32_t n_samples, float* z, void* stream);
int snb_stratified_z_bwd(const float* z_steps, const float* jitter, int64_t n_rays, int32_t n_samples, const float* g_z,
                         float* g_near, float* g_far, void* stream);
int snb_sample_shell_fwd(const float* rays_o, const float* viewdir, const float* z, int64_t n_rays,
                         int32_t n_samples, float obj_diag, int32_t shapenet_swap,
                         float* xyz, float* viewdir_rep, void* stream);
int snb_sample_shell_bwd(const float* z, int64_t n_rays, int32_t n_samples, float obj_diag, int32_t shapenet_swap,
                         const float* g_xyz, const float* g_viewdir_rep,
                         float* g_rays_o, float* g_viewdir, void* stream);

/* Counter-based stratified jitter for the ray-sharded mode (no reference counterpart: the reference draws the (N, S) jitter
 * with one torch.rand_like, renderer.py:39-40, which a rank rendering a shard of the rays cannot slice without drawing all of
 * it).  out[r][k] = Philox4x32-10(counter = (ray id, k / 4), key = seed)[k % 4] * 2^-24 in [0, 1): a pure function of
 * (seed, ray id, k), so the union of the shards equals the one-GPU fill bit for bit.  ray_ids NULL = rays 0 .. n_rays-1. */
int snb_jitter_fill(uint64_t seed, const int64_t* ray_ids, int64_t n_rays, int32_t n_samples, float* out, void* stream);

/* ---- K2 / K2b: positional encoding + latent-conditioned decoder MLP -----------------------------
 * Replaces CodeNeRF.forward (model_codenerf.py:39-63) ≡ AutoRFMix.forward (model_autorf.py:226-250)
 * ≡ SUPNeRF.forward (model_supnerf.py:241-269), and AutoRF.forward (model_autorf.py:156-186).
 * Weight ABI = the reference's state_dict order restricted to the decoder (see DESIGN.md):
 *   CODENERF: encoding_xyz.0, [shape_latent_layer_j.0, shape_layer_j.0]_{j=1..Bs}, encoding_shape,
 *             sigma.0, encoding_viewdir.0, [texture_latent_layer_j.0, texture_layer_j.0]_{j=1..Bt},
 *             rgb.0, rgb.2 — each as (weight (out,in) row-major, bias).
 *   AUTORF:   encoding_xyz.0, shape_layer_{0..Bs-2}.0, sigma.0, texture_layer_{0..Bt-2}.0, rgb.0.
 * snb_set_weights borrows the fp32 device pointers (2 per layer); they must stay valid until the
 * next snb_set_weights / snb_destroy. */
int snb_create(snb_handle* out, const snb_arch* arch);
int snb_destroy(snb_handle h);
int snb_num_weight_tensors(snb_handle h);
int snb_layer_shape(snb_handle h, int32_t layer, int32_t* out_dim, int32_t* in_dim);
int snb_set_weights(snb_handle h, const float* const* tensors, int32_t n_tensors);
/* bf16 mode only: re-tile the fp32 weights into the bf16 shared-memory images the tcgen05 kernels
 * stream with bulk copies.  packed must hold snb_packed_bytes(h).  Call again after weights change. */
size_t snb_packed_bytes(snb_handle h);
/* The four hooks below are PER HANDLE (no process-global state): they affect only calls made through `h`.
 * Test hook: when non-NULL, the next bf16 forwards also dump every step's post-epilogue fp32 activations to
 * acts [n_steps][n_rows][256] (n_steps = shape_blocks + texture_blocks + 4).  Pass NULL to switch it off. */
int snb_tc_set_debug(snb_handle h, float* acts);
/* Tuning hook: when non-NULL (device memory, >= 8 B x 4 x 2 x steps x tile pairs of CTA 0), CTA 0 of the next bf16 decoder
 * kernels writes clock64 stamps [pair][step][slot][4] = {operand-ready seen by the MMA warp, MMAs issued, accumulator-ready
 * seen by the epilogue, epilogue published}.  tools/trace_pipeline.py prints the timeline.  Pass NULL to switch it off. */
int snb_tc_set_trace(snb_handle h, long long* stamps);
/* Test / tuning hook: which two-tile decoder kernels frozen-weight calls use.  1: the cta_group::2 kernels (one M = 256 MMA over
 * the CTA pair, half of every weight stage per SM) wherever they apply (every object owns a multiple of 256 rows); 0: always the
 * cta_group::1 kernels; -1 (initial state): the SNB_TC_CG2 environment variable, default 1.  Both give the same arithmetic. */
int snb_tc_set_cg2(snb_handle h, int32_t mode);
/* Measurement hook (bench.py roofline): while enabled, every bf16 decoder call records a CUDA-event pair on its
 * launch stream around the tcgen05 kernel alone.  snb_kernel_timing_read (after a synchronize) copies up to max_n
 * durations in ms to HOST memory and returns how many; which = 0 forward, 1 backward.  Enabling clears old events. */
int snb_kernel_timing_enable(snb_handle h, int32_t on);
int snb_kernel_timing_read(snb_handle h, int32_t which, float* ms_host, int32_t max_n);
int snb_pack_weights(snb_handle h, void* packed, void* stream);
/* Scratch the forward needs (and the backward re-reads): activations in fp32 mode, ReLU masks +
 * per-sample sigma/rgb in bf16 mode.  n_rows = N*S samples. */
size_t snb_mlp_workspace_bytes(snb_handle h, int64_t n_rows, int64_t n_objs, int32_t precision);
/* xyz, viewdir (n_rows,3); latents (n_objs, latent_dim); object b owns rows
 * [b*n_rows/n_objs, (b+1)*n_rows/n_objs).  sigma (n_rows), rgb (n_rows,3). */
int snb_mlp_fwd(snb_handle h, int32_t precision, const float* xyz, const float* viewdir, int64_t n_rows,
                int64_t n_objs, const float* shape_latent, const float* texture_latent,
                float* sigma, float* rgb, void* workspace, void* stream);
/* g_xyz / g_viewdir (n_rows,3) may be NULL (no pose gradient wanted).  g_weights: NULL, or
 * snb_num_weight_tensors device pointers that receive (are overwritten with) the weight grads.
 * scratch: snb_mlp_bwd_scratch_bytes. */
size_t snb_mlp_bwd_scratch_bytes(snb_handle h, int64_t n_rows, int64_t n_objs, int32_t precision);
int snb_mlp_bwd(snb_handle h, int32_t precision, const float* xyz, const float* viewdir, int64_t n_rows,
                int64_t n_objs, const float* shape_latent, const float* texture_latent,
                const float* sigma, const float* g_sigma, const float* g_rgb, const void* workspace,
                void* scratch, float* g_xyz, float* g_viewdir, float* g_shape_latent,
                float* g_texture_latent, float* const* g_weights, void* stream);

/* ---- fused render: rays -> slab test + stratified samples -> decoder -> compositing, one object per call ----------
 * Replaces the body of NeRFRenderer.render_rays / render_rays_specified between the target resize and the return
 * (renderer.py:125-165, :178-199: get_rays -> prepare_sampled_rays -> model(...) -> volume_render) and, for
 * snb_render_bwd, the autograd backward of that chain (optimizer_nuscenes.py:737 `loss.backward()`).
 * Same operands as the stage calls above (px, py, K, c2w, z_steps, jitter; latents (1, latent_dim)).  All
 * intermediates live in `workspace` (snb_render_workspace_bytes, 256-byte aligned, kept by the caller until the
 * backward has run) and `scratch` (snb_render_bwd_scratch_bytes).  Outputs: out_rgb (N,3), out_depth (N), out_acc (N),
 * out_hit (N) uint8.  Backward: g_c2w (12 floats, overwritten; NULL = no pose gradient, which also skips the d xyz /
 * d viewdir part of the decoder backward), g_shape_latent / g_texture_latent (latent_dim each, overwritten),
 * g_weights as in snb_mlp_bwd (NULL = frozen weights). */
typedef struct {
  int64_t n_rays;
  int32_t n_samples;
  int32_t precision;  /* SNB_PREC_* */
  int32_t flags;      /* SNB_WHITE_BKGD | SNB_SIGMA_RELU */
  float half_diag;    /* diag / 2, the reference's host-rounded float32 (renderer.py:92) */
  float aabb_half[3]; /* (l, w, h) / diag (renderer.py:97-100) */
  int32_t mode;       /* SNB_RENDER_BOX: the renderer.py stack above.  SNB_RENDER_SHELL: the utils.py stack every refine loop
                         calls (utils.render_rays_v2 utils.py:435-502, render_rays :380-432, render_rays_specified :504-551):
                         z_steps then holds the SHARED sample vector z (S) built by the caller as utils.sample_from_rays does
                         (utils.py:154-167), jitter is unused (may be NULL), compositing is utils.volume_rendering2 (shared z) */
  float obj_diag;     /* shell mode: xyz /= obj_diag (utils.py:472) */
  int32_t shapenet_swap; /* shell mode: (x,y,z) -> (-y,x,z) of xyz and viewdir (utils.py:491-495) */
} snb_render_desc;
#define SNB_RENDER_BOX 0
#define SNB_RENDER_SHELL 1
size_t snb_render_workspace_bytes(snb_handle h, const snb_render_desc* d);
size_t snb_render_bwd_scratch_bytes(snb_handle h, const snb_render_desc* d);
int snb_render_fwd(snb_handle h, const snb_render_desc* d, const float* px, const float* py, const float* K,
                   const float* c2w, const float* z_steps, const float* jitter, const float* shape_latent,
                   const float* texture_latent, float* out_rgb, float* out_depth, float* out_acc, uint8_t* out_hit,
                   void* workspace, void* stream);
int snb_render_bwd(snb_handle h, const snb_render_desc* d, const float* px, const float* py, const float* K,
                   const float* c2w, const float* z_steps, const float* jitter, const float* shape_latent,
                   const float* texture_latent, const void* workspace, const float* g_rgb, const float* g_depth,
                   const float* g_acc, void* scratch, float* g_c2w, float* g_shape_latent, float* g_texture_latent,
                   float* const* g_weights, void* stream);

/* ---- batched fused box render: ONE launch set for n_objs objects -----------------------------------------------------
 * The loops that call NeRFRenderer.render_rays once per object (optimizer_nuscenes.py:716-726 over the objects of a scene;
 * configs[1]: 16 objects per step) become two C calls for the whole batch.  Same arithmetic per object as snb_render_fwd / bwd
 * in SNB_RENDER_BOX mode with miss-ray compaction; frozen weights, bf16 decoder.  Every object brings rays_per_obj rays.
 *   px, py (B,N) pixel coordinates; K (B,3,3); c2w (B,3,4); box (B,4) = {diag/2, l/diag, w/diag, h/diag} per object
 *   (renderer.py:92-100, rounded to float32 on the host as the reference does); z_steps (S); jitter (B,N,S);
 *   shape_latent / texture_latent (B,D).  Outputs rgb (B,N,3), depth (B,N), acc (B,N), hit (B,N; may be NULL).
 *   workspace: snb_render_batch_workspace_bytes, 256-byte aligned, kept until the backward; scratch likewise.
 *   Backward: g_rgb (B,N,3), g_depth / g_acc (B,N; NULL = zero) -> g_c2w (B,3,4; NULL = not wanted), g_shape_latent,
 *   g_texture_latent (B,D). */
typedef struct snb_batch_desc {
  int32_t n_objs;
  int32_t n_samples;
  int64_t rays_per_obj;
  int32_t flags;        /* SNB_WHITE_BKGD | SNB_SIGMA_RELU [| SNB_BATCH_FUSED_SAMPLER | SNB_BATCH_FP32_TC] */
  int32_t reserved;
} snb_batch_desc;
/* opt-in: the forward decoder computes every row's stratified sample itself from the ray (32 B) and its jitter (4 B) -- no sampler
 * kernel and no per-row coordinates in HBM on the forward path; the backward re-materialises them in its scratch.  Bit-identical
 * results; measured ~0.7 % slower per forward + backward step than the default (DESIGN.md, row N1). */
#define SNB_BATCH_FUSED_SAMPLER 4
/* the decoder of the batched render in SNB_PREC_FP32_TC arithmetic (fp32-grade on the tensor cores) instead of bf16; not together
 * with SNB_BATCH_FUSED_SAMPLER */
#define SNB_BATCH_FP32_TC 8
size_t snb_render_batch_workspace_bytes(snb_handle h, const snb_batch_desc* d);
size_t snb_render_batch_scratch_bytes(snb_handle h, const snb_batch_desc* d);
int snb_render_batch_fwd(snb_handle h, const snb_batch_desc* d, const float* px, const float* py, const float* K,
                         const float* c2w, const float* box, const float* z_steps, const float* jitter,
                         const float* shape_latent, const float* texture_latent, float* out_rgb, float* out_depth,
                         float* out_acc, uint8_t* out_hit, void* workspace, void* stream);
int snb_render_batch_bwd(snb_handle h, const snb_batch_desc* d, const float* px, const float* py, const float* K,
                         const float* c2w, const float* box, const float* z_steps, const float* jitter,
                         const float* shape_latent, const float* texture_latent, const void* workspace,
                         const float* g_rgb, const float* g_depth, const float* g_acc, void* scratch, float* g_c2w,
                         float* g_shape_latent, float* g_texture_latent, void* stream);
/* Dataset-side sample preparation on the device (SURVEY 8f rank 3): utils.prepare_pixel_samples (utils.py:330-377), which the
 * reference's DataLoader workers run per object on the CPU (data_nuscenes.py:615-658), for n_objs objects in one launch.
 * px, py (B,n) pixel coordinates of the chosen rays; K (B,3,3); c2w (B,3,4); z (B,S) every object's shared sample vector
 * (utils.sample_from_rays, built by the caller with the reference's torch calls); obj_diag (B); flip (B) int32 or NULL (sym_aug
 * taken: y components negated); shapenet_swap: (x, y, z) -> (-y, x, z).  -> xyz, viewdir_rep (B,n,S,3), forward only. */
int snb_prepare_samples_batch(const float* px, const float* py, const float* K, const float* c2w, const float* z,
                              const float* obj_diag, const int32_t* flip, int32_t n_objs, int64_t rays_per_obj,
                              int32_t n_samples, int32_t shapenet_swap, float* xyz, float* viewdir_rep, void* stream);
/* The refine losses (below) of n_objs objects in one launch per direction: rgb, tgt (B,N,3); acc, occ (B,N);
 * out3 (B,3) = {loss, loss_rgb, loss_occ} per object, each over its own denominator; g_loss (B) or NULL (= ones). */
size_t snb_refine_loss_batch_scratch_bytes(int32_t n_objs);
int snb_refine_loss_batch_fwd(const float* rgb, const float* acc, const float* tgt, const float* occ, int32_t n_objs,
                              int64_t rays_per_obj, float occ_coef, float* out3, void* scratch, void* stream);
int snb_refine_loss_batch_bwd(const float* rgb, const float* acc, const float* tgt, const float* occ, int32_t n_objs,
                              int64_t rays_per_obj, float occ_coef, const void* scratch, const float* g_loss, float* g_rgb,
                              float* g_acc, void* stream);

/* ---- gradient all-reduce of the sharded modes (SURVEY 8b, 8e) --------------------------------------------------------
 * No reference counterpart (the reference only has nn.DataParallel, trainer_nerf_nuscenes.py:94-95).  ONE in-place
 * ncclAllReduce(sum, fp32) of `flat` (n floats, device memory) over the caller's communicator (an ncclComm_t, passed as void*)
 * on the caller's stream: the ray-sharded mode reduces [d cam_pose (12) | d shapecode (D) | d texturecode (D) | loss] (2.1 KB),
 * the data-parallel mode its flat weight-gradient buffer.  NCCL is resolved at run time from the libnccl.so.2 the process
 * already uses (torch.distributed's); the library does not link it. */
int snb_allreduce_grads(snb_handle h, void* nccl_comm, float* flat, size_t n, void* stream);

/* ---- refine-iteration loss (the caller just above the render; SURVEY 8(f) rank 1) -------------------------------
 * Replaces the inline loss of optimizer_nuscenes.py:729-736 (= optimizer_kitti.py / optimizer_waymo.py, and the render
 * losses of trainer_unified_nuscenes.py:316-332):
 *   den = sum|occ| + 1e-9; loss_rgb = sum((rgb - tgt)^2 |occ|) / den; loss_occ = sum(exp(-occ (0.5 - acc)) |occ|) / den;
 *   loss = loss_rgb + occ_coef * loss_occ.
 * rgb, tgt (N,3); acc (N); occ (N) in {-1,0,+1}.  den: NULL, or a device float holding a caller-computed denominator (the
 * ray-sharded mode passes the GLOBAL sum|occ| + 1e-9).  out3 = {loss, loss_rgb, loss_occ}.  scratch:
 * snb_refine_loss_scratch_bytes(), kept until the backward.  Backward: g_loss = device float (NULL = 1), writes
 * g_rgb (N,3) and g_acc (N). */
size_t snb_refine_loss_scratch_bytes(void);
int snb_refine_loss_fwd(const float* rgb, const float* acc, const float* tgt, const float* occ, int64_t n_rays,
                        float occ_coef, const float* den, float* out3, void* scratch, void* stream);
int snb_refine_loss_bwd(const float* rgb, const float* acc, const float* tgt, const float* occ, int64_t n_rays,
                        float occ_coef, const void* scratch, const float* g_loss, float* g_rgb, float* g_acc, void* stream);

/* ---- multi-object scene compositor, merge step (SURVEY 8(f) rank 4) ------------------------------------------------
 * Replaces scripts/demo.py:560-567: z_sort = sort(z_vals).values; z_args = searchsorted(z_sort, z_vals);
 * sigmas_sort / rgbs_sort = zeros.scatter_(1, z_args, .) -- ties collide, the last element in index order wins, the other
 * slots of the tie group stay zero.  z, sigma (R, K), rgb (R, K, 3) with K = objects x samples <= 1024; z_args (R, K) int64
 * may be NULL.  Follow with snb_composite_fwd(sigma_sort, rgb_sort, z_sort, 1, R, K, SNB_WHITE_BKGD | SNB_SIGMA_RELU)
 * (= volume_rendering3(..., white_bkgd=True), demo.py:569). */
int snb_merge_sort_samples(const float* z, const float* sigma, const float* rgb, int64_t n_rays, int32_t n_per_ray,
                           float* z_sort, float* sigma_sort, float* rgb_sort, int64_t* z_args, void* stream);

/* ---- refine-iteration glue around the render (SURVEY 8(f) rank 1), for B objects side by side --------------------------
 * (one object is B = 1; one GPU's share of config C3 -- 32 objects over 8 GPUs -- or C fixed slots of a stream of objects)
 * snb_refine_pose_slots_fwd: optimizer_nuscenes.py:684-699 -- rot_vec (B,3, axis-angle; Rodrigues = what
 * pytorch3d.transforms.axis_angle_to_matrix evaluates), trans_vec (B,3) -> cam2opt (B,3,4) = [R | t] (opt_cam_pose != 0) or
 * [R^T | -R^T t] (opt_cam_pose == 0, every shipped config), and every object's shared sample vector z (B,S) of
 * utils.sample_from_rays (utils.py:154-167) with near/far = ||cam2opt[:,3]|| -/+ obj_diag/2 (obj_diag (B), device;
 * utils.py:468-469, detached).  Object b's jitter is row int(step_counters[b]) of its table (B, table_rows, S) -- the
 * torch.rand(n_samples) draw of that iteration, picked by the object's AdamW step counter of snb_adamw_step_rows, so a
 * captured iteration needs neither an index_select nor a counter launch.  z2 / jitter2: a second sample vector from the same
 * pose and another draw (the lidar-pixel evaluation of optimizer_nuscenes.py:759-769); both NULL = not wanted.  active (B
 * bytes): an active object whose counter lies outside [0, table_rows) gets NaN in its z / z2 and sets *err_flag to 1 (a
 * device int32, NULL = not reported); an inactive one reads a row inside the table and reports nothing.
 * snb_refine_pose_batch_bwd: g_cam (B,3,4) -> g_rot, g_trans (B,3).
 * snb_adamw_step_rows: torch.optim.AdamW's update (optimizer_nuscenes.py:757-769, groups of :1762-1769) on n_rows independent
 * rows of up to 8 tensors with their own learning rates (row r of tensor i: row_sizes[i] elements at r * row_sizes[i]).
 * steps (n_rows device floats): each row's step count -- its bias corrections -- incremented by the call; active (n_rows
 * bytes): an inactive row's parameters, moments and count stay bit-for-bit unchanged.  loss_history (NULL = none):
 * (n_rows, history_rows, 4); an active row r with 0 <= steps[r] < history_rows first writes {loss3[3r .. 3r+2],
 * loss_rgb2[r * loss_rgb2_stride]} to row steps[r]. */
int snb_refine_pose_slots_fwd(const float* rot_vec, const float* trans_vec, int32_t n_slots, int32_t opt_cam_pose,
                              const float* obj_diag, int32_t n_samples, const float* jitter, const float* jitter2,
                              const float* step_counters, int32_t table_rows, const uint8_t* active, int32_t* err_flag,
                              float* cam, float* z, float* z2, void* stream);
int snb_refine_pose_batch_bwd(const float* rot_vec, const float* trans_vec, int32_t n_objs, int32_t opt_cam_pose,
                              const float* g_cam, float* g_rot, float* g_trans, void* stream);
int snb_adamw_step_rows(int32_t n_groups, float* const* params, const float* const* grads, float* const* exp_avg,
                        float* const* exp_avg_sq, const int32_t* row_sizes, const float* lrs, float beta1, float beta2,
                        float eps, float weight_decay, int32_t n_rows, float* steps, const uint8_t* active,
                        const float* loss3, const float* loss_rgb2, int32_t loss_rgb2_stride, float* loss_history,
                        int32_t history_rows, void* stream);

/* ---- the render for B objects side by side ---------------------------------------------------------------------------
 * snb_render_shell_batch_fwd/bwd: utils.render_rays_v2 (utils.py:435-502) for B objects in one launch set: px, py (B,N); K
 * (B,3,3); c2w (B,3,4); z (B,S); obj_diag (B); latents (B,D) -> rgb (B,N,3), depth, acc (B,N).  Frozen weights; bf16 needs
 * N * S to be a multiple of 128.  Backward: g_rgb (B,N,3), g_depth, g_acc (B,N) -> g_c2w (B,3,4; NULL = not wanted),
 * g_shape_latent, g_texture_latent (B,D).  Workspace / scratch: 256-byte aligned, sizes from the *_bytes calls. */
typedef struct snb_shell_batch_desc {
  int32_t n_objs;
  int32_t n_samples;
  int64_t rays_per_obj;
  int32_t precision;     /* SNB_PREC_FP32 | SNB_PREC_BF16 */
  int32_t flags;         /* SNB_SIGMA_RELU [| SNB_WHITE_BKGD] */
  int32_t shapenet_swap;
  int32_t reserved;
} snb_shell_batch_desc;
size_t snb_render_shell_batch_workspace_bytes(snb_handle h, const snb_shell_batch_desc* d);
size_t snb_render_shell_batch_scratch_bytes(snb_handle h, const snb_shell_batch_desc* d);
int snb_render_shell_batch_fwd(snb_handle h, const snb_shell_batch_desc* d, const float* px, const float* py, const float* K,
                               const float* c2w, const float* z, const float* obj_diag, const float* shape_latent,
                               const float* texture_latent, float* out_rgb, float* out_depth, float* out_acc, void* workspace,
                               void* stream);
int snb_render_shell_batch_bwd(snb_handle h, const snb_shell_batch_desc* d, const float* px, const float* py, const float* K,
                               const float* c2w, const float* z, const float* obj_diag, const float* shape_latent,
                               const float* texture_latent, const void* workspace, const float* g_rgb, const float* g_depth,
                               const float* g_acc, void* scratch, float* g_c2w, float* g_shape_latent, float* g_texture_latent,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif
