// Internal interface of the decoder MLP.  decoder.cu picks the back end for (architecture, precision), lays out its workspace
// and packed weights and runs it; the back ends below are the kernel files' host entry points it calls.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "handle.h"
#include "rb_rows.cuh"

namespace snb {

// Ffma: SNB_PREC_FP32 (mlp_f32.cu).  OneTile: SNB_PREC_BF16 where the two-tile kernels do not apply (mlp_tc.cu).
// OneTileSplit: SNB_PREC_FP32_TC, the split-precision one-tile kernels (mlp_tc.cu).  TwoTile: SNB_PREC_BF16 / SNB_PREC_BF16_TRAIN
// (mlp_tc2.cu).
enum class Backend { Ffma, OneTile, OneTileSplit, TwoTile };

// The back end that runs the decoder for (architecture, precision): nullptr and *be set, or why there is none.
const char* select_backend(const snb_handle_s* h, int32_t precision, Backend* be);

// Rows the tensor-core back ends find on the device instead of taking M at face value.
struct DeviceRows {
  const int64_t* m_dev = nullptr;       // number of rows actually present (a multiple of 128, <= M)
  const int32_t* tile_start = nullptr;  // B + 1 ascending, even ints: object b owns the 128-row tiles [tile_start[b], tile_start[b+1])
  const rb::RowSrc* rs = nullptr;       // forward only: the two-tile kernels compute each row's sample (xyz / viewdir unused)
  // backward only (frozen weights, per-object tile offsets): the 256-row super tiles to run, ascending, and their count.  A super tile
  // left out has upstream gradients that are exactly zero: its rows' d xyz / d viewdir are not written and it adds nothing to the
  // latent gradients.  Null: every super tile.
  const int32_t* live = nullptr;
  const int32_t* n_live = nullptr;
};

size_t decoder_workspace_bytes(const snb_handle_s* h, int32_t precision, int64_t M, int64_t B);
size_t decoder_scratch_bytes(const snb_handle_s* h, int32_t precision, int64_t M, int64_t B);
size_t decoder_packed_bytes(const snb_handle_s* h);
int decoder_pack_weights(snb_handle_s* h, void* packed, cudaStream_t st);
int decoder_forward(const snb_handle_s* h, int32_t precision, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                    const float* shape_latent, const float* texture_latent, float* sigma, float* rgb, void* ws, cudaStream_t st,
                    const DeviceRows& rows = {});
int decoder_backward(const snb_handle_s* h, int32_t precision, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                     const float* shape_latent, const float* texture_latent, const float* sigma, const float* g_sigma,
                     const float* g_rgb, const void* ws, void* scratch, float* g_xyz, float* g_viewdir, float* g_shape_latent,
                     float* g_texture_latent, float* const* g_weights, cudaStream_t st, const DeviceRows& rows = {});
// zeroes the given gradients (null ones are skipped): latents (B, latent_dim), every weight and bias
int decoder_zero_grads(const snb_handle_s* h, int64_t B, float* g_shape_latent, float* g_texture_latent, float* const* g_weights,
                       cudaStream_t st);
// kernel-only timing (bench.py roofline): CUDA events around every tcgen05 decoder kernel; read after a synchronize
void decoder_timing_enable(snb_handle_s* h, int on);
int decoder_timing_read(snb_handle_s* h, int which, float* ms, int max_n);

// ---- FFMA back end (mlp_f32.cu)
size_t f32_workspace_floats(const snb_handle_s* h, int64_t M, int64_t B);
size_t f32_bwd_scratch_floats(const snb_handle_s* h, int64_t M, int64_t B);
int f32_forward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                const float* shape_latent, const float* texture_latent, float* sigma, float* rgb, float* ws,
                cudaStream_t st);
int f32_backward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                 const float* shape_latent, const float* texture_latent, const float* sigma, const float* g_sigma,
                 const float* g_rgb, const float* ws, float* scratch, float* g_xyz, float* g_viewdir,
                 float* g_shape_latent, float* g_texture_latent, float* const* g_weights, cudaStream_t st);

// ---- per-object latent layers (latent.cu), shared by all back ends.  zlat / dz: [(Bs+Bt)][B][W] (shape slots first).
// Forward of all slots, + the effective biases if ebias != NULL: ebias[slot][b][:] = bias + W z of the layer that consumes latent slot
// `slot` (shape_layer_j / texture_layer_j), the latent add folded through the layer, exact in fp32 (SURVEY 8(a')3).
// eimg != NULL: also write every effective bias as a tcgen05 bias-stage row (32 B each, [(Bs+Bt)][B][W]; tc_ptx.cuh)
int latent_forward_fused(const snb_handle_s* h, int64_t B, const float* shape_latent, const float* texture_latent, float* zlat,
                         float* ebias, cudaStream_t st, uint8_t* eimg = nullptr);
// fold_tmp != NULL: dz holds the column sums of the consuming layers' pre-activation gradients (two-tile tcgen05 backward);
// they are first folded through W_layer^T into fold_tmp (same size as dz).
int latent_backward_fused(const snb_handle_s* h, int64_t B, const float* zlat, const float* dz, float* g_shape_latent,
                          float* g_texture_latent, cudaStream_t st, float* fold_tmp = nullptr);

// ---- one-tile tensor-core back end (mlp_tc.cu); X = split precision.  The launch functions launch one kernel and leave the
// launch count to the caller.
bool tc1_supported(const snb_handle_s* h, const char** why);
size_t tc1_image_bytes(const snb_handle_s* h, bool split);
int tc1_pack_weights(const snb_handle_s* h, bool split, void* packed, cudaStream_t st);
template <bool X>
int tc1_launch_fwd(const snb_handle_s* h, const void* packed, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const float* ebias, uint32_t* masks, float* sigma, float* rgb, cudaStream_t st, const int64_t* m_dev,
                   const int32_t* tile_start);
template <bool X>
int tc1_launch_bwd(const snb_handle_s* h, const void* packed, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const float* zlat, uint32_t* masks, const float* sigma, const float* g_sigma, const float* g_rgb, float* g_xyz,
                   float* g_viewdir, float* g_zlat, cudaStream_t st, const int64_t* m_dev, const int32_t* tile_start,
                   const int32_t* live, const int32_t* n_live);

// ---- two-tile tensor-core back end (mlp_tc2.cu).  Same launch-count convention for tc2_launch_fwd / tc2_launch_bwd.
bool tc2_supported(const snb_handle_s* h);
size_t tc2_packed_bytes(const snb_handle_s* h);
int tc2_pack_weights(const snb_handle_s* h, void* packed, cudaStream_t st);
int tc2_launch_fwd(const snb_handle_s* h, const void* packed2, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const uint8_t* eimg, uint32_t* masks, float* sigma, float* rgb, float* dbg, uint8_t* save, cudaStream_t st,
                   const int64_t* m_dev, const int32_t* tile_start, const rb::RowSrc* rs);
int tc2_launch_bwd(const snb_handle_s* h, const void* packed2, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const uint32_t* masks, const float* sigma, const float* g_sigma, const float* g_rgb, float* g_xyz,
                   float* g_viewdir, float* g_zlat, uint8_t* save, cudaStream_t st, const int64_t* m_dev, const int32_t* tile_start,
                   const int32_t* live, const int32_t* n_live);
// training mode: bytes of the operand tiles the forward / backward keep for the weight-gradient kernels
size_t tc2_fwd_save_bytes(const snb_handle_s* h, int64_t M);
size_t tc2_bwd_save_bytes(const snb_handle_s* h, int64_t M);
int tc2_launch_wgrad(const snb_handle_s* h, int64_t M, int64_t B, const uint8_t* fsave, const uint8_t* bsave, const float* sigma,
                     const float* g_sigma, const float* g_rgb, const float* s_lat, const float* zlat, float* const* gw,
                     cudaStream_t st, const int64_t* m_dev);
int tc2_launch_latent_wgrad(const snb_handle_s* h, int64_t B, const float* zlat, const float* dz, const float* shape_latent,
                            const float* texture_latent, float* const* gw, cudaStream_t st);

}  // namespace snb
