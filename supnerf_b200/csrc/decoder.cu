// Host side of the decoder MLP: which back end runs for (architecture, precision), the workspace and packed-weight layouts of the
// tensor-core back ends, and the forward / backward dispatch around their kernels (latent layers, memsets, kernel timing).
#include "common.cuh"
#include "decoder.h"
#include "tc_ptx.cuh"

namespace snb {

static const char kNoTwoTileTraining[] = "weight gradients need the two-tile tcgen05 kernels (W = 256, shape_blocks + "
                                         "texture_blocks <= 4); use precision='fp32' for this architecture";

const char* select_backend(const snb_handle_s* h, int32_t precision, Backend* be) {
  if (precision == SNB_PREC_FP32) { *be = Backend::Ffma; return nullptr; }
  const char* why = nullptr;
  if (!tc1_supported(h, &why)) return why;
  if (precision == SNB_PREC_FP32_TC) { *be = Backend::OneTileSplit; return nullptr; }
  if (tc2_supported(h)) { *be = Backend::TwoTile; return nullptr; }
  if (precision == SNB_PREC_BF16_TRAIN) return kNoTwoTileTraining;
  *be = Backend::OneTile;
  return nullptr;
}

// error text of the decoder entry points for a configuration select_backend rejects
static int reject(const char* who, const char* why) {
  set_error("%s(%s): %s", who, why == kNoTwoTileTraining ? "bf16, training" : "bf16", why);
  return 2;
}

static bool tc_precision(int32_t precision) {
  return precision == SNB_PREC_BF16 || precision == SNB_PREC_BF16_TRAIN || precision == SNB_PREC_FP32_TC;
}

static inline size_t al256(size_t b) { return (b + 255) & ~size_t(255); }
static inline size_t al1k(size_t b) { return (b + 1023) & ~size_t(1023); }
static inline uint8_t* align1k(uint8_t* p) { return (uint8_t*)(((uintptr_t)p + 1023) & ~uintptr_t(1023)); }

// Workspace and backward scratch of the tensor-core back ends (byte offsets):
//   workspace  zlat (Bs+Bt)*B*W fp32 | effective biases (same) | their bias-stage images, 32 B per unit | ReLU masks, 1 bit per unit
//              | training: the forward's operand tiles (1 KB aligned in memory)
//   scratch    latent column sums (zlat's shape) | their W^T fold | training: the backward's operand tiles (1 KB aligned), then a
//              d xyz / d viewdir dummy (the training backward always runs the full program)
struct TcLayout {
  size_t zlat_bytes, ebias, eimg, masks, fsave, ws_bytes;
  size_t fold, bsave, sc_bytes;
  bool train;
  TcLayout(const snb_handle_s* h, int32_t precision, int64_t M, int64_t B) {
    const int slots = h->arch.shape_blocks + h->arch.texture_blocks, W = h->arch.W;
    const size_t tiles = (size_t)((M + tc::kTileM - 1) / tc::kTileM);
    train = precision == SNB_PREC_BF16_TRAIN && tc2_supported(h);
    zlat_bytes = (size_t)slots * B * W * sizeof(float);
    ebias = zlat_bytes;
    eimg = al256(2 * zlat_bytes);
    masks = al256(eimg + 8 * zlat_bytes);
    fsave = masks + tiles * (slots + 3) * (W / 32) * 128 * 4 + 256;
    ws_bytes = fsave + (train ? tc2_fwd_save_bytes(h, M) + 1024 : 0);
    fold = zlat_bytes;
    bsave = al256(2 * zlat_bytes) + 256;
    sc_bytes = bsave + (train ? tc2_bwd_save_bytes(h, M) + (size_t)M * 24 + 1024 : 0);
  }
};

size_t decoder_workspace_bytes(const snb_handle_s* h, int32_t precision, int64_t M, int64_t B) {
  if (!tc_precision(precision)) return f32_workspace_floats(h, M, B) * sizeof(float);
  return TcLayout(h, precision, M, B).ws_bytes;
}

size_t decoder_scratch_bytes(const snb_handle_s* h, int32_t precision, int64_t M, int64_t B) {
  if (!tc_precision(precision)) return f32_bwd_scratch_floats(h, M, B) * sizeof(float);
  return TcLayout(h, precision, M, B).sc_bytes;
}

// The packed weight buffer: the one-tile bf16 image, the two-tile image (where those kernels apply), the split-precision image.
static const snb_packed_layout& packed_layout(const snb_handle_s* h) {
  snb_packed_layout& L = h->packed_layout;
  if (L.bytes == 0) {
    L.two_tile = al1k(tc1_image_bytes(h, false) + 1024);
    L.split = al1k(L.two_tile + tc2_packed_bytes(h));
    L.bytes = L.split + al1k(tc1_image_bytes(h, true) + 1024);
  }
  return L;
}

size_t decoder_packed_bytes(const snb_handle_s* h) {
  Backend be;
  return select_backend(h, SNB_PREC_BF16, &be) ? 16 : packed_layout(h).bytes;
}

int decoder_pack_weights(snb_handle_s* h, void* packed, cudaStream_t st) {
  Backend be;
  const char* why = select_backend(h, SNB_PREC_BF16, &be);
  SNB_REQUIRE(why == nullptr, "snb_pack_weights: %s", why);
  SNB_REQUIRE(((uintptr_t)packed & 15) == 0, "snb_pack_weights: buffer must be 16-byte aligned");
  const snb_packed_layout& L = packed_layout(h);
  if (tc1_pack_weights(h, false, packed, st) || tc1_pack_weights(h, true, (uint8_t*)packed + L.split, st)) return 1;
  if (be == Backend::TwoTile && tc2_pack_weights(h, (uint8_t*)packed + L.two_tile, st)) return 1;
  h->packed = packed;
  return 0;
}

void decoder_timing_enable(snb_handle_s* h, int on) {
  h->timing_on = on != 0;
  for (auto* v : {&h->ev_fwd, &h->ev_bwd}) {
    for (auto& e : *v) { cudaEventDestroy((cudaEvent_t)e.first); cudaEventDestroy((cudaEvent_t)e.second); }
    v->clear();
  }
}

int decoder_timing_read(snb_handle_s* h, int which, float* ms, int max_n) {
  auto& v = which == 0 ? h->ev_fwd : h->ev_bwd;
  int n = 0;
  for (auto& e : v) {
    if (n >= max_n) break;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, (cudaEvent_t)e.first, (cudaEvent_t)e.second) == cudaSuccess) ms[n++] = t;
  }
  return n;
}

struct ScopedKernelTimer {
  cudaStream_t st; std::pair<cudaEvent_t, cudaEvent_t> ev; bool on;
  ScopedKernelTimer(cudaStream_t s, bool enable) : st(s), on(enable) {
    if (on) { cudaEventCreate(&ev.first); cudaEventCreate(&ev.second); cudaEventRecord(ev.first, st); }
  }
  void stop(std::vector<std::pair<void*, void*>>& into) { if (on) { cudaEventRecord(ev.second, st); into.push_back({(void*)ev.first, (void*)ev.second}); } }
};

int decoder_zero_grads(const snb_handle_s* h, int64_t B, float* g_shape_latent, float* g_texture_latent, float* const* g_weights,
                       cudaStream_t st) {
  if (g_shape_latent) SNB_CHECK_CUDA(cudaMemsetAsync(g_shape_latent, 0, sizeof(float) * B * h->arch.latent_dim, st));
  if (g_texture_latent) SNB_CHECK_CUDA(cudaMemsetAsync(g_texture_latent, 0, sizeof(float) * B * h->arch.latent_dim, st));
  if (g_weights)
    for (size_t i = 0; i < h->layers.size(); ++i) {
      SNB_CHECK_CUDA(cudaMemsetAsync(g_weights[2 * i], 0, sizeof(float) * h->layers[i].out * h->layers[i].in, st));
      SNB_CHECK_CUDA(cudaMemsetAsync(g_weights[2 * i + 1], 0, sizeof(float) * h->layers[i].out, st));
    }
  return 0;
}

// checks every tensor-core back end shares
static int tc_checks(const snb_handle_s* h, int64_t M, int64_t B, const char* who, const DeviceRows& r) {
  SNB_REQUIRE(h->packed != nullptr, "%s: weights not packed (call snb_pack_weights)", who);
  SNB_REQUIRE(r.tile_start != nullptr || (M / B) % tc::kTileM == 0,
              "%s: bf16 mode needs samples-per-object (%lld) to be a multiple of %d; use fp32 mode", who, (long long)(M / B), tc::kTileM);
  return 0;
}

int decoder_forward(const snb_handle_s* h, int32_t precision, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                    const float* shape_latent, const float* texture_latent, float* sigma, float* rgb, void* ws, cudaStream_t st,
                    const DeviceRows& r) {
  Backend be;
  if (const char* why = select_backend(h, precision, &be)) return reject("mlp_fwd", why);
  if (be == Backend::Ffma) return f32_forward(h, xyz, viewdir, M, B, shape_latent, texture_latent, sigma, rgb, (float*)ws, st);
  if (tc_checks(h, M, B, "mlp_fwd(bf16)", r)) return 2;
  if (be == Backend::OneTileSplit) {   // fp16 (hi, lo) operands, three MMAs per product (frozen weights)
    SNB_REQUIRE(r.rs == nullptr && xyz != nullptr && viewdir != nullptr, "mlp_fwd(fp32_tc): frozen weights and explicit coordinates only");
    SNB_REQUIRE(r.tile_start == nullptr || r.m_dev != nullptr, "mlp_fwd(fp32_tc): per-object tile offsets need a device-side row count");
  } else {
    SNB_REQUIRE(r.rs == nullptr || (r.tile_start != nullptr && r.rs->rays8 && r.rs->box && r.rs->z_steps && r.rs->jitter && r.rs->order &&
                                    r.rs->counts), "mlp_fwd(bf16): a row source needs per-object tile offsets and all of its pointers");
    SNB_REQUIRE(r.rs != nullptr || (xyz != nullptr && viewdir != nullptr), "mlp_fwd(bf16): null coordinates");
    SNB_REQUIRE(r.m_dev == nullptr || B == 1 || r.tile_start != nullptr,
                "mlp_fwd(bf16): a device-side row count needs one object (or per-object tile offsets)");
    SNB_REQUIRE(r.tile_start == nullptr || (r.m_dev != nullptr && precision != SNB_PREC_BF16_TRAIN),
                "mlp_fwd(bf16): per-object tile offsets need frozen weights and a device-side row count");
    SNB_REQUIRE(r.rs == nullptr || be == Backend::TwoTile, "mlp_fwd(bf16): the fused sampler needs the two-tile kernels");
  }
  const TcLayout L(h, precision, M, B);
  uint8_t* w = (uint8_t*)ws;
  float* zlat = (float*)w;
  float* ebias = (float*)(w + L.ebias);
  uint8_t* eimg = w + L.eimg;
  uint32_t* masks = (uint32_t*)(w + L.masks);
  const uint8_t* packed = (const uint8_t*)h->packed;
  const bool two = be == Backend::TwoTile;
  if (latent_forward_fused(h, B, shape_latent, texture_latent, zlat, ebias, st, two ? eimg : nullptr)) return 1;
  ScopedKernelTimer tm(st, h->timing_on);
  int rc;
  if (two)
    rc = tc2_launch_fwd(h, packed + packed_layout(h).two_tile, xyz, viewdir, M, B, eimg, masks, sigma, rgb, h->dbg_acts,
                        L.train ? align1k(w + L.fsave) : nullptr, st, r.m_dev, r.tile_start, r.rs);
  else if (be == Backend::OneTileSplit)
    rc = tc1_launch_fwd<true>(h, packed + packed_layout(h).split, xyz, viewdir, M, B, ebias, masks, sigma, rgb, st, r.m_dev, r.tile_start);
  else
    rc = tc1_launch_fwd<false>(h, packed, xyz, viewdir, M, B, ebias, masks, sigma, rgb, st, r.m_dev, r.tile_start);
  if (rc) return 1;
  tm.stop(const_cast<snb_handle_s*>(h)->ev_fwd);
  SNB_LAUNCH_CHECK();
  return 0;
}

int decoder_backward(const snb_handle_s* h, int32_t precision, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                     const float* shape_latent, const float* texture_latent, const float* sigma, const float* g_sigma,
                     const float* g_rgb, const void* ws, void* scratch, float* g_xyz, float* g_viewdir, float* g_shape_latent,
                     float* g_texture_latent, float* const* g_weights, cudaStream_t st, const DeviceRows& r) {
  Backend be;
  if (const char* why = select_backend(h, precision, &be)) return reject("mlp_bwd", why);
  if (be == Backend::Ffma)
    return f32_backward(h, xyz, viewdir, M, B, shape_latent, texture_latent, sigma, g_sigma, g_rgb, (const float*)ws, (float*)scratch,
                        g_xyz, g_viewdir, g_shape_latent, g_texture_latent, g_weights, st);
  if (tc_checks(h, M, B, "mlp_bwd(bf16)", r)) return 2;
  SNB_REQUIRE(r.live == nullptr || (r.n_live != nullptr && r.tile_start != nullptr && g_weights == nullptr),
              "mlp_bwd: a list of live super tiles needs its count, per-object tile offsets and frozen weights");
  const TcLayout L(h, precision, M, B);
  if (be == Backend::OneTileSplit) {
    SNB_REQUIRE(g_weights == nullptr, "mlp_bwd(fp32_tc): frozen weights only (weight gradients: precision='fp32' runs the FFMA back end)");
    SNB_REQUIRE((g_xyz == nullptr) == (g_viewdir == nullptr), "mlp_bwd(fp32_tc): request both g_xyz and g_viewdir or neither");
    SNB_REQUIRE(r.tile_start == nullptr || r.m_dev != nullptr, "mlp_bwd(fp32_tc): per-object tile offsets need a device-side row count");
  } else {
    SNB_REQUIRE(r.m_dev == nullptr || B == 1 || r.tile_start != nullptr,
                "mlp_bwd(bf16): a device-side row count needs one object (or per-object tile offsets)");
    SNB_REQUIRE(r.tile_start == nullptr || (r.m_dev != nullptr && precision != SNB_PREC_BF16_TRAIN),
                "mlp_bwd(bf16): per-object tile offsets need frozen weights and a device-side row count");
    SNB_REQUIRE(g_weights == nullptr || L.train,
                "mlp_bwd(bf16): weight gradients need the forward to have run in training mode (SNB_PREC_BF16_TRAIN: the python "
                "modules select it when a weight requires grad) on an architecture the two-tile kernels cover; otherwise freeze "
                "the weights (requires_grad_(False)) or use precision='fp32'");
    SNB_REQUIRE((g_xyz == nullptr) == (g_viewdir == nullptr), "mlp_bwd(bf16): request both g_xyz and g_viewdir or neither");
  }
  const uint8_t* w = (const uint8_t*)ws;
  const float* zlat = (const float*)w;
  uint32_t* masks = (uint32_t*)(w + L.masks);
  float* g_zlat = (float*)scratch;
  float* fold_tmp = (float*)((uint8_t*)scratch + L.fold);
  const uint8_t* packed = (const uint8_t*)h->packed;
  SNB_CHECK_CUDA(cudaMemsetAsync(g_zlat, 0, L.zlat_bytes, st));
  uint8_t* bsave = nullptr;
  if (g_weights != nullptr) {   // training: keep every step's d pre-activation tile, run the full program (d xyz into a dummy if unwanted)
    bsave = align1k((uint8_t*)scratch + L.bsave);
    float* dummy = (float*)(bsave + tc2_bwd_save_bytes(h, M));
    if (g_xyz == nullptr) { g_xyz = dummy; g_viewdir = dummy + 3 * M; }
    if (decoder_zero_grads(h, B, nullptr, nullptr, g_weights, st)) return 1;   // every weight gradient is accumulated (atomics / +=)
  }
  ScopedKernelTimer tm(st, h->timing_on);
  int rc;
  if (be == Backend::TwoTile)
    rc = tc2_launch_bwd(h, packed + packed_layout(h).two_tile, xyz, viewdir, M, B, masks, sigma, g_sigma, g_rgb, g_xyz, g_viewdir,
                        g_zlat, bsave, st, r.m_dev, r.tile_start, r.live, r.n_live);
  else if (be == Backend::OneTileSplit)
    rc = tc1_launch_bwd<true>(h, packed + packed_layout(h).split, xyz, viewdir, M, B, zlat, masks, sigma, g_sigma, g_rgb, g_xyz,
                              g_viewdir, g_zlat, st, r.m_dev, r.tile_start, r.live, r.n_live);
  else
    rc = tc1_launch_bwd<false>(h, packed, xyz, viewdir, M, B, zlat, masks, sigma, g_sigma, g_rgb, g_xyz, g_viewdir, g_zlat, st,
                               r.m_dev, r.tile_start, r.live, r.n_live);
  if (rc) return 1;
  tm.stop(const_cast<snb_handle_s*>(h)->ev_bwd);
  SNB_LAUNCH_CHECK();
  if (be != Backend::TwoTile) return latent_backward_fused(h, B, zlat, g_zlat, g_shape_latent, g_texture_latent, st);
  if (g_weights == nullptr) return latent_backward_fused(h, B, zlat, g_zlat, g_shape_latent, g_texture_latent, st, fold_tmp);
  if (tc2_launch_wgrad(h, M, B, align1k((uint8_t*)w + L.fsave), bsave, sigma, g_sigma, g_rgb, g_zlat, zlat, g_weights, st, r.m_dev))
    return 1;
  // latent layers (per object): fold the column sums through W_layer^T (= d loss / d z), d latent, then their weight gradients
  if (latent_backward_fused(h, B, zlat, g_zlat, g_shape_latent, g_texture_latent, st, fold_tmp)) return 1;
  return tc2_launch_latent_wgrad(h, B, zlat, fold_tmp, shape_latent, texture_latent, g_weights, st);
}

}  // namespace snb
