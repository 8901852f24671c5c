// Per-object latent layers of the CodeNeRF-family decoder (model_codenerf.py:51,59: `*_latent_layer_j`), hoisted
// out of the per-sample path (exact restructuring, SURVEY 8(a')3).  One launch computes, for every object and
// every latent slot,  z = ReLU(W_lat latent + b_lat)  and the EFFECTIVE BIAS  W_layer z + b_layer  of the layer
// that consumes z (the latent add folded through that layer, used by the tcgen05 back end).  One launch does
// the backward (ReLU mask, then d latent = sum_slots W_lat^T d_pre).
#include "common.cuh"
#include "decoder.h"
#include "tc_ptx.cuh"

namespace snb {

constexpr int kMaxSlots = 32;
struct LatentLayers {
  int n_shape, n_total, W, D;
  const float* wl[kMaxSlots]; const float* bl[kMaxSlots];   // latent layers (W, D), (W)
  const float* wc[kMaxSlots]; const float* bc[kMaxSlots];   // consuming layers (W, W), (W)
};

// One warp per output unit, 8 outputs per 256-thread block: grid (slots, B, W/8) so even one object fills the machine
// (the single-block-per-slot version took ~250 us per launch: 20 % of a refine step, profiles/r1_launches_v5.md).
// PHASE 0: zlat[slot][b][o] = ReLU(W_lat[o,:] . latent[b,:] + b_lat[o]).
// PHASE 1: ebias[slot][b][o] = W_layer[o,:] . zlat[slot][b][:] + b_layer[o].
template <int PHASE>
__global__ void __launch_bounds__(256) latent_fwd_kernel(const __grid_constant__ LatentLayers L, int64_t B,
                                                        const float* __restrict__ shape_latent,
                                                        const float* __restrict__ texture_latent,
                                                        float* __restrict__ zlat, float* __restrict__ ebias,
                                                        uint8_t* __restrict__ eimg) {
  const int slot = blockIdx.x;
  const int64_t b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int o = blockIdx.z * 8 + warp;
  if (o >= L.W) return;
  const int K = PHASE == 0 ? L.D : L.W;
  const float* x = PHASE == 0 ? (slot < L.n_shape ? shape_latent : texture_latent) + b * L.D
                              : zlat + ((size_t)slot * B + b) * L.W;
  const float* w = (PHASE == 0 ? L.wl[slot] : L.wc[slot]) + (size_t)o * K;
  float acc = 0.f;
  if ((((uintptr_t)w | (uintptr_t)x) & 15) == 0) {
    for (int k = lane * 4; k < K; k += 128) {   // K is a multiple of 4 (checked on the host)
      const float4 a = __ldg(reinterpret_cast<const float4*>(w + k));
      const float4 v = *reinterpret_cast<const float4*>(x + k);
      acc = fmaf(a.x, v.x, acc); acc = fmaf(a.y, v.y, acc); acc = fmaf(a.z, v.z, acc); acc = fmaf(a.w, v.w, acc);
    }
  } else {   // caller handed an unaligned view
    for (int k = lane; k < K; k += 32) acc = fmaf(__ldg(w + k), x[k], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (PHASE == 0) zlat[((size_t)slot * B + b) * L.W + o] = fmaxf(acc + __ldg(L.bl[slot] + o), 0.f);
    else {
      const float eb = acc + __ldg(L.bc[slot] + o);
      ebias[((size_t)slot * B + b) * L.W + o] = eb;
      if (eimg != nullptr) tc::bias_stage_row(eimg + (((size_t)slot * B + b) * L.W + o) * 32, eb);   // tcgen05 bias-stage image
    }
  }
}

// grid (2, B, D/32): type 0 = shape slots, 1 = texture slots; the block owns 32 latent units, its 32 warps split the W
// hidden units of every slot (8 independent loads in flight per lane), partial sums meet in shared memory.
// dz [slot][b][W] = d loss / d z (post-ReLU).
__global__ void __launch_bounds__(1024) latent_bwd_kernel(const __grid_constant__ LatentLayers L, int64_t B,
                                                         const float* __restrict__ zlat, const float* __restrict__ dz,
                                                         float* __restrict__ g_shape, float* __restrict__ g_texture) {
  __shared__ float part[32][33];
  const int type = blockIdx.x;
  const int64_t b = blockIdx.y;
  float* out = type == 0 ? g_shape : g_texture;
  if (out == nullptr) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = blockIdx.z * 32 + lane;
  const int s0 = type == 0 ? 0 : L.n_shape, s1 = type == 0 ? L.n_shape : L.n_total;
  float acc = 0.f;
  if (k < L.D) {
    for (int slot = s0; slot < s1; ++slot) {
      const float* z = zlat + ((size_t)slot * B + b) * L.W;
      const float* g = dz + ((size_t)slot * B + b) * L.W;
      const float* w = L.wl[slot] + k;
      for (int o0 = warp; o0 < L.W; o0 += 32 * 8) {
        float wv[8], gm[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int o = o0 + 32 * u;
          const bool ok = o < L.W;
          wv[u] = ok ? __ldg(w + (size_t)o * L.D) : 0.f;
          gm[u] = (ok && z[o] > 0.f) ? g[o] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) acc = fmaf(gm[u], wv[u], acc);
      }
    }
  }
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && k < L.D) {
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) v += part[i][lane];
    out[b * L.D + k] = v;
  }
}

// The two-tile tcgen05 backward hands over s[slot][b][o] = sum_samples d loss / d pre-activation of the CONSUMING layer
// (column sums of its A operand).  Fold it through that layer once per object:  dz[slot][b][i] = sum_o Wc[o][i] s[o]
// (= sum_samples d loss / d (x + z), what latent_bwd_kernel expects).  grid (slots, B, W/32), 32 warps split o.
__global__ void __launch_bounds__(1024) latent_fold_kernel(const __grid_constant__ LatentLayers L, int64_t B,
                                                          const float* __restrict__ s, float* __restrict__ dz) {
  __shared__ float part[32][33];
  const int slot = blockIdx.x;
  const int64_t b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.z * 32 + lane;
  const float* sv = s + ((size_t)slot * B + b) * L.W;
  const float* w = L.wc[slot] + i;
  float acc = 0.f;
  if (i < L.W) {
    for (int o0 = warp; o0 < L.W; o0 += 32 * 8) {
      float wv[8], gv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int o = o0 + 32 * u;
        const bool ok = o < L.W;
        wv[u] = ok ? __ldg(w + (size_t)o * L.W) : 0.f;
        gv[u] = ok ? sv[o] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) acc = fmaf(gv[u], wv[u], acc);
    }
  }
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && i < L.W) {
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) v += part[k][lane];
    dz[((size_t)slot * B + b) * L.W + i] = v;
  }
}

static int fill_layers(const snb_handle_s* h, LatentLayers& L) {
  L.n_shape = h->arch.shape_blocks;
  L.n_total = h->arch.shape_blocks + h->arch.texture_blocks;
  L.W = h->arch.W; L.D = h->arch.latent_dim;
  SNB_REQUIRE(L.n_total <= kMaxSlots && L.D <= 1024, "latent layers: too many blocks or latent_dim > 1024");
  for (int j = 1; j <= L.n_total; ++j) {
    const bool s = j <= L.n_shape;
    const int ll = s ? h->iSL(j) : h->iTL(j - L.n_shape), lc = s ? h->iS(j) : h->iT(j - L.n_shape);
    L.wl[j - 1] = h->layers[ll].w; L.bl[j - 1] = h->layers[ll].b;
    L.wc[j - 1] = h->layers[lc].w; L.bc[j - 1] = h->layers[lc].b;
  }
  return 0;
}

int latent_forward_fused(const snb_handle_s* h, int64_t B, const float* shape_latent, const float* texture_latent,
                         float* zlat, float* ebias, cudaStream_t st, uint8_t* eimg) {
  LatentLayers L;
  if (fill_layers(h, L)) return 2;
  SNB_REQUIRE(L.D % 4 == 0 && L.W % 4 == 0, "latent layers: latent_dim and W must be multiples of 4");
  dim3 grid(L.n_total, (unsigned)B, (unsigned)((L.W + 7) / 8));
  latent_fwd_kernel<0><<<grid, 256, 0, st>>>(L, B, shape_latent, texture_latent, zlat, ebias, nullptr);
  SNB_LAUNCH_CHECK();
  if (ebias != nullptr) {
    latent_fwd_kernel<1><<<grid, 256, 0, st>>>(L, B, shape_latent, texture_latent, zlat, ebias, eimg);
    SNB_LAUNCH_CHECK();
  }
  return 0;
}

int latent_backward_fused(const snb_handle_s* h, int64_t B, const float* zlat, const float* dz, float* g_shape_latent,
                          float* g_texture_latent, cudaStream_t st, float* fold_tmp) {
  LatentLayers L;
  if (fill_layers(h, L)) return 2;
  if (fold_tmp != nullptr) {   // dz holds pre-activation column sums of the consuming layers: fold through W^T first
    dim3 gridf(L.n_total, (unsigned)B, (unsigned)((L.W + 31) / 32));
    latent_fold_kernel<<<gridf, 1024, 0, st>>>(L, B, dz, fold_tmp);
    SNB_LAUNCH_CHECK();
    dz = fold_tmp;
  }
  dim3 grid(2, (unsigned)B, (unsigned)((L.D + 31) / 32));
  latent_bwd_kernel<<<grid, 1024, 0, st>>>(L, B, zlat, dz, g_shape_latent, g_texture_latent);
  SNB_LAUNCH_CHECK();
  return 0;
}

}  // namespace snb
