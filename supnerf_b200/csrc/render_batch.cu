// Batched fused box render: ONE launch set for B objects (config C2: 16 objects x 128x128 rays x 64 samples per step).
//
// The per-object entry points of render.cu enqueue ~24 launches per object (the step of configs[1] was host-bound: 384 launches,
// profiles/r1_launches_v29.md).  Here every stage runs once over all objects:
//
//   forward   rb_setup      (B*N rays)   pixel -> ray (utils.get_rays, utils.py:107-135), origin / (diag/2), slab test
//                                         (utils.py:283-327) -> rays8 = {o, d, near, far} (the reference's `rays`, renderer.py:103-110) + hit
//             rb_plan       (B blocks)   per object: hit rays first, then miss rays (compact.cu's plan); the last block turns the
//                                         per-object row counts (S rows per hit ray + ONE per miss ray, padded to 256) into row / tile offsets
//             rb_gather     (rows)       compact row -> stratified sample (renderer.py:27-41, :111-114): xyz, viewdir, z_vals of the
//                                         EXECUTED rows only (no dense (N,S,3) tensors exist)
//             latent layers + tcgen05 decoder over all objects' rows (mlp_tc2.cu: per-tile object lookup through tile_start)
//             rb_composite_fwd           compositing straight on the compact rows (hit rays: S-sample scan; miss rays: their single
//                                         sample in closed form) -> rgb / depth / acc per ray
//   backward  rb_composite_bwd (+ the list of live super tiles) -> decoder backward over the live super tiles only -> rb_rays_bwd
//             (per-ray fold of d xyz / d viewdir / d z through the sampler, the slab test and get_rays; per-object fp64 block sums
//             -> d cam_pose (B,3,4))
//
// Frozen weights, bf16 decoder (two-tile kernels).
#include "common.cuh"
#include "compact.h"
#include "decoder.h"
#include "sampler.cuh"
#include "composite.cuh"
#include "rb_rows.cuh"

namespace snb {
namespace rb {

struct Meta { int64_t total_rows; unsigned int done, pad; };

constexpr int kMaxObjs = 1024;

// --------------------------------------------------------------------------------------------------------------- setup
__global__ void __launch_bounds__(256) rb_setup_kernel(const float* __restrict__ px, const float* __restrict__ py,
                                                      const float* __restrict__ K, const float* __restrict__ c2w,
                                                      const float* __restrict__ box, int64_t N, int64_t total,
                                                      float* __restrict__ rays8, uint8_t* __restrict__ hit) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / N;
    const float* P = c2w + 12 * b;
    const float* bx = box + 4 * b;
    float o[3], d[3];
    pixel_dir(K + 9 * b, P, __ldg(px + i), __ldg(py + i), d);
    const float half_diag = __ldg(bx);
    const float half[3] = {__ldg(bx + 1), __ldg(bx + 2), __ldg(bx + 3)};
#pragma unroll
    for (int a = 0; a < 3; ++a) o[a] = __fdiv_rn(__ldg(P + 4 * a + 3), half_diag);   // rays_o / (obj_diag / 2), renderer.py:102
    const Slab sl = slab_test(o, d, half);
    float4* dst = reinterpret_cast<float4*>(rays8 + 8 * i);
    dst[0] = make_float4(o[0], o[1], o[2], d[0]);
    dst[1] = make_float4(d[1], d[2], sl.hit ? sl.t_near : -1.f, sl.hit ? sl.t_far : -1.f);
    hit[i] = sl.hit ? 1 : 0;
  }
}

// --------------------------------------------------------------------------------------------------------------- plan
// block b: object b's rays ranked hit-first (compact.h); the last block to finish makes the row offsets: object b owns rows
// [row_start, row_start + rows) of the decoder's input, padded to 256 (one cta_group::2 super tile)
__global__ void __launch_bounds__(1024) rb_plan_kernel(const uint8_t* __restrict__ hit_all, int64_t N, int S, int B,
                                                      int32_t* __restrict__ order_all, int32_t* __restrict__ pos_all,
                                                      ObjCounts* __restrict__ counts, int32_t* __restrict__ tile_start,
                                                      Meta* __restrict__ meta) {
  const int b = blockIdx.x;
  const int n_hit = rank_hits_first(hit_all + (int64_t)b * N, N, order_all + (int64_t)b * N, pos_all + (int64_t)b * N);
  __syncthreads();
  if (threadIdx.x == 0) {
    const int64_t n_miss = N - n_hit;
    counts[b].n_hit = n_hit; counts[b].n_miss = n_miss; counts[b].rows = (int64_t)n_hit * S + n_miss;
    __threadfence();
    const unsigned t = atomicAdd(&meta->done, 1u);
    if (t == gridDim.x - 1) {
      __threadfence();
      int64_t acc = 0;
      for (int j = 0; j < B; ++j) {
        const int64_t rows = *reinterpret_cast<volatile int64_t*>(&counts[j].rows);
        counts[j].row_start = acc;
        tile_start[j] = (int32_t)(acc / 128);
        acc += (rows + 255) / 256 * 256;
      }
      tile_start[B] = (int32_t)(acc / 128);
      meta->total_rows = acc;
    }
  }
}

__global__ void __launch_bounds__(256) rb_gather_kernel(const float* __restrict__ rays8, const float* __restrict__ box,
                                                       const float* __restrict__ z_steps, const float* __restrict__ jitter,
                                                       const int32_t* __restrict__ order_all, const ObjCounts* __restrict__ counts,
                                                       const Meta* __restrict__ meta, int B, int64_t N, int S,
                                                       float* __restrict__ xyz_c, float* __restrict__ vrep_c, float* __restrict__ z_c) {
  const int64_t total = meta->total_rows;
  const float fstep = (float)(1.0 / (double)S);
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < total; r += (int64_t)gridDim.x * blockDim.x) {
    const int b = obj_of_row(counts, B, r);
    const ObjCounts c = counts[b];
    int64_t ray; int k;
    row_source(c, order_all + (int64_t)b * N, r - c.row_start, S, &ray, &k);
    const int64_t gi = (int64_t)b * N + ray;
    const SamplePt s = sample_point(rays8 + 8 * gi, __ldg(z_steps + k), __ldg(jitter + gi * S + k), fstep, __ldg(box + 4 * b));
#pragma unroll
    for (int a = 0; a < 3; ++a) { xyz_c[3 * r + a] = s.x[a]; vrep_c[3 * r + a] = s.d[a]; }
    z_c[r] = s.zv;
  }
}

// --------------------------------------------------------------------------------------------------------------- live super tiles
// The decoder backward is linear in (g_sigma, g_rgb) of a row: a 256-row super tile whose rows all have exactly zero upstream
// gradients (rays the loss gives no weight, e.g. occ == 0 in the refine loss; pad rows) has exactly zero outputs.  The compositing
// backward sets one flag byte per super tile that has a nonzero (or NaN) upstream gradient; its last block lists the flagged super
// tiles in ascending order for the decoder backward, which runs only those.  All on the device: a captured graph replays it as is.
struct LiveHdr { int32_t n_live; unsigned int ticket; };

// rows `row` of the calling lanes: flag their super tiles where nz; one store per warp and super tile
__device__ __forceinline__ void mark_live(uint8_t* __restrict__ live, int64_t row, bool nz) {
  const unsigned am = __activemask();
  const unsigned lv = __ballot_sync(am, nz);
  if (lv == 0u) return;
  const unsigned sup = (unsigned)(row >> 8);
  const unsigned peers = __match_any_sync(am, sup) & lv;
  if (nz && (unsigned)(__ffs(peers) - 1) == (threadIdx.x & 31u)) live[sup] = 1;
}

// one block of 256 threads: the flagged super tiles of [0, total_rows / 256), ascending -> list, their count -> hdr->n_live.  Each
// thread counts a contiguous run of 4-flag words (a flag byte is 0 or 1), one block scan, then each thread writes its run's entries.
__device__ void build_live_list(const uint8_t* __restrict__ live, int64_t total_rows, int32_t* __restrict__ list, LiveHdr* hdr) {
  __shared__ int warp_tot[8];
  const int n_words = (int)(((total_rows >> 8) + 3) >> 2);
  const int per = (n_words + 255) / 256;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int w0 = tid * per, w1 = min(w0 + per, n_words);
  const unsigned int* words = reinterpret_cast<const unsigned int*>(live);
  int cnt = 0;
  for (int w = w0; w < w1; ++w) cnt += __popc(__ldcg(words + w));
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int before = incl - cnt, total = 0;
  for (int k = 0; k < 8; ++k) { if (k < warp) before += warp_tot[k]; total += warp_tot[k]; }
  for (int w = w0; w < w1; ++w) {
    const unsigned int f = __ldcg(words + w);
#pragma unroll
    for (int b = 0; b < 4; ++b)
      if ((f >> (8 * b)) & 1u) list[before++] = 4 * w + b;
  }
  if (tid == 0) hdr->n_live = total;
}

// --------------------------------------------------------------------------------------------------------------- compositing
// z_vals of a lane's 4 samples (+ the next one) recomputed from the ray: the forward keeps no per-row coordinates or depths in HBM
__device__ __forceinline__ void lane_z_from_ray(const float* __restrict__ r8, const float* __restrict__ jit_row, const float* __restrict__ z_steps,
                                                int k0, int S, float fstep, float half_diag, float (&z)[5]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(r8)), b = __ldg(reinterpret_cast<const float4*>(r8) + 1);
  const float o[3] = {a.x, a.y, a.z}, d[3] = {a.w, b.x, b.y};
  if (k0 < S) {
    const float4 j4 = __ldg(reinterpret_cast<const float4*>(jit_row + k0)), s4 = __ldg(reinterpret_cast<const float4*>(z_steps + k0));
    z[0] = sample_zv(o, d, b.z, b.w, s4.x, j4.x, fstep, half_diag);
    z[1] = sample_zv(o, d, b.z, b.w, s4.y, j4.y, fstep, half_diag);
    z[2] = sample_zv(o, d, b.z, b.w, s4.z, j4.z, fstep, half_diag);
    z[3] = sample_zv(o, d, b.z, b.w, s4.w, j4.w, fstep, half_diag);
    z[4] = (k0 + 4 < S) ? sample_zv(o, d, b.z, b.w, __ldg(z_steps + k0 + 4), __ldg(jit_row + k0 + 4), fstep, half_diag) : 0.f;
  } else {
#pragma unroll
    for (int j = 0; j < 5; ++j) z[j] = 0.f;
  }
}

struct ZSrc {   // z_c != NULL: depths of the compact rows are read; else recomputed from the rays
  const float* z_c; const float* rays8; const float* box; const float* z_steps; const float* jitter;
};

template <int LPR>
__global__ void __launch_bounds__(256) rb_composite_fwd_kernel(const float* __restrict__ sigma_c, const float* __restrict__ rgb_c,
                                                              const ZSrc zs, const int32_t* __restrict__ order_all,
                                                              const ObjCounts* __restrict__ counts, int64_t N, int S, int flags,
                                                              float* __restrict__ out_rgb, float* __restrict__ out_depth,
                                                              float* __restrict__ out_acc) {
  const float* __restrict__ z_c = zs.z_c;
  const float fstep = (float)(1.0 / (double)S);
  constexpr int RPW = 32 / LPR;
  const int b = blockIdx.y;
  const ObjCounts c = counts[b];
  const int32_t* order = order_all + (int64_t)b * N;
  const int lane = threadIdx.x & 31, sl = lane % LPR, sub = lane / LPR;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool relu = flags & SNB_SIGMA_RELU, white = flags & SNB_WHITE_BKGD;
  const int k0 = sl * 4;
  for (int64_t seg0 = warp * RPW; seg0 < c.n_hit; seg0 += nwarps * RPW) {      // hit rays: S rows each
    const int64_t seg = seg0 + sub;
    const bool rv = seg < c.n_hit;
    const int64_t rr = rv ? seg : c.n_hit - 1;
    const int64_t row0 = c.row_start + rr * S;
    Lane4 L = load_lane4<LPR>(sigma_c + row0, rgb_c + row0 * 3, z_c ? z_c + row0 : nullptr, k0, S);
    if (z_c == nullptr) {
      const int64_t gi = (int64_t)b * N + order[rr];
      lane_z_from_ray(zs.rays8 + 8 * gi, zs.jitter + gi * S, zs.z_steps, k0, S, fstep, __ldg(zs.box + 4 * b), L.z);
    }
    float al[4], tl[4], tp = 1.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      SampleTerms q = sample_terms(L.s[j], L.z[j], L.z[j + 1], k0 + j == S - 1, relu);
      if (!L.valid) { q.alpha = 0.f; q.t = 1.f; }
      al[j] = q.alpha; tl[j] = tp; tp *= q.t;
    }
    float total;
    const float T0 = seg_excl_prod<LPR>(tp, sl, &total);
    float ar = 0.f, ag = 0.f, ab = 0.f, ad = 0.f, aw = 0.f, A = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float T = T0 * tl[j];
      const float w = al[j] * T;
      ar += w * L.c[j][0]; ag += w * L.c[j][1]; ab += w * L.c[j][2]; ad += w * L.z[j]; aw += w;
      if (k0 + j == S - 1) A = T;
    }
    ar = seg_sum<LPR>(ar); ag = seg_sum<LPR>(ag); ab = seg_sum<LPR>(ab); ad = seg_sum<LPR>(ad); aw = seg_sum<LPR>(aw);
    A = __shfl_sync(0xffffffffu, A, (S - 1) / 4, LPR);
    if (sl == 0 && rv) {
      const int64_t ray = (int64_t)b * N + order[rr];
      if (white) { ar = ar + 1.f - aw; ag = ag + 1.f - aw; ab = ab + 1.f - aw; }
      out_rgb[ray * 3 + 0] = ar; out_rgb[ray * 3 + 1] = ag; out_rgb[ray * 3 + 2] = ab;
      out_depth[ray] = ad;
      out_acc[ray] = A;
    }
  }
  // miss rays: S samples at ONE point => deltas 0 (alpha 0, t = 1 + 1e-10 = 1 in fp32) up to the last sample (delta 1e10)
  const int64_t mbase = c.row_start + c.n_hit * S;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < c.n_miss; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = mbase + j;
    const int64_t ray = (int64_t)b * N + order[c.n_hit + j];
    float zk;
    if (z_c != nullptr) zk = __ldg(z_c + row);
    else zk = sample_point(zs.rays8 + 8 * ray, __ldg(zs.z_steps + S - 1), __ldg(zs.jitter + ray * S + S - 1), fstep, __ldg(zs.box + 4 * b)).zv;
    const SampleTerms q = sample_terms(__ldg(sigma_c + row), zk, 0.f, true, relu);
    const float w = q.alpha;   // T = 1
    float cr = w * __ldg(rgb_c + 3 * row), cg = w * __ldg(rgb_c + 3 * row + 1), cb = w * __ldg(rgb_c + 3 * row + 2);
    if (white) { cr = cr + 1.f - w; cg = cg + 1.f - w; cb = cb + 1.f - w; }
    out_rgb[ray * 3 + 0] = cr; out_rgb[ray * 3 + 1] = cg; out_rgb[ray * 3 + 2] = cb;
    out_depth[ray] = w * zk;
    out_acc[ray] = 1.f;
  }
}

template <int LPR>
__global__ void __launch_bounds__(256) rb_composite_bwd_kernel(const float* __restrict__ sigma_c, const float* __restrict__ rgb_c,
                                                              const float* __restrict__ z_c, const int32_t* __restrict__ order_all,
                                                              const ObjCounts* __restrict__ counts, int64_t N, int S, int flags,
                                                              const float* __restrict__ g_rgb, const float* __restrict__ g_depth,
                                                              const float* __restrict__ g_acc, float* __restrict__ g_sigma_c,
                                                              float* __restrict__ g_rgb_c, float* __restrict__ g_z_c,
                                                              const int64_t* __restrict__ total_rows, uint8_t* __restrict__ live,
                                                              int32_t* __restrict__ live_list, LiveHdr* __restrict__ live_hdr) {
  constexpr int RPW = 32 / LPR;
  const int b = blockIdx.y;
  const ObjCounts c = counts[b];
  const int32_t* order = order_all + (int64_t)b * N;
  const int lane = threadIdx.x & 31, sl = lane % LPR, sub = lane / LPR;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool relu = flags & SNB_SIGMA_RELU, white = flags & SNB_WHITE_BKGD;
  const int k0 = sl * 4;
  for (int64_t seg0 = warp * RPW; seg0 < c.n_hit; seg0 += nwarps * RPW) {
    const int64_t seg = seg0 + sub;
    const bool rv = seg < c.n_hit;
    const int64_t rr = rv ? seg : c.n_hit - 1;
    const int64_t row0 = c.row_start + rr * S;
    const int64_t ray = (int64_t)b * N + order[rr];
    const Lane4 L = load_lane4<LPR>(sigma_c + row0, rgb_c + row0 * 3, z_c + row0, k0, S);
    const float gc0 = __ldg(g_rgb + ray * 3), gc1 = __ldg(g_rgb + ray * 3 + 1), gc2 = __ldg(g_rgb + ray * 3 + 2);
    const float gD = g_depth ? __ldg(g_depth + ray) : 0.f, gA = g_acc ? __ldg(g_acc + ray) : 0.f;
    const float gsum = gc0 + gc1 + gc2;
    SampleTerms q[4];
    float tl[4], tp = 1.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      q[j] = sample_terms(L.s[j], L.z[j], L.z[j + 1], k0 + j == S - 1, relu);
      if (!L.valid) { q[j].alpha = 0.f; q[j].t = 1.f; }
      tl[j] = tp; tp *= q[j].t;
    }
    float total;
    const float T0 = seg_excl_prod<LPR>(tp, sl, &total);
    float T[4], w[4], gw[4], x[4], A = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      T[j] = T0 * tl[j];
      w[j] = q[j].alpha * T[j];
      gw[j] = gc0 * L.c[j][0] + gc1 * L.c[j][1] + gc2 * L.c[j][2] + gD * L.z[j];
      if (white) gw[j] -= gsum;
      x[j] = L.valid ? gw[j] * w[j] : 0.f;
      if (k0 + j == S - 1) A = T[j];
    }
    A = __shfl_sync(0xffffffffu, A, (S - 1) / 4, LPR);
    const float gAA = gA * A;
    const float later = seg_rev_excl_sum<LPR>((x[0] + x[1]) + (x[2] + x[3]), sl);
    float suf[4];
    suf[3] = later; suf[2] = suf[3] + x[3]; suf[1] = suf[2] + x[2]; suf[0] = suf[1] + x[1];
    float gs[4], gdel[4], gcol[4][3];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool last = (k0 + j == S - 1);
      const float g_t = (suf[j] + (last ? 0.f : gAA)) / q[j].t;
      const float g_alpha = gw[j] * T[j] - g_t;
      gs[j] = g_alpha * q[j].delta * q[j].e;
      if (relu && !(L.s[j] > 0.f)) gs[j] = 0.f;
      gdel[j] = (last || !L.valid) ? 0.f : g_alpha * q[j].sr * q[j].e;
      gcol[j][0] = w[j] * gc0; gcol[j][1] = w[j] * gc1; gcol[j][2] = w[j] * gc2;
    }
    float gprev = __shfl_up_sync(0xffffffffu, gdel[3], 1, LPR);
    if (sl == 0) gprev = 0.f;
    bool nz = false;   // the lane's 4 rows (one super tile: rows start at multiples of 4) feed the decoder a nonzero gradient
#pragma unroll
    for (int j = 0; j < 4; ++j) nz |= (gs[j] != 0.f) | (gcol[j][0] != 0.f) | (gcol[j][1] != 0.f) | (gcol[j][2] != 0.f);
    mark_live(live, row0 + k0, nz && L.valid && rv);
    if (L.valid && rv) {
      *reinterpret_cast<float4*>(g_sigma_c + row0 + k0) = make_float4(gs[0], gs[1], gs[2], gs[3]);
      float* gr = g_rgb_c + (row0 + k0) * 3;
      *reinterpret_cast<float4*>(gr) = make_float4(gcol[0][0], gcol[0][1], gcol[0][2], gcol[1][0]);
      *reinterpret_cast<float4*>(gr + 4) = make_float4(gcol[1][1], gcol[1][2], gcol[2][0], gcol[2][1]);
      *reinterpret_cast<float4*>(gr + 8) = make_float4(gcol[2][2], gcol[3][0], gcol[3][1], gcol[3][2]);
      if (g_z_c != nullptr) {
        *reinterpret_cast<float4*>(g_z_c + row0 + k0) =
            make_float4(w[0] * gD + gprev - gdel[0], w[1] * gD + gdel[0] - gdel[1], w[2] * gD + gdel[1] - gdel[2],
                        w[3] * gD + gdel[2] - gdel[3]);
      }
    }
  }
  // miss rays (one row each, the ray's last sample: weight alpha, transmittance 1, no later sample), then the zero padding
  const int64_t mbase = c.row_start + c.n_hit * S;
  const int64_t n_tail = (c.rows + 255) / 256 * 256 - c.n_hit * S;    // miss rows + pad rows
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_tail; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = mbase + j;
    float gs = 0.f, r0 = 0.f, r1 = 0.f, r2 = 0.f, gz = 0.f;
    if (j < c.n_miss) {
      const int64_t ray = (int64_t)b * N + order[c.n_hit + j];
      const float s = __ldg(sigma_c + row), zk = __ldg(z_c + row);
      const SampleTerms q = sample_terms(s, zk, 0.f, true, relu);
      const float gc0 = __ldg(g_rgb + ray * 3), gc1 = __ldg(g_rgb + ray * 3 + 1), gc2 = __ldg(g_rgb + ray * 3 + 2);
      const float gD = g_depth ? __ldg(g_depth + ray) : 0.f;
      float gw = gc0 * __ldg(rgb_c + 3 * row) + gc1 * __ldg(rgb_c + 3 * row + 1) + gc2 * __ldg(rgb_c + 3 * row + 2) + gD * zk;
      if (white) gw -= gc0 + gc1 + gc2;
      gs = gw * q.delta * q.e;                   // g_alpha = gw * T - 0, T = 1
      if (relu && !(s > 0.f)) gs = 0.f;
      const float w = q.alpha;
      r0 = w * gc0; r1 = w * gc1; r2 = w * gc2; gz = w * gD;
    }
    g_sigma_c[row] = gs;
    g_rgb_c[3 * row] = r0; g_rgb_c[3 * row + 1] = r1; g_rgb_c[3 * row + 2] = r2;
    if (g_z_c != nullptr) g_z_c[row] = gz;
    mark_live(live, row, (gs != 0.f) | (r0 != 0.f) | (r1 != 0.f) | (r2 != 0.f));
  }
  // the last block lists the live super tiles (every block's flags are visible: bar.sync, then a cumulative fence before the ticket)
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(&live_hdr->ticket, 1u) == gridDim.x * gridDim.y - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    build_live_list(live, *total_rows, live_list, live_hdr);
  }
}

// --------------------------------------------------------------------------------------------------------------- rays backward
// Object b's pose gradient from the per-thread fp64 sums acc (c2w layout) of a 256-thread block: one block reduction and one atomic
// per entry into acc64[12 b ..]; the object's last block (tickets[b]) writes the totals to g_c2w[12 b ..].
__device__ __forceinline__ void flush_pose_grad(const double acc[12], int b, double* __restrict__ acc64, unsigned int* __restrict__ tickets,
                                                float* __restrict__ g_c2w) {
  __shared__ double red[8][12];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    double v = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[wib][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    double v = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) v += red[k][threadIdx.x];
    atomicAdd(acc64 + 12 * b + threadIdx.x, v);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned t = atomicAdd(tickets + b, 1u);
    if (t == gridDim.x - 1) {     // the object's last block: every partial is visible
      __threadfence();
      for (int i = 0; i < 12; ++i) g_c2w[12 * b + i] = (float)atomicAdd(acc64 + 12 * b + i, 0.0);
    }
  }
}

// d xyz / d viewdir / d z_vals of a ray's compact rows -> d (o, d, near, far) -> through the slab test -> d (rays_o, viewdir) ->
// through get_rays -> this object's d cam_pose (12 fp64 sums per thread, one block reduction + one atomic each per block).
// Two phases per group of 32 rays of a warp: (1) the warp walks its 32 rays one after the other, lanes over the ray's samples, and
// lane j keeps the nine sums of ray j; (2) every lane finishes ITS ray (slab backward, normalisation Jacobian, outer products) -- the
// per-ray tail is ~400 instructions, which a warp-per-ray layout would issue for one active lane (measured: 672 warp instructions
// per ray, 0.42 ms per 262 144 rays; this layout: ~60).
__global__ void __launch_bounds__(256) rb_rays_bwd_kernel(const float* __restrict__ px, const float* __restrict__ py,
                                                         const float* __restrict__ K, const float* __restrict__ c2w,
                                                         const float* __restrict__ box, const float* __restrict__ rays8,
                                                         const uint8_t* __restrict__ hit, const int32_t* __restrict__ pos_all,
                                                         const ObjCounts* __restrict__ counts, const float* __restrict__ z_steps,
                                                         const float* __restrict__ jitter, int64_t N, int S,
                                                         const float* __restrict__ g_xyz_c, const float* __restrict__ g_vrep_c,
                                                         const float* __restrict__ g_z_c, const uint8_t* __restrict__ live,
                                                         double* __restrict__ acc64, unsigned int* __restrict__ tickets,
                                                         float* __restrict__ g_c2w) {
  const int b = blockIdx.y;
  const ObjCounts c = counts[b];
  const float half_diag = __ldg(box + 4 * b);
  const float half[3] = {__ldg(box + 4 * b + 1), __ldg(box + 4 * b + 2), __ldg(box + 4 * b + 3)};
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const float fstep = (float)(1.0 / (double)S);
  double acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.0;
  for (int64_t base = (int64_t)blockIdx.x * 256 + wib * 32; base < N; base += (int64_t)gridDim.x * 256) {
    // ---- phase 1: the warp's 32 rays, FOUR at a time: 8 lanes walk one ray's samples, a 3-step butterfly inside the group sums them,
    // one shuffle hands ray j's sums to lane j (the first version walked one ray per iteration with a 5-step butterfly over 32 lanes:
    // 224 warp instructions per ray, 198 us per step)
    float k_gon[3] = {0.f, 0.f, 0.f}, k_gd[3] = {0.f, 0.f, 0.f}, k_gzabs = 0.f, k_gnear = 0.f, k_gfar = 0.f;
    const int n_here = (int)((N - base) < 32 ? (N - base) : 32);
    const int grp = lane >> 3, l8 = lane & 7;
    for (int jj = 0; jj < n_here; jj += 4) {
      const int j = jj + grp;
      float v[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // gon[3], gd[3], gzabs, gnear, gfar of ray j (this lane's share)
      if (j < n_here) {
        const int64_t gi = (int64_t)b * N + base + j;
        const float4 ra = __ldg(reinterpret_cast<const float4*>(rays8 + 8 * gi)), rb_ = __ldg(reinterpret_cast<const float4*>(rays8 + 8 * gi) + 1);
        const float d[3] = {ra.w, rb_.x, rb_.y};
        const bool h = hit[gi] != 0;
        const float near = rb_.z, far = rb_.w;
        const int p = pos_all[gi];
        const float dn = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        if (h) {
          for (int k = l8; k < S; k += 8) {
            const int64_t gidx = c.row_start + (int64_t)p * S + k;
            // a row of a super tile the decoder skipped has d xyz = d viewdir = 0 (its scratch rows hold an older call's values);
            // d z comes from the compositing backward and is always read.  Per row: a ray can span two super tiles.
            const bool lv = __ldg(live + (gidx >> 8)) != 0;
            fold_sample_grad(lv ? g_xyz_c + 3 * gidx : nullptr, lv ? g_vrep_c + 3 * gidx : nullptr, g_z_c ? g_z_c + gidx : nullptr,
                             __ldg(z_steps + k), __ldg(jitter + gi * S + k), fstep, near, far, d, dn, half_diag, v);
          }
        } else if (l8 == 0) {
          // a miss ray's single row stands for all its samples and is credited to the last one (k = S - 1)
          const int64_t gidx = c.row_start + c.n_hit * S + p;
          const bool lv = __ldg(live + (gidx >> 8)) != 0;
          fold_sample_grad(lv ? g_xyz_c + 3 * gidx : nullptr, lv ? g_vrep_c + 3 * gidx : nullptr, g_z_c ? g_z_c + gidx : nullptr,
                           __ldg(z_steps + S - 1), __ldg(jitter + gi * S + S - 1), fstep, near, far, d, dn, half_diag, v);
        }
      }
      const int src = ((lane - jj) & 3) * 8;            // lanes jj .. jj+3 take their ray's sums from the group that walked it
      const bool mine = (lane >> 2) == (jj >> 2);
#pragma unroll
      for (int i = 0; i < 9; ++i) {
        float t = v[i];
        t += __shfl_xor_sync(0xffffffffu, t, 1);
        t += __shfl_xor_sync(0xffffffffu, t, 2);
        t += __shfl_xor_sync(0xffffffffu, t, 4);
        t = __shfl_sync(0xffffffffu, t, src);
        if (mine) {
          if (i < 3) k_gon[i] = t; else if (i < 6) k_gd[i - 3] = t; else if (i == 6) k_gzabs = t; else if (i == 7) k_gnear = t; else k_gfar = t;
        }
      }
    }
    // ---- phase 2: every lane finishes its own ray
    if (lane < n_here) {
      const int64_t gi = (int64_t)b * N + base + lane;
      const float4 ra = __ldg(reinterpret_cast<const float4*>(rays8 + 8 * gi)), rb_ = __ldg(reinterpret_cast<const float4*>(rays8 + 8 * gi) + 1);
      const float o[3] = {ra.x, ra.y, ra.z}, d[3] = {ra.w, rb_.x, rb_.y};
      const bool h = hit[gi] != 0;
      const float dn = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
      float gon[3] = {k_gon[0], k_gon[1], k_gon[2]}, gd[3] = {k_gd[0], k_gd[1], k_gd[2]};
      if (dn > 0.f) {
#pragma unroll
        for (int a = 0; a < 3; ++a) gd[a] += k_gzabs * half_diag * d[a] / dn;
      }
      if (h) {
        const Slab sl = slab_test(o, d, half);
        const float lo[3] = {-half[0], -half[1], -half[2]};
        float go2[3], gd2[3], glo[3], ghi[3];
        slab_backward(sl, o, lo, half, k_gnear, k_gfar, go2, gd2, glo, ghi);
#pragma unroll
        for (int a = 0; a < 3; ++a) { gon[a] += go2[a]; gd[a] += gd2[a]; }
      }
      float pp[3], gr[3];
      dir_grad_to_pose(K + 9 * b, c2w + 12 * b, __ldg(px + gi), __ldg(py + gi), gd, pp, gr);
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        acc[4 * a + 0] += (double)(gr[a] * pp[0]);
        acc[4 * a + 1] += (double)(gr[a] * pp[1]);
        acc[4 * a + 2] += (double)(gr[a] * pp[2]);
        acc[4 * a + 3] += (double)(gon[a] / half_diag);
      }
    }
  }
  flush_pose_grad(acc, b, acc64, tickets, g_c2w);
}

// --------------------------------------------------------------------------------------------------------------- dataset-side ray prep
// SURVEY 8f rank 3: the samples a training batch needs -- utils.prepare_pixel_samples (utils.py:330-377) as the reference's DataLoader
// workers run it per object on the CPU (data_nuscenes.py:615-658), shipping (n_rays, S, 3) xyz + viewdir per object over PCIe --
// for B objects in one launch on the device: pixel -> ray (utils.get_rays), shared sample vector z_b (S) of the object (built on the host
// with the reference's torch calls, B x S floats), xyz = (o + d z) / obj_diag, optional y flip (sym_aug) and shapenet axis swap
// (utils.py:471-495).  One warp per ray, lanes over samples.  Same arithmetic as get_rays_fwd_kernel + sample_shell_fwd_kernel.
__global__ void __launch_bounds__(256) rb_shell_prep_kernel(const float* __restrict__ px, const float* __restrict__ py,
                                                           const float* __restrict__ K, const float* __restrict__ c2w,
                                                           const float* __restrict__ z, const float* __restrict__ obj_diag,
                                                           const int32_t* __restrict__ flip, int64_t n, int S, int swap, int64_t total,
                                                           float* __restrict__ xyz, float* __restrict__ vrep) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp; i < total; i += nwarps) {
    const int64_t b = i / n;
    const float* P = c2w + 12 * b;
    float o[3], d[3];
    pixel_dir(K + 9 * b, P, __ldg(px + i), __ldg(py + i), d);
#pragma unroll
    for (int a = 0; a < 3; ++a) o[a] = __ldg(P + 4 * a + 3);
    const float diag = __ldg(obj_diag + b);
    const float sy = (flip != nullptr && flip[b]) ? -1.f : 1.f;       // sym_aug: xyz[:, :, 1] *= -1, viewdir[:, :, 1] *= -1 (utils.py:474-477)
    const float* zb = z + b * S;
    for (int k = lane; k < S; k += 32) {
      const float zk = __ldg(zb + k);
      float x[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) x[a] = __fdiv_rn(__fadd_rn(o[a], __fmul_rn(d[a], zk)), diag);
      const float xy = x[1] * sy, dy = d[1] * sy;
      const int64_t idx = i * S + k;
      if (swap) {   // x' = (-y, x, z) (utils.py:492-495)
        xyz[3 * idx] = -xy; xyz[3 * idx + 1] = x[0]; xyz[3 * idx + 2] = x[2];
        vrep[3 * idx] = -dy; vrep[3 * idx + 1] = d[0]; vrep[3 * idx + 2] = d[2];
      } else {
        xyz[3 * idx] = x[0]; xyz[3 * idx + 1] = xy; xyz[3 * idx + 2] = x[2];
        vrep[3 * idx] = d[0]; vrep[3 * idx + 1] = dy; vrep[3 * idx + 2] = d[2];
      }
    }
  }
}

// Backward of rb_shell_prep_kernel through to the poses: per ray the fold of sample_shell_bwd_kernel (g_o = sum g_xyz / diag,
// g_d = sum z g_xyz / diag + sum g_viewdir, axis swap undone) and get_rays_bwd_kernel's g_r = (g_d - d (g_d . d)) / |r| (sampler.cu),
// then per-object fp64 block sums -> g_c2w (B,3,4), finished by the object's last block.  One warp per ray, lanes over samples; grid (x, B).
__global__ void __launch_bounds__(256) rb_shell_rays_bwd_kernel(const float* __restrict__ px, const float* __restrict__ py,
                                                               const float* __restrict__ K, const float* __restrict__ c2w,
                                                               const float* __restrict__ z, const float* __restrict__ obj_diag,
                                                               int64_t N, int S, int swap, const float* __restrict__ g_xyz,
                                                               const float* __restrict__ g_vrep, double* __restrict__ acc64,
                                                               unsigned int* __restrict__ tickets, float* __restrict__ g_c2w) {
  const int b = blockIdx.y;
  const float diag = __ldg(obj_diag + b);
  const float* zb = z + (int64_t)b * S;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.0;
  for (int64_t ray = (int64_t)blockIdx.x * 8 + wib; ray < N; ray += (int64_t)gridDim.x * 8) {
    const int64_t gi = (int64_t)b * N + ray;
    float go[3] = {0.f, 0.f, 0.f}, gd[3] = {0.f, 0.f, 0.f};
    for (int k = lane; k < S; k += 32) {
      const int64_t idx = gi * S + k;
      const float zk = __ldg(zb + k);
      float gx[3] = {__ldg(g_xyz + 3 * idx), __ldg(g_xyz + 3 * idx + 1), __ldg(g_xyz + 3 * idx + 2)};
      float gv[3] = {__ldg(g_vrep + 3 * idx), __ldg(g_vrep + 3 * idx + 1), __ldg(g_vrep + 3 * idx + 2)};
      if (swap) {  // out = (-in_y, in_x, in_z)
        float t0 = gx[1], t1 = -gx[0]; gx[0] = t0; gx[1] = t1;
        t0 = gv[1]; t1 = -gv[0]; gv[0] = t0; gv[1] = t1;
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float g = gx[a] / diag;
        go[a] += g; gd[a] += g * zk + gv[a];
      }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) { go[a] = warp_sum(go[a]); gd[a] = warp_sum(gd[a]); }
    if (lane == 0) {   // the other lanes' sums stay 0
      float pp[3], gr[3];
      dir_grad_to_pose(K + 9 * b, c2w + 12 * b, __ldg(px + gi), __ldg(py + gi), gd, pp, gr);
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        acc[4 * a + 0] += (double)(gr[a] * pp[0]);
        acc[4 * a + 1] += (double)(gr[a] * pp[1]);
        acc[4 * a + 2] += (double)(gr[a] * pp[2]);
        acc[4 * a + 3] += (double)go[a];
      }
    }
  }
  flush_pose_grad(acc, b, acc64, tickets, g_c2w);
}

}  // namespace rb

namespace {

inline size_t al(size_t bytes) { return (bytes + 255) & ~size_t(255); }

// the decoder precision of a batched render: frozen weights, bf16 or (SNB_BATCH_FP32_TC) split precision
inline int32_t batch_precision(const snb_batch_desc& d) { return (d.flags & SNB_BATCH_FP32_TC) ? SNB_PREC_FP32_TC : SNB_PREC_BF16; }

// forward workspace (kept for the backward).  Mmax = B * pad256(N * S): every object's rows if all of its rays hit.  With the fused
// sampler (SNB_BATCH_FUSED_SAMPLER) the forward keeps NO per-row coordinates: the decoder computes them from rays8 + jitter (K1), the
// compositing recomputes the depths, and the backward re-materialises them in its scratch
struct BatchLayout {
  size_t meta, counts, tile_start, rays8, hit, order, pos, xyz_c, vrep_c, z_c, sigma_c, rgb_c, mlp, total;
  int64_t Mmax;
  BatchLayout(snb_handle h, const snb_batch_desc& d) {
    const size_t B = (size_t)d.n_objs, N = (size_t)d.rays_per_obj, BN = B * N;
    Mmax = (int64_t)(B * ((N * (size_t)d.n_samples + 255) / 256 * 256));
    const size_t M = (size_t)Mmax;
    size_t o = 0;
    meta = o; o += al(sizeof(rb::Meta));
    counts = o; o += al(B * sizeof(rb::ObjCounts));
    tile_start = o; o += al((B + 1) * 4);
    rays8 = o; o += al(BN * 32);
    hit = o; o += al(BN);
    order = o; o += al(BN * 4);
    pos = o; o += al(BN * 4);
    const size_t Mc = (d.flags & SNB_BATCH_FUSED_SAMPLER) ? 0 : M;
    xyz_c = o; o += al(Mc * 12);
    vrep_c = o; o += al(Mc * 12);
    z_c = o; o += al(Mc * 4);
    sigma_c = o; o += al(M * 4);
    rgb_c = o; o += al(M * 12);
    mlp = o; o += al(decoder_workspace_bytes(h, batch_precision(d), Mmax, (int64_t)B));
    total = o;
  }
};

// backward scratch: the executed rows' coordinates and depths are re-materialised here (rb_gather_kernel: the decoder backward folds
// d PE through sin / cos of the coordinates), then the gradients, the live super tiles (header + one flag byte each, zeroed together;
// the list)
struct BatchScratch {
  size_t xyz_c, vrep_c, z_c, g_sigma_c, g_rgb_c, g_z_c, g_xyz_c, g_vrep_c, live_hdr, live, live_end, live_list, acc64, tickets, mlp, total;
  BatchScratch(snb_handle h, const snb_batch_desc& d, int64_t Mmax) {
    const size_t M = (size_t)Mmax, B = (size_t)d.n_objs;
    size_t o = 0;
    const size_t Mc = (d.flags & SNB_BATCH_FUSED_SAMPLER) ? M : 0;
    xyz_c = o; o += al(Mc * 12);
    vrep_c = o; o += al(Mc * 12);
    z_c = o; o += al(Mc * 4);
    g_sigma_c = o; o += al(M * 4);
    g_rgb_c = o; o += al(M * 12);
    g_z_c = o; o += al(M * 4);
    g_xyz_c = o; o += al(M * 12);
    g_vrep_c = o; o += al(M * 12);
    const size_t n_super = M / 256;
    live_hdr = o; o += al(sizeof(rb::LiveHdr));
    live = o; o += al(n_super);
    live_end = o;
    live_list = o; o += al(n_super * 4);
    acc64 = o; o += al(B * 12 * 8);
    tickets = o; o += al(B * 4);
    mlp = o; o += al(decoder_scratch_bytes(h, batch_precision(d), Mmax, (int64_t)B));
    total = o;
  }
};

int check_batch(snb_handle h, const snb_batch_desc* d, const char* who) {
  SNB_REQUIRE(h != nullptr && d != nullptr, "%s: null handle or descriptor", who);
  SNB_REQUIRE(d->n_objs >= 1 && d->n_objs <= rb::kMaxObjs && d->rays_per_obj >= 1, "%s: bad sizes", who);
  SNB_REQUIRE(d->n_samples >= 4 && d->n_samples % 4 == 0 && d->n_samples <= 128,
              "%s: the batched render needs n_samples in {4, 8, ..., 128} (vectorised compositing)", who);
  SNB_REQUIRE(d->rays_per_obj < ((int64_t)1 << 30) && d->rays_per_obj * d->n_samples < ((int64_t)1 << 31) &&
              (int64_t)d->n_objs * d->rays_per_obj < ((int64_t)1 << 31), "%s: too many rays", who);
  Backend be;
  SNB_REQUIRE(select_backend(h, batch_precision(*d), &be) == nullptr, "%s: the batched render runs on the tcgen05 decoder kernels "
              "(CodeNeRF family, W = 128 or 256, shape_blocks + texture_blocks <= 10); render the objects one by one for this architecture", who);
  if (d->flags & SNB_BATCH_FP32_TC)
    SNB_REQUIRE(!(d->flags & SNB_BATCH_FUSED_SAMPLER), "%s: SNB_BATCH_FP32_TC and SNB_BATCH_FUSED_SAMPLER exclude each other", who);
  if (d->flags & SNB_BATCH_FUSED_SAMPLER)
    SNB_REQUIRE(be == Backend::TwoTile, "%s: the fused sampler needs the two-tile kernels (shape_blocks + texture_blocks <= 4)", who);
  return 0;
}

template <typename T> inline T* at(void* base, size_t off) { return reinterpret_cast<T*>(static_cast<uint8_t*>(base) + off); }
template <typename T> inline const T* at(const void* base, size_t off) { return reinterpret_cast<const T*>(static_cast<const uint8_t*>(base) + off); }

// the compositing launches: LPR lanes per hit ray (4 samples each), 32 / LPR rays per warp, 8 warps per block; grid (x, objects)
struct CompositeGrid {
  int lpr;
  dim3 grid;
  CompositeGrid(int64_t N, int S, int B)
      : lpr(S <= 32 ? 8 : (S <= 64 ? 16 : 32)), grid((unsigned)grid_1d(N, 8 * (32 / lpr), 8, B), (unsigned)B) {}
};

}  // namespace
}  // namespace snb

using namespace snb;

extern "C" size_t snb_render_batch_workspace_bytes(snb_handle h, const snb_batch_desc* d) {
  if (!h || !d || d->n_objs < 1 || d->rays_per_obj < 1 || d->n_samples < 1) return 0;
  return BatchLayout(h, *d).total + 256;
}

extern "C" size_t snb_render_batch_scratch_bytes(snb_handle h, const snb_batch_desc* d) {
  if (!h || !d || d->n_objs < 1 || d->rays_per_obj < 1 || d->n_samples < 1) return 0;
  const BatchLayout L(h, *d);
  return BatchScratch(h, *d, L.Mmax).total + 256;
}

extern "C" int snb_render_batch_fwd(snb_handle h, const snb_batch_desc* d, const float* px, const float* py, const float* K,
                                    const float* c2w, const float* box, const float* z_steps, const float* jitter,
                                    const float* shape_latent, const float* texture_latent, float* out_rgb, float* out_depth,
                                    float* out_acc, uint8_t* out_hit, void* workspace, void* stream) {
  if (check_batch(h, d, "render_batch_fwd")) return 2;
  SNB_REQUIRE(px && py && K && c2w && box && z_steps && jitter && shape_latent && texture_latent && out_rgb && out_depth && out_acc &&
              workspace, "render_batch_fwd: null pointer");
  SNB_REQUIRE(((uintptr_t)workspace & 255) == 0, "render_batch_fwd: workspace must be 256-byte aligned");
  const BatchLayout L(h, *d);
  cudaStream_t st = (cudaStream_t)stream;
  void* ws = workspace;
  const int B = d->n_objs, S = d->n_samples;
  const int64_t N = d->rays_per_obj, BN = (int64_t)B * N;
  SNB_REQUIRE(sm_count() > 0, "render_batch_fwd: no CUDA device (there is no CPU fallback)");
  SNB_CHECK_CUDA(cudaMemsetAsync(at<uint8_t>(ws, L.meta), 0, sizeof(rb::Meta), st));
  rb::rb_setup_kernel<<<grid_1d(BN, 256, 8), 256, 0, st>>>(px, py, K, c2w, box, N, BN, at<float>(ws, L.rays8), at<uint8_t>(ws, L.hit));
  SNB_LAUNCH_CHECK();
  rb::rb_plan_kernel<<<B, 1024, 0, st>>>(at<uint8_t>(ws, L.hit), N, S, B, at<int32_t>(ws, L.order), at<int32_t>(ws, L.pos),
                                        at<rb::ObjCounts>(ws, L.counts), at<int32_t>(ws, L.tile_start), at<rb::Meta>(ws, L.meta));
  SNB_LAUNCH_CHECK();
  if (out_hit) SNB_CHECK_CUDA(cudaMemcpyAsync(out_hit, at<uint8_t>(ws, L.hit), (size_t)BN, cudaMemcpyDeviceToDevice, st));
  const bool fused = (d->flags & SNB_BATCH_FUSED_SAMPLER) != 0;
  rb::ZSrc zsrc{nullptr, at<float>(ws, L.rays8), box, z_steps, jitter};
  if (fused) {
    // K1: no sampler kernel on the forward path -- the decoder's epilogue warps compute every row's stratified sample from the ray
    // (32 B per ray) and its jitter (4 B per row) and build PE(xyz) / PE(viewdir) straight in shared memory; compositing recomputes z
    rb::RowSrc rs;
    rs.rays8 = at<float>(ws, L.rays8); rs.box = box; rs.z_steps = z_steps; rs.jitter = jitter; rs.order = at<int32_t>(ws, L.order);
    rs.counts = at<rb::ObjCounts>(ws, L.counts); rs.N = N; rs.S = S;
    if (decoder_forward(h, SNB_PREC_BF16, nullptr, nullptr, L.Mmax, B, shape_latent, texture_latent, at<float>(ws, L.sigma_c),
                        at<float>(ws, L.rgb_c), at<uint8_t>(ws, L.mlp), st,
                        {&at<rb::Meta>(ws, L.meta)->total_rows, at<int32_t>(ws, L.tile_start), &rs}))
      return 1;
  } else {
    // default: the stratified samples of the EXECUTED rows are written once (28 B per row) and read back by the decoder -- measured
    // faster than the fused sampler: the extra ~150 instructions per row sit on the decoder's critical tile-boundary chain
    rb::rb_gather_kernel<<<grid_1d(L.Mmax, 256, 8), 256, 0, st>>>(at<float>(ws, L.rays8), box, z_steps, jitter, at<int32_t>(ws, L.order),
                                                            at<rb::ObjCounts>(ws, L.counts), at<rb::Meta>(ws, L.meta), B, N, S,
                                                            at<float>(ws, L.xyz_c), at<float>(ws, L.vrep_c), at<float>(ws, L.z_c));
    SNB_LAUNCH_CHECK();
    if (decoder_forward(h, batch_precision(*d), at<float>(ws, L.xyz_c), at<float>(ws, L.vrep_c), L.Mmax, B, shape_latent, texture_latent,
                        at<float>(ws, L.sigma_c), at<float>(ws, L.rgb_c), at<uint8_t>(ws, L.mlp), st,
                        {&at<rb::Meta>(ws, L.meta)->total_rows, at<int32_t>(ws, L.tile_start)}))
      return 1;
    zsrc.z_c = at<float>(ws, L.z_c);
  }
  const CompositeGrid cg(N, S, B);
#define SNB_RBF(LL) rb::rb_composite_fwd_kernel<LL><<<cg.grid, 256, 0, st>>>(at<float>(ws, L.sigma_c), at<float>(ws, L.rgb_c), zsrc, \
    at<int32_t>(ws, L.order), at<rb::ObjCounts>(ws, L.counts), N, S, d->flags, out_rgb, out_depth, out_acc)
  if (cg.lpr == 8) SNB_RBF(8); else if (cg.lpr == 16) SNB_RBF(16); else SNB_RBF(32);
#undef SNB_RBF
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_render_batch_bwd(snb_handle h, const snb_batch_desc* d, const float* px, const float* py, const float* K,
                                    const float* c2w, const float* box, const float* z_steps, const float* jitter,
                                    const float* shape_latent, const float* texture_latent, const void* workspace,
                                    const float* g_rgb, const float* g_depth, const float* g_acc, void* scratch, float* g_c2w,
                                    float* g_shape_latent, float* g_texture_latent, void* stream) {
  if (check_batch(h, d, "render_batch_bwd")) return 2;
  SNB_REQUIRE(px && py && K && c2w && box && z_steps && jitter && shape_latent && texture_latent && workspace && g_rgb && scratch &&
              g_shape_latent && g_texture_latent, "render_batch_bwd: null pointer");
  SNB_REQUIRE((((uintptr_t)workspace | (uintptr_t)scratch) & 255) == 0, "render_batch_bwd: workspace/scratch must be 256-byte aligned");
  const BatchLayout L(h, *d);
  const BatchScratch G(h, *d, L.Mmax);
  cudaStream_t st = (cudaStream_t)stream;
  const void* ws = workspace;
  void* sc = scratch;
  const int B = d->n_objs, S = d->n_samples;
  const int64_t N = d->rays_per_obj;
  SNB_REQUIRE(sm_count() > 0, "render_batch_bwd: no CUDA device (there is no CPU fallback)");
  const bool pose = g_c2w != nullptr;
  const CompositeGrid cg(N, S, B);
  float* gz = pose ? at<float>(sc, G.g_z_c) : nullptr;
  const bool fused = (d->flags & SNB_BATCH_FUSED_SAMPLER) != 0;
  const float *xyz_c = at<float>(ws, L.xyz_c), *vrep_c = at<float>(ws, L.vrep_c), *z_c = at<float>(ws, L.z_c);
  if (fused) {   // the executed rows' coordinates and depths for the backward (the forward kept none)
    rb::rb_gather_kernel<<<grid_1d(L.Mmax, 256, 8), 256, 0, st>>>(at<float>(ws, L.rays8), box, z_steps, jitter, at<int32_t>(ws, L.order),
                                                            at<rb::ObjCounts>(ws, L.counts), at<rb::Meta>(ws, L.meta), B, N, S,
                                                            at<float>(sc, G.xyz_c), at<float>(sc, G.vrep_c), at<float>(sc, G.z_c));
    SNB_LAUNCH_CHECK();
    xyz_c = at<float>(sc, G.xyz_c); vrep_c = at<float>(sc, G.vrep_c); z_c = at<float>(sc, G.z_c);
  }
  const int64_t* total_rows = &at<rb::Meta>(ws, L.meta)->total_rows;
  SNB_CHECK_CUDA(cudaMemsetAsync(at<uint8_t>(sc, G.live_hdr), 0, G.live_end - G.live_hdr, st));   // count, ticket, flags
#define SNB_RBB(LL) rb::rb_composite_bwd_kernel<LL><<<cg.grid, 256, 0, st>>>(at<float>(ws, L.sigma_c), at<float>(ws, L.rgb_c), z_c, \
    at<int32_t>(ws, L.order), at<rb::ObjCounts>(ws, L.counts), N, S, d->flags, g_rgb, g_depth, g_acc, at<float>(sc, G.g_sigma_c), \
    at<float>(sc, G.g_rgb_c), gz, total_rows, at<uint8_t>(sc, G.live), at<int32_t>(sc, G.live_list), at<rb::LiveHdr>(sc, G.live_hdr))
  if (cg.lpr == 8) SNB_RBB(8); else if (cg.lpr == 16) SNB_RBB(16); else SNB_RBB(32);
#undef SNB_RBB
  SNB_LAUNCH_CHECK();
  if (decoder_backward(h, batch_precision(*d), xyz_c, vrep_c, L.Mmax, B, shape_latent, texture_latent, at<float>(ws, L.sigma_c),
                       at<float>(sc, G.g_sigma_c), at<float>(sc, G.g_rgb_c), at<uint8_t>(ws, L.mlp), at<uint8_t>(sc, G.mlp),
                       pose ? at<float>(sc, G.g_xyz_c) : nullptr, pose ? at<float>(sc, G.g_vrep_c) : nullptr, g_shape_latent, g_texture_latent,
                       nullptr, st, {total_rows, at<int32_t>(ws, L.tile_start), nullptr, at<int32_t>(sc, G.live_list),
                                     &at<rb::LiveHdr>(sc, G.live_hdr)->n_live}))
    return 1;
  if (!pose) return 0;
  SNB_CHECK_CUDA(cudaMemsetAsync(at<uint8_t>(sc, G.acc64), 0, G.mlp - G.acc64, st));   // fp64 sums + tickets
  rb::rb_rays_bwd_kernel<<<dim3((unsigned)grid_1d(N, 256, 8, B), (unsigned)B), 256, 0, st>>>(px, py, K, c2w, box, at<float>(ws, L.rays8), at<uint8_t>(ws, L.hit),
      at<int32_t>(ws, L.pos), at<rb::ObjCounts>(ws, L.counts), z_steps, jitter, N, S, at<float>(sc, G.g_xyz_c), at<float>(sc, G.g_vrep_c), gz,
      at<uint8_t>(sc, G.live), at<double>(sc, G.acc64), at<unsigned int>(sc, G.tickets), g_c2w);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_prepare_samples_batch(const float* px, const float* py, const float* K, const float* c2w, const float* z,
                                         const float* obj_diag, const int32_t* flip, int32_t n_objs, int64_t rays_per_obj,
                                         int32_t n_samples, int32_t shapenet_swap, float* xyz, float* viewdir_rep, void* stream) {
  SNB_REQUIRE(n_objs >= 1 && rays_per_obj >= 0 && n_samples >= 1, "prepare_samples_batch: bad sizes");
  if (rays_per_obj == 0) return 0;
  SNB_REQUIRE(px && py && K && c2w && z && obj_diag && xyz && viewdir_rep, "prepare_samples_batch: null pointer");
  const int64_t total = (int64_t)n_objs * rays_per_obj;
  const int grid = grid_1d(total, 8, 8);
  SNB_REQUIRE(grid > 0, "prepare_samples_batch: no CUDA device (there is no CPU fallback)");
  rb::rb_shell_prep_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(px, py, K, c2w, z, obj_diag, flip, rays_per_obj, n_samples,
                                                                           shapenet_swap, total, xyz, viewdir_rep);
  SNB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------------------- batched shell render
// The utils.py stack (utils.render_rays_v2, utils.py:435-502: shared sample vector per object, xyz / obj_diag, optional shapenet axis
// swap, volume_rendering2) for B objects in ONE launch set -- what render.cu's shell mode enqueues per object.  Dense rows (no slab test
// in this stack): B * N * S decoder rows, N * S a multiple of 128 in bf16 mode.
namespace snb {
namespace {
struct ShellLayout {   // forward workspace, kept for the backward
  size_t xyz, vrep, sigma, rgb, mlp, total;
  ShellLayout(snb_handle h, const snb_shell_batch_desc& d) {
    const size_t M = (size_t)d.n_objs * (size_t)d.rays_per_obj * (size_t)d.n_samples;
    size_t o = 0;
    xyz = o; o += al(M * 12);
    vrep = o; o += al(M * 12);
    sigma = o; o += al(M * 4);
    rgb = o; o += al(M * 12);
    mlp = o; o += al(snb_mlp_workspace_bytes(h, (int64_t)M, d.n_objs, d.precision));
    total = o;
  }
};
struct ShellScratch {
  size_t g_sigma, g_rgbs, g_xyz, g_vrep, acc64, tickets, mlp, total;
  ShellScratch(snb_handle h, const snb_shell_batch_desc& d) {
    const size_t B = (size_t)d.n_objs, M = B * (size_t)d.rays_per_obj * (size_t)d.n_samples;
    size_t o = 0;
    g_sigma = o; o += al(M * 4);
    g_rgbs = o; o += al(M * 12);
    g_xyz = o; o += al(M * 12);
    g_vrep = o; o += al(M * 12);
    acc64 = o; o += al(B * 12 * 8);
    tickets = o; o += al(B * 4);
    mlp = o; o += al(snb_mlp_bwd_scratch_bytes(h, (int64_t)M, d.n_objs, d.precision));
    total = o;
  }
};
int check_shell(snb_handle h, const snb_shell_batch_desc* d, const char* who) {
  SNB_REQUIRE(h != nullptr && d != nullptr, "%s: null handle or descriptor", who);
  SNB_REQUIRE(d->n_objs >= 1 && d->n_objs <= rb::kMaxObjs && d->rays_per_obj >= 1 && d->n_samples >= 1, "%s: bad sizes", who);
  SNB_REQUIRE(d->precision == SNB_PREC_FP32 || d->precision == SNB_PREC_BF16 || d->precision == SNB_PREC_FP32_TC,
              "%s: precision must be fp32, fp32_tc or bf16 (frozen weights)", who);
  SNB_REQUIRE((int64_t)d->n_objs * d->rays_per_obj * d->n_samples < ((int64_t)1 << 40), "%s: too many rows", who);
  return 0;
}
}  // namespace
}  // namespace snb

extern "C" size_t snb_render_shell_batch_workspace_bytes(snb_handle h, const snb_shell_batch_desc* d) {
  if (!h || !d || d->n_objs < 1 || d->rays_per_obj < 1 || d->n_samples < 1) return 0;
  return ShellLayout(h, *d).total + 256;
}

extern "C" size_t snb_render_shell_batch_scratch_bytes(snb_handle h, const snb_shell_batch_desc* d) {
  if (!h || !d || d->n_objs < 1 || d->rays_per_obj < 1 || d->n_samples < 1) return 0;
  return ShellScratch(h, *d).total + 256;
}

extern "C" int snb_render_shell_batch_fwd(snb_handle h, const snb_shell_batch_desc* d, const float* px, const float* py, const float* K,
                                          const float* c2w, const float* z, const float* obj_diag, const float* shape_latent,
                                          const float* texture_latent, float* out_rgb, float* out_depth, float* out_acc, void* workspace,
                                          void* stream) {
  if (check_shell(h, d, "render_shell_batch_fwd")) return 2;
  SNB_REQUIRE(px && py && K && c2w && z && obj_diag && shape_latent && texture_latent && out_rgb && out_depth && out_acc && workspace,
              "render_shell_batch_fwd: null pointer");
  SNB_REQUIRE(((uintptr_t)workspace & 255) == 0, "render_shell_batch_fwd: workspace must be 256-byte aligned");
  const ShellLayout L(h, *d);
  void* ws = workspace;
  const int64_t N = d->rays_per_obj, BN = (int64_t)d->n_objs * N, M = BN * d->n_samples;
  if (snb_prepare_samples_batch(px, py, K, c2w, z, obj_diag, nullptr, d->n_objs, N, d->n_samples, d->shapenet_swap, at<float>(ws, L.xyz),
                                at<float>(ws, L.vrep), stream)) return 1;
  if (snb_mlp_fwd(h, d->precision, at<float>(ws, L.xyz), at<float>(ws, L.vrep), M, d->n_objs, shape_latent, texture_latent,
                  at<float>(ws, L.sigma), at<float>(ws, L.rgb), at<uint8_t>(ws, L.mlp), stream)) return 1;
  return snb_composite_fwd(at<float>(ws, L.sigma), at<float>(ws, L.rgb), z, N, BN, d->n_samples, d->flags, out_rgb, out_depth, out_acc, stream);
}

extern "C" int snb_render_shell_batch_bwd(snb_handle h, const snb_shell_batch_desc* d, const float* px, const float* py, const float* K,
                                          const float* c2w, const float* z, const float* obj_diag, const float* shape_latent,
                                          const float* texture_latent, const void* workspace, const float* g_rgb, const float* g_depth,
                                          const float* g_acc, void* scratch, float* g_c2w, float* g_shape_latent, float* g_texture_latent,
                                          void* stream) {
  if (check_shell(h, d, "render_shell_batch_bwd")) return 2;
  SNB_REQUIRE(px && py && K && c2w && z && obj_diag && shape_latent && texture_latent && workspace && g_rgb && g_depth && g_acc && scratch &&
              g_shape_latent && g_texture_latent, "render_shell_batch_bwd: null pointer");
  SNB_REQUIRE((((uintptr_t)workspace | (uintptr_t)scratch) & 255) == 0, "render_shell_batch_bwd: workspace/scratch must be 256-byte aligned");
  const ShellLayout L(h, *d);
  const ShellScratch G(h, *d);
  cudaStream_t st = (cudaStream_t)stream;
  const void* ws = workspace;
  void* sc = scratch;
  const int B = d->n_objs;
  const int64_t N = d->rays_per_obj, BN = (int64_t)B * N, M = BN * d->n_samples;
  const bool pose = g_c2w != nullptr;
  // the shared sample vectors are built from detached python floats (utils.py:468-469): no gradient through z
  if (snb_composite_bwd(at<float>(ws, L.sigma), at<float>(ws, L.rgb), z, N, BN, d->n_samples, d->flags, g_rgb, g_depth, g_acc,
                        at<float>(sc, G.g_sigma), at<float>(sc, G.g_rgbs), nullptr, stream)) return 1;
  if (snb_mlp_bwd(h, d->precision, at<float>(ws, L.xyz), at<float>(ws, L.vrep), M, B, shape_latent, texture_latent, at<float>(ws, L.sigma),
                  at<float>(sc, G.g_sigma), at<float>(sc, G.g_rgbs), at<uint8_t>(ws, L.mlp), at<uint8_t>(sc, G.mlp),
                  pose ? at<float>(sc, G.g_xyz) : nullptr, pose ? at<float>(sc, G.g_vrep) : nullptr, g_shape_latent, g_texture_latent, nullptr,
                  stream)) return 1;
  if (!pose) return 0;
  const int gx = grid_1d(N, 8, 8, B);
  SNB_REQUIRE(gx > 0, "render_shell_batch_bwd: no CUDA device (there is no CPU fallback)");
  SNB_CHECK_CUDA(cudaMemsetAsync(at<uint8_t>(sc, G.acc64), 0, G.mlp - G.acc64, st));   // fp64 sums + tickets
  rb::rb_shell_rays_bwd_kernel<<<dim3((unsigned)gx, (unsigned)B), 256, 0, st>>>(px, py, K, c2w, z, obj_diag, N, d->n_samples, d->shapenet_swap,
      at<float>(sc, G.g_xyz), at<float>(sc, G.g_vrep), at<double>(sc, G.acc64), at<unsigned int>(sc, G.tickets), g_c2w);
  SNB_LAUNCH_CHECK();
  return 0;
}
