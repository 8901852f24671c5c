// K2 / K2b, one-tile tensor-core back end (SNB_PREC_BF16 for decoders the two-tile kernels of mlp_tc2.cu do not cover, and
// SNB_PREC_FP32_TC, the split-precision mode described below): the CodeNeRF-family decoder as ONE persistent, warp-specialised
// tcgen05 kernel per direction.  A 128-sample tile enters as fp32 xyz / viewdir; the positional
// encoding is built straight into shared memory as bf16 (never to HBM); every layer is a
// tcgen05.mma (bf16 x bf16 -> fp32 in TMEM, M=128, N<=256) whose A operand is the previous layer's
// epilogue output kept in shared memory and whose B operand (pre-tiled, pre-swizzled bf16 weight
// images) is streamed from L2 by the bulk-copy engine (cp.async.bulk + mbarrier) through a 3-stage
// ring.  Accumulators ping-pong between the two 256-column halves of TMEM so that the epilogue of
// layer l (bias, ReLU, latent add, mask bits, bf16 pack) overlaps the MMAs of layer l+1 chunk by
// chunk.  The W->1 (sigma) and W/2->3 (rgb) heads run on CUDA cores inside the epilogues.
// The hidden width W (128 or 256) is a template parameter of the kernels: W / 64 K chunks per hidden layer, W / 32 ReLU-mask words
// per layer.  Shared-memory tables keep a row stride of 256 at either width.
// Backward: same machinery with transposed weight images; ReLU masks come back as 1 bit/unit;
// latent gradients are per-object column sums reduced by warp butterflies; d(PE) is folded to
// d xyz / d viewdir in the epilogue.
//
// Warp roles (320 threads): warps 0-7 epilogue (warp w owns TMEM lanes 32*(w%4).. and the column
// half w/4 of every 64-column chunk), warp 8 weight producer (+ TMEM alloc), warp 9 MMA issuer.
//
// Host side: the step programs and weight-packing jobs (build_plan), the packing launches and one launch function per direction
// (tc1_launch_fwd / tc1_launch_bwd).  Back-end selection, workspace and packed-buffer layout, the latent layers and the timing live in
// decoder.cu.
#include "common.cuh"
#include "decoder.h"
#include "tc_ptx.cuh"
#include "rb_rows.cuh"
#include <math.h>
#include <algorithm>
#include <stdlib.h>
#include <vector>

namespace snb {
namespace tc {

#ifndef SNB_TC_STAGES
#define SNB_TC_STAGES 3
#endif
constexpr int kStages = SNB_TC_STAGES;   // weight-ring depth (tuning builds: -DSNB_TC_STAGES=2 measures the ring's share of the time)
constexpr int kMaxSteps = 16;
constexpr int kMaxFwdSteps = 14;        // 5 + 5 blocks (the SUPNeRF() / AutoRFMix() class defaults): 1 + 5 + 1 + 1 + 5 + 1
constexpr int kThreads = 320;
constexpr int kMaxLatentSlots = 10;

// Split mode (template parameter X = true; SNB_PREC_FP32_TC): fp32-grade arithmetic on the same tensor-core pipeline.  Every MMA
// operand is held as TWO fp16 parts (x = hi + lo, |lo| <= 2^-12 |x|) and each product is issued as three MMAs (hi*hi, lo*hi, hi*lo;
// lo*lo ~ 2^-24 is dropped) accumulating into the same fp32 TMEM columns.  Weights are packed as 256 * w (a power of two keeps the low
// part out of fp16's subnormal range; |w| < 255), forward A operands are the activations themselves (|a| < 65504), backward A operands
// are each row's gradient normalised by a power of two taken from its upstream gradient (the backward pass is linear in it), undone
// where values leave the tile (latent column sums, d xyz, d viewdir).  Shared memory: every logical 64-column A chunk is a (hi, lo)
// pair of physical chunks, the weight ring carries [128 n][64 k] stages (hi and lo of each N half, one after the other), and one 10 KB
// table holds the forward's (effective) biases / the backward's column sums (tools/experiments/split_precision_emulation.py and
// tests/test_split_precision_numerics.py: the arithmetic's errors vs fp64 are on par with fp32 FFMA).
constexpr float kWScale = 256.f, kWScaleInv = 1.f / 256.f;
// Order of the three products of a layer's K chunks (see mma_loop).  1: every chunk's correction products first, then all leading ones
// (the hi weight image is streamed twice: 3 stages per chunk and N half); 0: chunk by chunk (2 stages); 2: corrections first for all
// chunks but the LAST one the epilogue publishes, whose three products are issued together -- the leading products of the earlier
// chunks then run while the epilogue still works on the last chunk.
#ifndef SNB_SPLIT_CORR_FIRST
#define SNB_SPLIT_CORR_FIRST 1
#endif
constexpr int kOrder = SNB_SPLIT_CORR_FIRST;
constexpr bool kCorrFirst = kOrder != 0;
__host__ __device__ constexpr int split_stages_per_half(int n_chunks) {
  return kOrder == 0 ? 2 * n_chunks : (kOrder == 1 ? 3 * n_chunks : 3 * (n_chunks - 1) + 2);
}
constexpr int kSplitBiasSteps = kMaxLatentSlots;   // split mode, forward: steps whose (effective) bias sits in shared memory (the 8 KB the backward uses for column sums)

// shared-memory map (bytes from the 1024-aligned base)
template <bool X> struct Map {
  static constexpr uint32_t kAChunks = X ? 10u : 5u;                 // A chunks 0..3, AUX chunk 4 (split: physical chunk 2c + part)
  static constexpr uint32_t kStageBytes = X ? 16384u : 32768u;       // [256 n][64 k] bf16, split: [128 n][64 k] fp16
  static constexpr uint32_t SM_W = kAChunks * kChunkBytes;           // then the weight ring
  static constexpr uint32_t SM_TAB = SM_W + kStages * kStageBytes;   // fp32 tables
  static constexpr uint32_t TAB_BIAS = 0;                            // fwd: [kMaxFwdSteps][256] (split: [kSplitBiasSteps][256])  bwd: colsum [slots][256]
  static constexpr uint32_t TAB_Z = TAB_BIAS + (X ? kMaxLatentSlots : kMaxFwdSteps) * 256 * 4;   // fwd: [8][256] per-object effective biases (split: none)
  static constexpr uint32_t TAB_WSIG = TAB_Z + (X ? 0 : kMaxLatentSlots * 256 * 4);   // [256]
  static constexpr uint32_t TAB_W2 = TAB_WSIG + 256 * 4;             // [3][128]
  static constexpr uint32_t TAB_PART = TAB_W2 + 384 * 4;             // fwd: sig_part [2][128] + rgb_part [2][128][3]; bwd: xyz_part [2][128][3]
  static constexpr uint32_t TAB_BYTES = TAB_PART + (256 + 768) * 4;
  static constexpr uint32_t SM_BARS = SM_TAB + TAB_BYTES;
  static constexpr uint32_t SM_TOTAL = SM_BARS + 32 * 8 + 16;
  static constexpr uint32_t SM_ALLOC = SM_TOTAL + 1024;              // + alignment slack
};
static_assert(Map<false>::SM_ALLOC <= 232448 && Map<true>::SM_ALLOC <= 232448, "shared memory budget");

enum Epi : int { EPI_RELU = 0, EPI_LINEAR_SIGMA = 1, EPI_RGB_HEAD = 2, EPI_B_MASK = 3, EPI_B_EV = 4, EPI_B_XYZ = 5 };

struct Step {
  uint32_t w_off, w2_off;      // byte offsets of the first weight chunk of MMA group 1 / 2 in the packed buffer
  uint16_t n_chunks, n_out;    // K chunks (64 wide), N of group 1
  uint16_t n2_out;             // N of group 2 (0: none); group 2 re-reads the same A chunks
  uint8_t a_chunk[6];          // shared-memory chunk index per K chunk (0..3 = A, 4 = AUX)
  int8_t epi, mask_slot, latent_slot, produce_a;
  const float* bias;           // fp32 bias of the layer (forward)
};

struct Program {
  int n_steps, n_mask_slots;
  Step s[kMaxSteps];
};

struct Params {
  const float* xyz; const float* viewdir;
  int64_t M, rows_per_obj, B;
  const uint8_t* packed;
  const float* zlat;            // fwd: per-object effective biases b + W z, [(Bs+Bt)][B][W]; bwd: unused
  const float* wsig; const float* bsig; const float* w2; const float* b2;
  uint32_t* masks;              // [tile][slot][W / 32 words][128 rows]
  // forward
  float* sigma; float* rgb; float* dbg;
  // backward
  const float* sigma_in; const float* g_sigma; const float* g_rgb;
  float* g_xyz; float* g_viewdir; float* g_zlat;   // g_zlat [(Bs+Bt)][B][W], accumulated with atomics
  int r0_mask_slot, n_latent, ev_step;
  const int64_t* m_dev;         // device-side row count (a multiple of 128, <= M) or null
  const int32_t* tile_start;    // per-object first tile (B + 1 ints) or null = M / B rows per object
  Program prog;
  const int32_t* live;          // backward: the 256-row super tiles to run (ascending) or null = every tile (decoder.h: DeviceRows)
  const int32_t* n_live;        // ... and their count, on the device
};

template <bool X> struct SmemT {
  using M = Map<X>;
  uint8_t* base;
  uint32_t base_u32;
  // logical A chunk c (0..4); split mode: part 0 = hi, 1 = lo
  __device__ uint8_t* chunk(int c, int part = 0) const { return base + (uint32_t)(X ? 2 * c + part : c) * kChunkBytes; }
  __device__ uint32_t chunk_u32(int c, int part = 0) const { return base_u32 + (uint32_t)(X ? 2 * c + part : c) * kChunkBytes; }
  __device__ uint32_t stage_u32(int s) const { return base_u32 + M::SM_W + (uint32_t)s * M::kStageBytes; }
  __device__ float* tab(uint32_t off) const { return reinterpret_cast<float*>(base + M::SM_TAB + off); }
  __device__ uint32_t bar(int i) const { return base_u32 + M::SM_BARS + 8u * i; }
};

__device__ __forceinline__ int64_t rows_present(const Params& p) { return p.m_dev ? *p.m_dev : p.M; }
// the object a tile belongs to: binary search of the per-object first tiles (batched render), else uniform rows per object
__device__ __forceinline__ int64_t obj_of_tile(const Params& p, int64_t tile) {
  if (p.tile_start == nullptr) return (tile * kTileM) / p.rows_per_obj;
  int lo = 0, hi = (int)p.B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((int64_t)__ldg(p.tile_start + mid) <= tile) lo = mid; else hi = mid - 1;
  }
  return lo;
}
// tile of the backward's j-th work item: its 128-row half of live super tile j / 2, or tile j without a list
__device__ __forceinline__ int64_t work_tile(const Params& p, int64_t j) {
  return p.live ? 2 * (int64_t)__ldg(p.live + (j >> 1)) + (j & 1) : j;
}
// barrier indices
constexpr int BAR_WFULL = 0, BAR_WEMPTY = 4, BAR_AREADY = 8, BAR_ACC = 13;

// per-thread view of the epilogue role
struct EpiCtx {
  uint32_t lane, hh, row, lane_field, tmem_base;
  int64_t grow;      // global sample row of this thread
  bool valid;
};

// ------------------------------------------------------------------------------------------ roles shared by fwd / bwd
// weight stages of one K chunk of an MMA group: plain mode one [n][64 k] image; split mode per N half (<= 128 columns) the hi image,
// then the lo image
__device__ __forceinline__ uint32_t n_half_of(uint32_t n) { return n < 128u ? n : 128u; }

template <bool X>
__device__ __forceinline__ void producer_loop(const Params& p, const SmemT<X>& sm, int64_t n_tiles, uint32_t lane) {
  uint32_t it = 0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    for (int si = 0; si < p.prog.n_steps; ++si) {
      const Step& st = p.prog.s[si];
      const int groups = st.n2_out ? 2 : 1;
      for (int g = 0; g < groups; ++g) {
        const uint32_t n = (uint32_t)(g == 0 ? st.n_out : st.n2_out);
        const uint32_t bytes = (X ? n_half_of(n) : n) * 128u;
        const uint32_t off0 = g == 0 ? st.w_off : st.w2_off;
        const int entries = X ? split_stages_per_half((int)st.n_chunks) * (int)(n / n_half_of(n)) : (int)st.n_chunks;   // split: see mma_loop
        for (int e = 0; e < entries; ++e, ++it) {
          const uint32_t stage = it % kStages, ph = (it / kStages) & 1u;
          if (lane == 0) {
            mbar_wait(sm.bar(BAR_WEMPTY + stage), ph ^ 1u);
            mbar_expect_tx(sm.bar(BAR_WFULL + stage), bytes);
            bulk_g2s(sm.stage_u32(stage), p.packed + off0 + (size_t)e * bytes, bytes, sm.bar(BAR_WFULL + stage));
          }
          __syncwarp();
        }
      }
    }
  }
}

template <bool X>
__device__ __forceinline__ void mma_loop(const Params& p, const SmemT<X>& sm, int64_t n_tiles, uint32_t lane, uint32_t tmem_base) {
  uint32_t it = 0, gstep = 0;
  uint32_t a_phase = 0;  // bit c = parity of the next completion of a_ready[c] to wait for
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    for (int si = 0; si < p.prog.n_steps; ++si, ++gstep) {
      const Step& st = p.prog.s[si];
      const uint32_t half = gstep & 1u;
      const int groups = st.n2_out ? 2 : 1;
      for (int g = 0; g < groups; ++g) {
        const uint32_t n = g == 0 ? st.n_out : st.n2_out;
        const uint32_t d_tmem = tmem_base + (g == 0 ? half : (half ^ 1u)) * 256u;
        if (!X) {
          const uint32_t idesc = umma_idesc(128, n);
          for (int kc = 0; kc < st.n_chunks; ++kc, ++it) {
            const int ac = st.a_chunk[kc];
            const uint32_t stage = it % kStages, ph = (it / kStages) & 1u;
            if (lane == 0) {
              if (g == 0) mbar_wait(sm.bar(BAR_AREADY + ac), (a_phase >> ac) & 1u);
              mbar_wait(sm.bar(BAR_WFULL + stage), ph);
              tc_fence_after();
              const uint32_t a0 = sm.chunk_u32(ac), b0 = sm.stage_u32(stage);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_bf16(d_tmem, umma_desc(a0 + kk * 32), umma_desc(b0 + kk * 32), idesc, (kc > 0 || kk > 0) ? 1u : 0u);
              umma_commit(sm.bar(BAR_WEMPTY + stage));
            }
            if (g == 0) a_phase ^= 1u << ac;
            __syncwarp();
          }
        } else {
          // FIRST every K chunk's correction products (a_lo * w_hi, a_hi * w_lo), THEN the leading products (a_hi * w_hi).
          // The tensor core truncates the fp32 accumulator after every instruction (an error of up to one ulp of its CURRENT
          // magnitude each): the 2 x 16 correction instructions run while it only holds the ~2^-11 times smaller correction sum, so
          // only the 16 leading instructions truncate at full scale.  (The hi image of every chunk is streamed twice for this.)
          const uint32_t nh_n = n_half_of(n), halves = n / nh_n;
          const uint32_t idesc = umma_idesc_f16(128, nh_n);
          // one weight stage: `n_mma` products per 16-wide K step against it
          auto run_stage = [&](uint32_t d, uint32_t a_first, uint32_t a_second, bool two, bool fresh, int wait_chunk) {
            const uint32_t stage = it % kStages, ph = (it / kStages) & 1u;
            if (lane == 0) {
              if (wait_chunk >= 0) mbar_wait(sm.bar(BAR_AREADY + wait_chunk), (a_phase >> wait_chunk) & 1u);
              mbar_wait(sm.bar(BAR_WFULL + stage), ph);
              tc_fence_after();
              const uint32_t b0 = sm.stage_u32(stage);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                umma_bf16(d, umma_desc(a_first + kk * 32), umma_desc(b0 + kk * 32), idesc, (fresh && kk == 0) ? 0u : 1u);
                if (two) umma_bf16(d, umma_desc(a_second + kk * 32), umma_desc(b0 + kk * 32), idesc, 1u);
              }
              umma_commit(sm.bar(BAR_WEMPTY + stage));
            }
            ++it;
          };
          // K chunk by K chunk (a chunk's products start as soon as the epilogue has published it), both N halves per chunk
          const int n_corr = kOrder == 1 ? (int)st.n_chunks : (kOrder == 2 ? (int)st.n_chunks - 1 : 0);   // chunks whose corrections go first
          for (int kc = 0; kc < n_corr; ++kc) {              // corrections only: a_lo * w_hi, a_hi * w_lo
            const int ac = st.a_chunk[kc];
            const uint32_t a_hi = sm.chunk_u32(ac, 0), a_lo = sm.chunk_u32(ac, 1);
            for (uint32_t nh = 0; nh < halves; ++nh) {
              const uint32_t d = d_tmem + nh * 128u;
              run_stage(d, a_lo, 0u, false, kc == 0, (g == 0 && nh == 0) ? ac : -1);
              run_stage(d, a_hi, 0u, false, false, -1);
            }
            if (g == 0) a_phase ^= 1u << ac;
            __syncwarp();
          }
          for (int kc = 0; kc < n_corr; ++kc) {              // their leading products, into accumulators that hold the corrections
            const uint32_t a_hi = sm.chunk_u32(st.a_chunk[kc], 0);
            for (uint32_t nh = 0; nh < halves; ++nh) run_stage(d_tmem + nh * 128u, a_hi, 0u, false, false, -1);
            __syncwarp();
          }
          for (int kc = n_corr; kc < st.n_chunks; ++kc) {    // the remaining chunks: all three products, (a_lo, a_hi) * w_hi, a_hi * w_lo
            const int ac = st.a_chunk[kc];
            const uint32_t a_hi = sm.chunk_u32(ac, 0), a_lo = sm.chunk_u32(ac, 1);
            for (uint32_t nh = 0; nh < halves; ++nh) {
              const uint32_t d = d_tmem + nh * 128u;
              run_stage(d, a_lo, a_hi, true, kc == 0, (g == 0 && nh == 0) ? ac : -1);
              run_stage(d, a_hi, 0u, false, false, -1);
            }
            if (g == 0) a_phase ^= 1u << ac;
            __syncwarp();
          }
        }
      }
      if (lane == 0) umma_commit(sm.bar(BAR_ACC + half));
      __syncwarp();
    }
  }
}

// after this thread's generic-proxy stores into an A chunk: publish to the async proxy and signal the MMA warp
template <bool X>
__device__ __forceinline__ void publish_chunk(const SmemT<X>& sm, int c, uint32_t lane) {
  tc_fence_before();
  fence_async_smem();
  __syncwarp();
  if (lane == 0) mbar_arrive(sm.bar(BAR_AREADY + c));
}

__device__ __forceinline__ void store_row32(uint8_t* chunk, uint32_t row, uint32_t hh, const uint32_t (&pk)[16]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    uint4 q = make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
    *reinterpret_cast<uint4*>(chunk + swz(row, hh * 4 + u)) = q;
  }
}

// A-operand writer of one 32-column half row: plain mode one bf16 chunk, split mode the fp16 (hi, lo) chunk pair
template <bool X> struct RowPack {
  uint32_t hi[16], lo[X ? 16 : 1];
  __device__ __forceinline__ void set(int i, float a, float b) {   // word i = columns (2i, 2i + 1)
    if constexpr (X) split_f16x2(a, b, hi[i], lo[i]); else hi[i] = pack_bf16(a, b);
  }
  __device__ __forceinline__ void set_relu(int i, float a, float b) {
    if constexpr (X) split_f16x2(fmaxf(a, 0.f), fmaxf(b, 0.f), hi[i], lo[i]); else hi[i] = pack_bf16_relu(a, b);
  }
  __device__ __forceinline__ void store(const SmemT<X>& sm, int c, uint32_t row, uint32_t hh) const {
    store_row32(sm.chunk(c, 0), row, hh, hi);
    if constexpr (X) store_row32(sm.chunk(c, 1), row, hh, lo);
  }
};

// PE(x) of this thread's half row into the AUX chunk (split mode: both parts)
template <int DEG, bool X>
__device__ __forceinline__ void write_pe(const SmemT<X>& sm, uint32_t row, uint32_t hh, const float x[3]) {
  if constexpr (!X) {
    write_pe_row<DEG>(sm.chunk(4), row, hh, x);
  } else {
    float v[32];
    pe_half_f32<DEG>(x, hh, v);
    RowPack<X> rp;
#pragma unroll
    for (int i = 0; i < 16; ++i) rp.set(i, v[2 * i], v[2 * i + 1]);
    rp.store(sm, 4, row, hh);
  }
}

template <bool X>
__device__ __forceinline__ void kernel_prologue(SmemT<X>& sm, uint8_t* smem_raw, uint32_t tid, uint32_t warp, uint32_t& tmem_base) {
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
  sm.base = smem_raw + pad;
  sm.base_u32 = raw + pad;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm.base + Map<X>::SM_BARS + 32 * 8);
  if (tid == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(sm.bar(BAR_WFULL + i), 1); mbar_init(sm.bar(BAR_WEMPTY + i), 1); }
    for (int i = 0; i < 5; ++i) mbar_init(sm.bar(BAR_AREADY + i), 8);
    for (int i = 0; i < 2; ++i) mbar_init(sm.bar(BAR_ACC + i), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  tmem_base = *tmem_slot;
}

// ------------------------------------------------------------------------------------------ forward epilogues
// One layer's epilogue for this thread's row: TMEM -> (+bias, ReLU, mask bits, +latent) -> bf16 -> shared-memory A operand.
// The TMEM load of chunk c+1 is in flight while chunk c is processed.  Split mode: accumulators carry the weight scale; the bias /
// per-object effective bias is read through L1 from `bias_g` (every lane of a warp reads the same address).
template <int EPI, bool LAT, bool DBG, bool X, int W>
__device__ __forceinline__ void fwd_epilogue(const Params& p, const SmemT<X>& sm, const Step& st, int si, uint32_t half, const EpiCtx& e,
                                             uint32_t* mask_tile, float& sig_acc, float (&rgb_acc)[3], const float* bias_g) {
  using MP = Map<X>;
  constexpr int NC = (EPI == EPI_RGB_HEAD ? W / 2 : W) / 64;   // 64-column chunks of the layer's outputs
  // latent-conditioned layers read their per-object EFFECTIVE bias  b + W z_obj  (the latent add folded through the layer)
  const float* bias_s = X ? bias_g : (LAT ? sm.tab(MP::TAB_Z) + st.latent_slot * 256 : sm.tab(MP::TAB_BIAS) + si * 256);
  const float* wsig_s = sm.tab(MP::TAB_WSIG);
  const float* w2_s = sm.tab(MP::TAB_W2);
  const uint32_t t0 = e.tmem_base + half * 256u + e.hh * 32u + e.lane_field;
  uint32_t ra[32], rb[32];
  tmem_ld32_issue(t0, ra);
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    uint32_t (&r)[32] = (c & 1) ? rb : ra;
    tmem_ld_wait();
    if (c + 1 < NC) tmem_ld32_issue(t0 + (uint32_t)(c + 1) * 64u, (c & 1) ? ra : rb);
    const int col0 = c * 64 + (int)e.hh * 32;
    RowPack<X> rp;
    uint32_t nmask = 0;   // nmask collects SIGN bits (1 = negative pre-activation); stored inverted
#pragma unroll
    for (int i4 = 0; i4 < 8; ++i4) {
      const float4 bb = *reinterpret_cast<const float4*>(bias_s + col0 + 4 * i4);
      float v[4];
      if (X) {
        v[0] = fmaf(__uint_as_float(r[4 * i4]), kWScaleInv, bb.x); v[1] = fmaf(__uint_as_float(r[4 * i4 + 1]), kWScaleInv, bb.y);
        v[2] = fmaf(__uint_as_float(r[4 * i4 + 2]), kWScaleInv, bb.z); v[3] = fmaf(__uint_as_float(r[4 * i4 + 3]), kWScaleInv, bb.w);
      } else {
        v[0] = __uint_as_float(r[4 * i4]) + bb.x; v[1] = __uint_as_float(r[4 * i4 + 1]) + bb.y;
        v[2] = __uint_as_float(r[4 * i4 + 2]) + bb.z; v[3] = __uint_as_float(r[4 * i4 + 3]) + bb.w;
      }
      if (EPI != EPI_LINEAR_SIGMA) {
#pragma unroll
        for (int u = 0; u < 4; ++u) nmask = __funnelshift_l(__float_as_uint(v[u]), nmask, 1);
      }
      if (EPI == EPI_LINEAR_SIGMA) {
        const float4 ws = *reinterpret_cast<const float4*>(wsig_s + col0 + 4 * i4);
        sig_acc += v[0] * ws.x + v[1] * ws.y + v[2] * ws.z + v[3] * ws.w;
      }
      if (EPI == EPI_RGB_HEAD) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float4 ww = *reinterpret_cast<const float4*>(w2_s + k * (W / 2) + col0 + 4 * i4);
          rgb_acc[k] += fmaxf(v[0], 0.f) * ww.x + fmaxf(v[1], 0.f) * ww.y + fmaxf(v[2], 0.f) * ww.z + fmaxf(v[3], 0.f) * ww.w;
        }
      }
      if (DBG) {
        if (e.valid) {
          float* d = p.dbg + ((size_t)si * p.M + e.grow) * 256 + col0 + 4 * i4;
#pragma unroll
          for (int u = 0; u < 4; ++u) d[u] = (EPI == EPI_LINEAR_SIGMA) ? v[u] : fmaxf(v[u], 0.f);
        }
      }
      if (EPI == EPI_LINEAR_SIGMA) {
        rp.set(2 * i4, v[0], v[1]);
        rp.set(2 * i4 + 1, v[2], v[3]);
      } else if (EPI == EPI_RELU) {
        rp.set_relu(2 * i4, v[0], v[1]);
        rp.set_relu(2 * i4 + 1, v[2], v[3]);
      }
    }
    const uint32_t mask = ~nmask;
    if (EPI != EPI_LINEAR_SIGMA) mask_tile[((size_t)st.mask_slot * (W / 32) + c * 2 + e.hh) * 128 + e.row] = mask;
    if (EPI != EPI_RGB_HEAD) {
      rp.store(sm, c, e.row, e.hh);
      publish_chunk(sm, c, e.lane);
    }
  }
}

template <bool DBG, bool X, int W>
__device__ __forceinline__ void fwd_epilogue_dispatch(const Params& p, const SmemT<X>& sm, const Step& st, int si, uint32_t half,
                                                      const EpiCtx& e, uint32_t* mask_tile, float& sig_acc, float (&rgb_acc)[3],
                                                      const float* bias_g) {
  if (st.epi == EPI_RELU) {
    if (st.latent_slot >= 0) fwd_epilogue<EPI_RELU, true, DBG, X, W>(p, sm, st, si, half, e, mask_tile, sig_acc, rgb_acc, bias_g);
    else fwd_epilogue<EPI_RELU, false, DBG, X, W>(p, sm, st, si, half, e, mask_tile, sig_acc, rgb_acc, bias_g);
  } else if (st.epi == EPI_LINEAR_SIGMA) {
    fwd_epilogue<EPI_LINEAR_SIGMA, false, DBG, X, W>(p, sm, st, si, half, e, mask_tile, sig_acc, rgb_acc, bias_g);
  } else {
    fwd_epilogue<EPI_RGB_HEAD, false, DBG, X, W>(p, sm, st, si, half, e, mask_tile, sig_acc, rgb_acc, bias_g);
  }
}

// ------------------------------------------------------------------------------------------ forward kernel
template <bool X, int W>
__global__ void __launch_bounds__(kThreads, 1) tc_fwd_kernel(const __grid_constant__ Params p) {
  using MP = Map<X>;
  extern __shared__ uint8_t smem_raw[];
  SmemT<X> sm;
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t tmem_base;
  {  // static tables: every layer's bias (plain mode), the sigma / rgb head weights
    const uint32_t raw = smem_u32(smem_raw);
    uint8_t* b = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
    {  // split mode: the table has room for the first kSplitBiasSteps steps; later steps (more than 10: no supported architecture) read L1 / L2
      float* bias_s = reinterpret_cast<float*>(b + MP::SM_TAB + MP::TAB_BIAS);
      const int n_tab = X ? (p.prog.n_steps < kSplitBiasSteps ? p.prog.n_steps : kSplitBiasSteps) : p.prog.n_steps;
      for (int i = tid; i < n_tab * 256; i += kThreads) {
        const int si = i >> 8, c = i & 255;
        bias_s[i] = c < p.prog.s[si].n_out ? __ldg(p.prog.s[si].bias + c) : 0.f;
      }
    }
    float* wsig_s = reinterpret_cast<float*>(b + MP::SM_TAB + MP::TAB_WSIG);
    for (int i = tid; i < W; i += kThreads) wsig_s[i] = __ldg(p.wsig + i);
    float* w2_s = reinterpret_cast<float*>(b + MP::SM_TAB + MP::TAB_W2);
    for (int i = tid; i < 3 * W / 2; i += kThreads) w2_s[i] = __ldg(p.w2 + i);
  }
  kernel_prologue(sm, smem_raw, tid, warp, tmem_base);
  const int64_t M = rows_present(p);
  const int64_t n_tiles = (M + kTileM - 1) / kTileM;

  if (warp == 8) {
    producer_loop<X>(p, sm, n_tiles, lane);
  } else if (warp == 9) {
    mma_loop<X>(p, sm, n_tiles, lane, tmem_base);
  } else {
    EpiCtx e;
    e.lane = lane; e.hh = warp >> 2; e.row = (warp & 3u) * 32u + lane; e.lane_field = ((warp & 3u) * 32u) << 16;
    e.tmem_base = tmem_base;
    float* sig_part = sm.tab(MP::TAB_PART);          // [2][128]
    float* rgb_part = sm.tab(MP::TAB_PART) + 256;    // [2][128][3]
    float* z_s = sm.tab(MP::TAB_Z);
    uint32_t gstep = 0, acc_cnt[2] = {0, 0};
    const int nslots = p.prog.n_mask_slots;
    int64_t cur_obj = -1;
    // PE(xyz) of the first tile; later tiles are encoded one tile ahead (during the encoding_viewdir epilogue)
    if ((int64_t)blockIdx.x < n_tiles) {
      int64_t r0 = (int64_t)blockIdx.x * kTileM + e.row;
      if (r0 > M - 1) r0 = M - 1;
      const float x[3] = {__ldg(p.xyz + 3 * r0), __ldg(p.xyz + 3 * r0 + 1), __ldg(p.xyz + 3 * r0 + 2)};
      write_pe<10, X>(sm, e.row, e.hh, x);
      publish_chunk(sm, 4, lane);
    }
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      e.grow = tile * kTileM + e.row;
      e.valid = e.grow < M;
      const int64_t crow = e.valid ? e.grow : M - 1;
      const int64_t next_tile = tile + gridDim.x;
      float xn[3] = {0.f, 0.f, 0.f};
      // the next tile's coordinates, consumed by the encoding_viewdir epilogue.  W = 256: prefetched here, ~5 layers ahead.  W = 128:
      // loaded while that layer's MMAs run (holding them from here made the split-precision forward spill 52 more bytes)
      auto load_xn = [&] {
        int64_t rn = next_tile * kTileM + e.row;
        if (rn > M - 1) rn = M - 1;
        xn[0] = __ldg(p.xyz + 3 * rn); xn[1] = __ldg(p.xyz + 3 * rn + 1); xn[2] = __ldg(p.xyz + 3 * rn + 2);
      };
      if (W == 256 && next_tile < n_tiles) load_xn();
      const float dir[3] = {__ldg(p.viewdir + 3 * crow), __ldg(p.viewdir + 3 * crow + 1), __ldg(p.viewdir + 3 * crow + 2)};
      const int64_t obj = obj_of_tile(p, tile);   // tiles never straddle objects (checked on the host)
      if (obj != cur_obj) {  // (re)load the per-object effective biases; all epilogue warps are between tiles here
        cur_obj = obj;
        if (!X) {
          for (int i = tid; i < p.n_latent * 256; i += 256)   // [slot][256] in shared memory; column tid
            if (W == 256 || tid < W) z_s[i] = __ldg(p.zlat + ((size_t)(i >> 8) * p.B + obj) * W + (i & 255));
        } else {   // split mode: into the latent-conditioned steps' rows of the bias table
          float* bias_tab = sm.tab(MP::TAB_BIAS);
          for (int si = 0; si < p.prog.n_steps && si < kSplitBiasSteps; ++si) {
            const int slot = p.prog.s[si].latent_slot;
            if (slot >= 0 && (W == 256 || tid < W)) bias_tab[si * 256 + tid] = __ldg(p.zlat + ((size_t)slot * p.B + obj) * W + tid);
          }
        }
        epi_bar_sync();
      }
      uint32_t* mask_tile = p.masks + (size_t)tile * nslots * (W / 32) * 128;
      float sig_acc = 0.f, rgb_acc[3] = {0.f, 0.f, 0.f};
      for (int si = 0; si < p.prog.n_steps; ++si, ++gstep) {
        const Step& st = p.prog.s[si];
        const uint32_t half = gstep & 1u;
        const float* bias_g = nullptr;   // split mode: the step's (effective) bias, from the shared-memory table or through L1
        if (X) bias_g = si < kSplitBiasSteps ? sm.tab(MP::TAB_BIAS) + si * 256
                                             : (st.latent_slot >= 0 ? p.zlat + ((size_t)st.latent_slot * p.B + obj) * W : st.bias);
        if (W == 128 && si == p.ev_step && next_tile < n_tiles) load_xn();
        mbar_wait(sm.bar(BAR_ACC + half), acc_cnt[half] & 1u);
        acc_cnt[half]++;
        tc_fence_after();
        if (si == 0) {  // layer 0's MMAs are done with PE(xyz): the AUX chunk now takes PE(viewdir)
          write_pe<4, X>(sm, e.row, e.hh, dir);
          publish_chunk(sm, 4, lane);
        } else if (si == p.ev_step && next_tile < n_tiles) {  // encoding_viewdir's MMAs are done with PE(viewdir)
          write_pe<10, X>(sm, e.row, e.hh, xn);
          publish_chunk(sm, 4, lane);
        }
        if (p.dbg != nullptr) fwd_epilogue_dispatch<true, X, W>(p, sm, st, si, half, e, mask_tile, sig_acc, rgb_acc, bias_g);
        else fwd_epilogue_dispatch<false, X, W>(p, sm, st, si, half, e, mask_tile, sig_acc, rgb_acc, bias_g);
        tc_fence_before();
      }
      sig_part[e.hh * 128 + e.row] = sig_acc;
#pragma unroll
      for (int k = 0; k < 3; ++k) rgb_part[(e.hh * 128 + e.row) * 3 + k] = rgb_acc[k];
      epi_bar_sync();
      if (e.hh == 0 && e.valid) {
        const float sp = sig_part[e.row] + sig_part[128 + e.row] + __ldg(p.bsig);
        p.sigma[e.grow] = sp > 20.f ? sp : log1pf(expf(sp));   // nn.Softplus(): beta 1, threshold 20
#pragma unroll
        for (int k = 0; k < 3; ++k)
          p.rgb[3 * e.grow + k] = rgb_part[e.row * 3 + k] + rgb_part[(128 + e.row) * 3 + k] + __ldg(p.b2 + k);
      }
      epi_bar_sync();   // sig_part / rgb_part are rewritten at the end of the next tile only, but z_s may be reloaded next
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------ backward epilogues
template <int W>
__device__ __forceinline__ uint32_t mask_word(const uint32_t* mask_tile, int slot, int word, uint32_t row) {
  return __ldg(mask_tile + ((size_t)slot * (W / 32) + word) * 128 + row);
}

// acc = gradient w.r.t. the layer's input.  Optional: per-object column sums of it (latent gradient); then mask by the
// producing layer's ReLU bits and hand on as the next A operand.  EV: add the sigma-head gradient first, no mask.
// Split mode: acc is the row's gradient in units of 2^rexp (times the weight scale); gsp is the TRUE sigma-head gradient.  Gradients
// shrink (or grow) by a factor per layer, and an fp16 pair only resolves 2^-25 absolutely, so every layer re-centres the row: both
// threads of a row read the same 32 sample columns of the accumulator, take the power of two that brings their largest magnitude
// to [4, 8) (13 bits of headroom above the sample for the other columns) and fold it into rexp -- exact, and identical in both threads.
template <bool EV, bool COLSUM, bool MASK, bool PRODUCE, bool X, int W>
__device__ __forceinline__ void bwd_epilogue(const SmemT<X>& sm, const Step& st, uint32_t half, const EpiCtx& e,
                                             const uint32_t* mask_tile, float gsp, int& rexp) {
  using MP = Map<X>;
  constexpr int NC = W / 64;
  const float* wsig_s = sm.tab(MP::TAB_WSIG);
  float* colsum = sm.tab(MP::TAB_BIAS);
  const uint32_t t0 = e.tmem_base + half * 256u + e.hh * 32u + e.lane_field;
  uint32_t ra[32], rb[32];
  float in_scale = 1.f, a_scale = 1.f, row_scale = 1.f;   // accumulator -> v; v -> A operand; v -> true gradient
  if (X) {
    in_scale = kWScaleInv;
    row_scale = ldexpf(1.f, rexp);
    if (EV) gsp *= ldexpf(1.f, -rexp);
    if (PRODUCE) {
      tmem_ld32(e.tmem_base + half * 256u + e.lane_field, ra);   // columns 0..31 of the row: the sample both of its threads see
      float m = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float v = __uint_as_float(ra[i]) * kWScaleInv;
        if (EV) v += gsp * wsig_s[i];
        m = fmaxf(m, fabsf(v));
      }
      if (m > 0.f && m < 3.0e38f) {
        int ex;
        frexpf(m, &ex);
        int shift = ex - 3;                                    // m * 2^-shift in [4, 8)
        if (rexp + shift > 120) shift = 120 - rexp;
        if (rexp + shift < -120) shift = -120 - rexp;
        a_scale = ldexpf(1.f, -shift);
        rexp += shift;
      }
    }
  }
  tmem_ld32_issue(t0, ra);
  uint32_t mw_next = 0xffffffffu;
  if (MASK) mw_next = mask_word<W>(mask_tile, st.mask_slot, (int)e.hh, e.row);
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    uint32_t (&r)[32] = (c & 1) ? rb : ra;
    tmem_ld_wait();
    if (c + 1 < NC) tmem_ld32_issue(t0 + (uint32_t)(c + 1) * 64u, (c & 1) ? ra : rb);
    const uint32_t mw = mw_next;
    if (MASK && c + 1 < NC) mw_next = mask_word<W>(mask_tile, st.mask_slot, (c + 1) * 2 + (int)e.hh, e.row);
    const int col0 = c * 64 + (int)e.hh * 32;
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = X ? __uint_as_float(r[i]) * in_scale : __uint_as_float(r[i]);
    if (EV) {
#pragma unroll
      for (int i4 = 0; i4 < 8; ++i4) {
        const float4 ws = *reinterpret_cast<const float4*>(wsig_s + col0 + 4 * i4);
        v[4 * i4] += gsp * ws.x; v[4 * i4 + 1] += gsp * ws.y; v[4 * i4 + 2] += gsp * ws.z; v[4 * i4 + 3] += gsp * ws.w;
      }
    }
    if (PRODUCE) {
      RowPack<X> rp;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float a = (!MASK || mask_bit(mw, 2 * i)) ? v[2 * i] : 0.f;
        float b = (!MASK || mask_bit(mw, 2 * i + 1)) ? v[2 * i + 1] : 0.f;
        if (X) { a *= a_scale; b *= a_scale; }
        rp.set(i, a, b);
      }
      rp.store(sm, c, e.row, e.hh);
      publish_chunk(sm, c, e.lane);   // the MMA warp can start the next layer on this chunk while we reduce below
    }
    if (COLSUM) {
      if (X) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] *= row_scale;
      }
      const float cs = warp_colsum32(v, e.lane);
      atomicAdd(colsum + st.latent_slot * 256 + col0 + e.lane, cs);
    }
  }
}

template <bool X, int W>
__device__ __forceinline__ void bwd_epilogue_dispatch(const SmemT<X>& sm, const Step& st, uint32_t half, const EpiCtx& e,
                                                      const uint32_t* mask_tile, float gsp, int& rexp) {
  if (st.epi == EPI_B_EV) {
    bwd_epilogue<true, false, false, true, X, W>(sm, st, half, e, mask_tile, gsp, rexp);
  } else if (st.latent_slot >= 0) {
    if (st.produce_a) bwd_epilogue<false, true, true, true, X, W>(sm, st, half, e, mask_tile, gsp, rexp);
    else bwd_epilogue<false, true, false, false, X, W>(sm, st, half, e, mask_tile, gsp, rexp);
  } else {
    bwd_epilogue<false, false, true, true, X, W>(sm, st, half, e, mask_tile, gsp, rexp);
  }
}

// ------------------------------------------------------------------------------------------ backward kernel
template <bool X, int W>
__global__ void __launch_bounds__(kThreads, 1) tc_bwd_kernel(const __grid_constant__ Params p) {
  using MP = Map<X>;
  extern __shared__ uint8_t smem_raw[];
  SmemT<X> sm;
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t tmem_base;
  {
    const uint32_t raw = smem_u32(smem_raw);
    uint8_t* b = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
    float* colsum0 = reinterpret_cast<float*>(b + MP::SM_TAB + MP::TAB_BIAS);
    for (uint32_t i = tid; i < kMaxLatentSlots * 256; i += kThreads) colsum0[i] = 0.f;
    float* wsig_s = reinterpret_cast<float*>(b + MP::SM_TAB + MP::TAB_WSIG);
    for (int i = tid; i < W; i += kThreads) wsig_s[i] = __ldg(p.wsig + i);
    float* w2_s = reinterpret_cast<float*>(b + MP::SM_TAB + MP::TAB_W2);
    for (int i = tid; i < 3 * W / 2; i += kThreads) w2_s[i] = __ldg(p.w2 + i);
  }
  kernel_prologue(sm, smem_raw, tid, warp, tmem_base);
  const int64_t M = rows_present(p);
  const int64_t n_tiles = p.live ? 2 * (int64_t)__ldg(p.n_live) : (M + kTileM - 1) / kTileM;   // work items (work_tile)

  if (warp == 8) {
    producer_loop<X>(p, sm, n_tiles, lane);
  } else if (warp == 9) {
    mma_loop<X>(p, sm, n_tiles, lane, tmem_base);
  } else {
    EpiCtx e;
    e.lane = lane; e.hh = warp >> 2; e.row = (warp & 3u) * 32u + lane; e.lane_field = ((warp & 3u) * 32u) << 16;
    e.tmem_base = tmem_base;
    float* xyz_part = sm.tab(MP::TAB_PART);          // [2][128][3]
    float* colsum = sm.tab(MP::TAB_BIAS);            // [slots][256]
    const float* w2_s = sm.tab(MP::TAB_W2);
    uint32_t gstep = 0, acc_cnt[2] = {0, 0};
    const int nslots = p.prog.n_mask_slots;
    for (int64_t j = blockIdx.x; j < n_tiles; j += gridDim.x) {
      const int64_t tile = work_tile(p, j);
      e.grow = tile * kTileM + e.row;
      e.valid = e.grow < M;
      const int64_t crow = e.valid ? e.grow : M - 1;
      const int64_t obj = obj_of_tile(p, tile);  // tiles never straddle objects (checked on the host)
      const uint32_t* mask_tile = p.masks + (size_t)tile * nslots * (W / 32) * 128;
      const float gsg = e.valid ? __ldg(p.g_sigma + e.grow) : 0.f;
      float gsp = gsg * (-expm1f(-__ldg(p.sigma_in + crow)));   // d softplus = 1 - exp(-softplus)
      float g3[3] = {0.f, 0.f, 0.f};
      if (e.valid) { g3[0] = __ldg(p.g_rgb + 3 * e.grow); g3[1] = __ldg(p.g_rgb + 3 * e.grow + 1); g3[2] = __ldg(p.g_rgb + 3 * e.grow + 2); }
      // split mode: the row's gradient is carried in units of 2^rexp (exact; the pass is linear in it): start with the upstream
      // gradient at [16, 32)
      int rexp = 0;
      if (X) {
        const float m = fmaxf(fmaxf(fabsf(gsp), fabsf(g3[0])), fmaxf(fabsf(g3[1]), fabsf(g3[2])));
        if (m > 0.f && m < 3.0e38f) {
          int ex;
          frexpf(m, &ex);
          ex = ex < -100 ? -100 : (ex > 100 ? 100 : ex);
          rexp = ex - 5;
          const float inv = ldexpf(1.f, -rexp);
          g3[0] *= inv; g3[1] *= inv; g3[2] *= inv;
        }
      }
      // ---- prologue: d pre-activation of rgb.0 = (g_rgb W2) * mask -> A chunks 0 .. W / 128 - 1 (W / 2 columns)
      {
#pragma unroll
        for (int c = 0; c < W / 128; ++c) {
          const int col0 = c * 64 + (int)e.hh * 32;
          const uint32_t mw = mask_word<W>(mask_tile, p.r0_mask_slot, c * 2 + e.hh, e.row);
          RowPack<X> rp;
#pragma unroll
          for (int i4 = 0; i4 < 8; ++i4) {
            const float4 w0 = *reinterpret_cast<const float4*>(w2_s + col0 + 4 * i4);
            const float4 w1 = *reinterpret_cast<const float4*>(w2_s + W / 2 + col0 + 4 * i4);
            const float4 w2 = *reinterpret_cast<const float4*>(w2_s + W + col0 + 4 * i4);
            float v[4] = {g3[0] * w0.x + g3[1] * w1.x + g3[2] * w2.x, g3[0] * w0.y + g3[1] * w1.y + g3[2] * w2.y,
                          g3[0] * w0.z + g3[1] * w1.z + g3[2] * w2.z, g3[0] * w0.w + g3[1] * w1.w + g3[2] * w2.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) if (!mask_bit(mw, 4 * i4 + u)) v[u] = 0.f;
            rp.set(2 * i4, v[0], v[1]);
            rp.set(2 * i4 + 1, v[2], v[3]);
          }
          rp.store(sm, c, e.row, e.hh);
          publish_chunk(sm, c, lane);
        }
      }
      for (int si = 0; si < p.prog.n_steps; ++si, ++gstep) {
        const Step& st = p.prog.s[si];
        const uint32_t half = gstep & 1u;
        mbar_wait(sm.bar(BAR_ACC + half), acc_cnt[half] & 1u);
        acc_cnt[half]++;
        tc_fence_after();
        const float out_scale = X ? ldexpf(kWScaleInv, rexp) : 1.f;   // accumulator -> true gradient
        if (st.epi == EPI_B_XYZ) {
          // acc = d PE(xyz) (64 columns): fold to d xyz.  g_x = g_0 + sum_f 2^f (g_sin,f cos_f - g_cos,f sin_f)
          uint32_t r[32];
          tmem_ld32(e.tmem_base + half * 256u + e.hh * 32u + e.lane_field, r);
          const float x[3] = {__ldg(p.xyz + 3 * crow), __ldg(p.xyz + 3 * crow + 1), __ldg(p.xyz + 3 * crow + 2)};
          float s[10][3], c[10][3];
          trig_ladder<10, X>(x, s, c);
          float g[3] = {0.f, 0.f, 0.f};
          if (e.hh == 0) {  // columns 0..31: x (0-2), sin f=0..8 (3-29), sin f=9 a=0,1 (30,31)
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float gv = __uint_as_float(r[i]);
              if (i < 3) g[i] += gv;
              else { const int f = (i - 3) / 3, a = (i - 3) % 3; g[a] += gv * (float)(1 << f) * c[f][a]; }
            }
          } else {        // columns 32..63: sin f=9 a=2 (32), cos f=0..9 (33-62), pad (63)
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float gv = __uint_as_float(r[i]);
              const int col = 32 + i;
              if (col == 32) g[2] += gv * 512.f * c[9][2];
              else if (col < 63) { const int f = (col - 33) / 3, a = (col - 33) % 3; g[a] -= gv * (float)(1 << f) * s[f][a]; }
            }
          }
#pragma unroll
          for (int a = 0; a < 3; ++a) xyz_part[(e.hh * 128 + e.row) * 3 + a] = g[a] * out_scale;
          tc_fence_before();
          continue;
        }
        if (st.epi == EPI_B_EV && st.n2_out && e.hh == 0) {
          // group 2 accumulators (other TMEM half, columns 0..31) = d PE(viewdir): fold to d viewdir (deg 4: 27 columns)
          uint32_t r[32];
          tmem_ld32(e.tmem_base + (half ^ 1u) * 256u + e.lane_field, r);
          const float d[3] = {__ldg(p.viewdir + 3 * crow), __ldg(p.viewdir + 3 * crow + 1), __ldg(p.viewdir + 3 * crow + 2)};
          float s[4][3], c[4][3];
          trig_ladder<4, X>(d, s, c);
          float g[3] = {0.f, 0.f, 0.f};
#pragma unroll
          for (int i = 0; i < 27; ++i) {
            const float gv = __uint_as_float(r[i]);
            if (i < 3) g[i] += gv;
            else if (i < 15) { const int f = (i - 3) / 3, a = (i - 3) % 3; g[a] += gv * (float)(1 << f) * c[f][a]; }
            else { const int f = (i - 15) / 3, a = (i - 15) % 3; g[a] -= gv * (float)(1 << f) * s[f][a]; }
          }
          if (e.valid && p.g_viewdir) {
            p.g_viewdir[3 * e.grow] = g[0] * out_scale; p.g_viewdir[3 * e.grow + 1] = g[1] * out_scale; p.g_viewdir[3 * e.grow + 2] = g[2] * out_scale;
          }
        }
        bwd_epilogue_dispatch<X, W>(sm, st, half, e, mask_tile, gsp, rexp);
        tc_fence_before();
      }
      // ---- tile end: d xyz, and flush the latent column sums when the next tile belongs to another object
      const int64_t next = j + gridDim.x;
      const bool flush = next >= n_tiles || obj_of_tile(p, work_tile(p, next)) != obj;
      epi_bar_sync();
      if (p.g_xyz != nullptr && e.hh == 0 && e.valid) {
#pragma unroll
        for (int a = 0; a < 3; ++a) p.g_xyz[3 * e.grow + a] = xyz_part[e.row * 3 + a] + xyz_part[(128 + e.row) * 3 + a];
      }
      if (flush) {
        for (int sl = 0; sl < p.n_latent; ++sl) {
          const float v = colsum[sl * 256 + tid];
          if (v != 0.f && (W == 256 || tid < W)) atomicAdd(p.g_zlat + ((size_t)sl * p.B + obj) * W + tid, v);
          colsum[sl * 256 + tid] = 0.f;
        }
      }
      epi_bar_sync();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------ weight packing
struct PackJob {
  const float* src; int ld; int transposed; int n_valid; int n_pad; int k0; int k_limit; uint32_t dst_off;
  int n0;      // first output row (split mode: N half)
  int part;    // -1: bf16 image; 0 / 1: fp16 hi / lo image of kWScale * w
};
constexpr int kJobsPerLaunch = 64;
struct PackJobs { int n; PackJob j[kJobsPerLaunch]; };

// one block per job: dst[n][k] (128B-swizzled rows of 64 16-bit values) = src'(n0 + n, k0 + k), zero outside the valid range
__global__ void __launch_bounds__(256) pack_kernel(const __grid_constant__ PackJobs jobs, uint8_t* __restrict__ packed) {
  const PackJob& jb = jobs.j[blockIdx.x];
  for (int e = threadIdx.x; e < jb.n_pad * 64; e += blockDim.x) {
    int n, k;
    if (jb.transposed) { k = e / jb.n_pad; n = e % jb.n_pad; }  // consecutive threads walk the contiguous source dimension
    else { n = e / 64; k = e % 64; }
    const int kg = jb.k0 + k, ng = jb.n0 + n;
    float v = 0.f;
    if (ng < jb.n_valid && kg < jb.k_limit) v = jb.transposed ? jb.src[(size_t)kg * jb.ld + ng] : jb.src[(size_t)ng * jb.ld + kg];
    const uint32_t off = jb.dst_off + (uint32_t)n * 128u + ((((uint32_t)k >> 3) ^ ((uint32_t)n & 7u)) << 4) + ((uint32_t)k & 7u) * 2u;
    if (jb.part < 0) {
      *reinterpret_cast<__nv_bfloat16*>(packed + off) = __float2bfloat16_rn(v);
    } else {
      const float x = v * kWScale;
      const __half hi = __float2half_rn(x);
      *reinterpret_cast<__half*>(packed + off) = jb.part == 0 ? hi : __float2half_rn(x - __half2float(hi));
    }
  }
}

}  // namespace tc

// ------------------------------------------------------------------------------------------ host side
using namespace tc;

bool tc1_supported(const snb_handle_s* h, const char** why) {
  const snb_arch& a = h->arch;
  if (a.arch != SNB_ARCH_CODENERF) { *why = "bf16 mode covers the CodeNeRF/AutoRFMix/SUPNeRF decoder only"; return false; }
  if (a.W != 128 && a.W != 256) { *why = "the tensor-core back ends need W == 128 or W == 256"; return false; }
  if (a.num_xyz_freq != 10 || a.num_dir_freq != 4) { *why = "bf16 mode needs num_xyz_freq == 10 and num_dir_freq == 4"; return false; }
  if (a.shape_blocks + a.texture_blocks > kMaxLatentSlots) { *why = "the tensor-core back ends need shape_blocks + texture_blocks <= 10"; return false; }
  return true;
}

struct TcPlan {
  Program fwd, bwd_full, bwd_noxyz;
  std::vector<PackJob> jobs;
  uint32_t total_bytes = 0;
  int r0_slot = 0;
  bool split = false;   // fp16 (hi, lo) weight images of the split-precision mode
};

// one 64-wide K chunk of an MMA group's B operand: columns [k0, k0 + 64) of `src`, valid below k_limit
struct ChunkSrc { const float* src; int k0; int k_limit; };

static void add_chunk_list(TcPlan& pl, const std::vector<ChunkSrc>& chunks, int ld, bool transposed, int n_valid, int n_pad,
                           uint32_t* first_off) {
  *first_off = pl.total_bytes;
  PackJob j;
  j.ld = ld; j.transposed = transposed ? 1 : 0; j.n_valid = n_valid;
  const int nh = (pl.split && n_pad > 128) ? 128 : n_pad;
  auto push = [&](const ChunkSrc& c, int n0, int part) {
    j.src = c.src; j.k0 = c.k0; j.k_limit = c.k_limit; j.n_pad = nh; j.n0 = n0; j.part = part; j.dst_off = pl.total_bytes;
    pl.jobs.push_back(j);
    pl.total_bytes += (uint32_t)nh * 128u;
  };
  if (!pl.split) {
    for (const ChunkSrc& c : chunks) push(c, 0, -1);
    return;
  }
  // split mode, in the order the MMA warp consumes the stages (mma_loop): the chunks whose corrections go first -- per chunk and N half
  // the (hi, lo) pair --, their hi images once more for the leading products, then the remaining chunks' (hi, lo) pairs
  const int n = (int)chunks.size();
  const int n_corr = kOrder == 1 ? n : (kOrder == 2 ? n - 1 : 0);
  for (int c = 0; c < n_corr; ++c)
    for (int n0 = 0; n0 < n_pad; n0 += nh) { push(chunks[c], n0, 0); push(chunks[c], n0, 1); }
  for (int c = 0; c < n_corr; ++c)
    for (int n0 = 0; n0 < n_pad; n0 += nh) push(chunks[c], n0, 0);
  for (int c = n_corr; c < n; ++c)
    for (int n0 = 0; n0 < n_pad; n0 += nh) { push(chunks[c], n0, 0); push(chunks[c], n0, 1); }
}

static void add_chunks(TcPlan& pl, const float* src, int ld, bool transposed, int n_valid, int n_pad, int k_limit, int n_chunks,
                       uint32_t* first_off) {
  std::vector<ChunkSrc> chunks;
  for (int c = 0; c < n_chunks; ++c) chunks.push_back({src, c * 64, k_limit});
  add_chunk_list(pl, chunks, ld, transposed, n_valid, n_pad, first_off);
}

// chunks: the shared-memory A chunk of each K chunk, in order
static Step make_step(int epi, int n_out, const std::vector<int>& chunks, int mask_slot, int latent_slot, int produce_a,
                      const float* bias) {
  Step s{};
  s.epi = (int8_t)epi; s.n_out = (uint16_t)n_out; s.n_chunks = (uint16_t)chunks.size(); s.mask_slot = (int8_t)mask_slot;
  s.latent_slot = (int8_t)latent_slot; s.produce_a = (int8_t)produce_a; s.bias = bias; s.n2_out = 0;
  int i = 0;
  for (int c : chunks) s.a_chunk[i++] = (uint8_t)c;
  return s;
}

// Builds the forward / backward step programs and the weight-image packing jobs for the handle's current pointers.
static TcPlan build_plan(const snb_handle_s* h, bool split = false) {
  TcPlan pl;
  pl.split = split;
  const int Bs = h->arch.shape_blocks, Bt = h->arch.texture_blocks, W = h->arch.W, dv = h->d_dir(), dx = h->d_xyz();
  const int KC = W / 64;                           // K chunks of a hidden layer
  std::vector<int> hid(KC);                        // ... held in A chunks 0 .. KC - 1
  for (int c = 0; c < KC; ++c) hid[c] = c;
  std::vector<int> ev_chunks = {4};                // encoding_viewdir: PE(viewdir) in the AUX chunk, then the hidden chunks
  ev_chunks.insert(ev_chunks.end(), hid.begin(), hid.end());
  const std::vector<int> r0_chunks(hid.begin(), hid.begin() + W / 128);   // backward through rgb.0: its W / 2 outputs
  const auto& ly = h->layers;
  const int slot_vv = Bs + 1, slot_r = Bs + Bt + 2;
  pl.r0_slot = slot_r;
  Program& f = pl.fwd;
  f.n_steps = 0; f.n_mask_slots = Bs + Bt + 3;
  auto push = [](Program& pr, const Step& s) { pr.s[pr.n_steps++] = s; };
  {  // ---------------- forward
    Step s = make_step(EPI_RELU, W, {4}, 0, -1, 1, ly[h->iX].b);
    add_chunks(pl, ly[h->iX].w, dx, false, W, W, dx, 1, &s.w_off);
    push(f, s);
    for (int j = 1; j <= Bs; ++j) {
      s = make_step(EPI_RELU, W, hid, j, j - 1, 1, ly[h->iS(j)].b);   // effective bias slot j-1 = b + W zs_j
      add_chunks(pl, ly[h->iS(j)].w, W, false, W, W, W, KC, &s.w_off);
      push(f, s);
    }
    s = make_step(EPI_LINEAR_SIGMA, W, hid, -1, -1, 1, ly[h->iES].b);
    add_chunks(pl, ly[h->iES].w, W, false, W, W, W, KC, &s.w_off);
    push(f, s);
    s = make_step(EPI_RELU, W, ev_chunks, slot_vv, -1, 1, ly[h->iEV].b);
    {  // chunk 0 = the PE(viewdir) columns [W, W+dv) of encoding_viewdir, chunks 1..KC = its first W columns
      std::vector<ChunkSrc> chunks = {{ly[h->iEV].w + W, 0, dv}};
      for (int c = 0; c < KC; ++c) chunks.push_back({ly[h->iEV].w, c * 64, W});
      add_chunk_list(pl, chunks, W + dv, false, W, W, &s.w_off);
    }
    push(f, s);
    for (int j = 1; j <= Bt; ++j) {
      s = make_step(EPI_RELU, W, hid, slot_vv + j, Bs + j - 1, 1, ly[h->iT(j)].b);
      add_chunks(pl, ly[h->iT(j)].w, W, false, W, W, W, KC, &s.w_off);
      push(f, s);
    }
    s = make_step(EPI_RGB_HEAD, W / 2, hid, slot_r, -1, 0, ly[h->iR0].b);
    add_chunks(pl, ly[h->iR0].w, W, false, W / 2, W / 2, W, KC, &s.w_off);
    push(f, s);
  }
  {  // ---------------- backward (B operand = W^T: n = input unit, k = output unit)
    Program& b = pl.bwd_full;
    b.n_steps = 0; b.n_mask_slots = f.n_mask_slots;
    Step s = make_step(EPI_B_MASK, W, r0_chunks, slot_vv + Bt, -1, 1, nullptr);           // through rgb.0 -> d T_Bt, mask of T_Bt
    add_chunks(pl, ly[h->iR0].w, W, true, W, W, W / 2, W / 128, &s.w_off);
    push(b, s);
    for (int j = Bt; j >= 1; --j) {                                                        // through texture_layer_j
      s = make_step(EPI_B_MASK, W, hid, slot_vv + j - 1, Bs + j - 1, 1, nullptr);
      add_chunks(pl, ly[h->iT(j)].w, W, true, W, W, W, KC, &s.w_off);
      push(b, s);
    }
    s = make_step(EPI_B_EV, W, hid, -1, -1, 1, nullptr);                                   // through encoding_viewdir
    add_chunks(pl, ly[h->iEV].w, W + dv, true, W, W, W, KC, &s.w_off);
    add_chunks(pl, ly[h->iEV].w + W, W + dv, true, dv, 64, W, KC, &s.w2_off);
    s.n2_out = 64;
    push(b, s);
    s = make_step(EPI_B_MASK, W, hid, Bs, -1, 1, nullptr);                                 // through encoding_shape, mask of H_Bs
    add_chunks(pl, ly[h->iES].w, W, true, W, W, W, KC, &s.w_off);
    push(b, s);
    for (int j = Bs; j >= 1; --j) {                                                        // through shape_layer_j
      s = make_step(EPI_B_MASK, W, hid, j - 1, j - 1, 1, nullptr);
      add_chunks(pl, ly[h->iS(j)].w, W, true, W, W, W, KC, &s.w_off);
      push(b, s);
    }
    s = make_step(EPI_B_XYZ, 64, hid, -1, -1, 0, nullptr);                                 // through encoding_xyz -> d PE(xyz)
    add_chunks(pl, ly[h->iX].w, dx, true, dx, 64, W, KC, &s.w_off);
    push(b, s);
    // variant without pose gradients: drop the last step and the d PE(viewdir) group; the new last step feeds nobody
    pl.bwd_noxyz = b;
    Program& n = pl.bwd_noxyz;
    n.n_steps = b.n_steps - 1;
    n.s[n.n_steps - 1].produce_a = 0;
    for (int i = 0; i < n.n_steps; ++i) if (n.s[i].epi == EPI_B_EV) n.s[i].n2_out = 0;
  }
  return pl;
}

size_t tc1_image_bytes(const snb_handle_s* h, bool split) { return build_plan(h, split).total_bytes; }

int tc1_pack_weights(const snb_handle_s* h, bool split, void* packed, cudaStream_t st) {
  TcPlan pl = build_plan(h, split);
  for (size_t i = 0; i < pl.jobs.size(); i += kJobsPerLaunch) {
    PackJobs jb;
    jb.n = (int)std::min<size_t>(kJobsPerLaunch, pl.jobs.size() - i);
    for (int k = 0; k < jb.n; ++k) jb.j[k] = pl.jobs[i + k];
    pack_kernel<<<jb.n, 256, 0, st>>>(jb, (uint8_t*)packed);
    SNB_LAUNCH_CHECK();
  }
  return 0;
}

static void fill_common(Params& p, const snb_handle_s* h, const void* packed, const float* xyz, const float* viewdir, int64_t M,
                        int64_t B, const float* zlat, uint32_t* masks, const int64_t* m_dev, const int32_t* tile_start) {
  p = Params{};
  p.xyz = xyz; p.viewdir = viewdir; p.M = M; p.B = B; p.rows_per_obj = M / B;
  p.packed = (const uint8_t*)packed; p.zlat = zlat; p.masks = masks;
  p.wsig = h->layers[h->iSG].w; p.bsig = h->layers[h->iSG].b;
  p.n_latent = h->arch.shape_blocks + h->arch.texture_blocks;
  p.ev_step = h->arch.shape_blocks + 2;  // forward step index of encoding_viewdir
  p.w2 = h->layers[h->iR2].w; p.b2 = h->layers[h->iR2].b;
  p.m_dev = m_dev; p.tile_start = tile_start;
}

static int tc_grid(int64_t M) {
  static const int cap = [] { const char* e = getenv("SNB_TC_GRID_CAP"); return e ? atoi(e) : 0; }();   // tuning: fewer CTAs than SMs
  int sms = sm_count();
  if (cap > 0 && cap < sms) sms = cap;
  const int64_t t = (M + kTileM - 1) / kTileM;
  return (int)(t < sms ? t : sms);
}

// forward: zlat holds the per-object effective biases (latent_forward_fused's ebias)
template <bool X>
int tc1_launch_fwd(const snb_handle_s* h, const void* packed, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const float* ebias, uint32_t* masks, float* sigma, float* rgb, cudaStream_t st, const int64_t* m_dev,
                   const int32_t* tile_start) {
  TcPlan pl = build_plan(h, X);
  Params p;
  fill_common(p, h, packed, xyz, viewdir, M, B, ebias, masks, m_dev, tile_start);
  p.sigma = sigma; p.rgb = rgb; p.dbg = h->dbg_acts;
  p.prog = pl.fwd;
  auto* kernel = h->arch.W == 128 ? tc_fwd_kernel<X, 128> : tc_fwd_kernel<X, 256>;   // tc1_supported: W is 128 or 256
  SNB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Map<X>::SM_ALLOC));
  kernel<<<tc_grid(M), kThreads, Map<X>::SM_ALLOC, st>>>(p);
  return 0;
}

template <bool X>
int tc1_launch_bwd(const snb_handle_s* h, const void* packed, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const float* zlat, uint32_t* masks, const float* sigma, const float* g_sigma, const float* g_rgb, float* g_xyz,
                   float* g_viewdir, float* g_zlat, cudaStream_t st, const int64_t* m_dev, const int32_t* tile_start,
                   const int32_t* live, const int32_t* n_live) {
  TcPlan pl = build_plan(h, X);
  Params p;
  fill_common(p, h, packed, xyz, viewdir, M, B, zlat, masks, m_dev, tile_start);
  p.live = live; p.n_live = n_live;
  p.sigma_in = sigma; p.g_sigma = g_sigma; p.g_rgb = g_rgb; p.g_xyz = g_xyz; p.g_viewdir = g_viewdir; p.g_zlat = g_zlat;
  p.r0_mask_slot = pl.r0_slot;
  p.prog = g_xyz ? pl.bwd_full : pl.bwd_noxyz;
  auto* kernel = h->arch.W == 128 ? tc_bwd_kernel<X, 128> : tc_bwd_kernel<X, 256>;
  SNB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Map<X>::SM_ALLOC));
  kernel<<<tc_grid(M), kThreads, Map<X>::SM_ALLOC, st>>>(p);
  return 0;
}

#define SNB_TC1_LAUNCHERS(X)                                                                                                       \
  template int tc1_launch_fwd<X>(const snb_handle_s*, const void*, const float*, const float*, int64_t, int64_t, const float*,     \
                                 uint32_t*, float*, float*, cudaStream_t, const int64_t*, const int32_t*);                         \
  template int tc1_launch_bwd<X>(const snb_handle_s*, const void*, const float*, const float*, int64_t, int64_t, const float*,     \
                                 uint32_t*, const float*, const float*, const float*, float*, float*, float*, cudaStream_t,        \
                                 const int64_t*, const int32_t*, const int32_t*, const int32_t*);
SNB_TC1_LAUNCHERS(false)
SNB_TC1_LAUNCHERS(true)
#undef SNB_TC1_LAUNCHERS

}  // namespace snb
