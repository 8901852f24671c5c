// K2 / K2b, SNB_PREC_BF16 back end, second generation: TWO 128-sample tiles in flight per CTA.
//
// Measured on B200 (profiles/r1_ubench_mma_latency.txt): a tcgen05.mma batch costs ~450-600 cycles of issue -> commit ->
// mbarrier -> waiting-warp latency on top of its 128 cycles per M128xN256xK16 instruction, and the first-generation kernel
// (mlp_tc.cu, one tile per CTA) serialises that latency AND most of each layer's epilogue behind the layer's MMAs
// (ncu: tensor pipe 39 % active, epilogue warps 37 % of their time waiting for the accumulator).  Here every CTA owns
// two tile slots with their own shared-memory A operand (4 x 16 KB chunks), their own 256-column TMEM accumulator and
// their own group of 8 epilogue warps; the single MMA-issuer warp alternates  slot 0 layer l, slot 1 layer l, slot 0
// layer l+1, ...  so the tensor pipe always has the other slot's layer to run while one slot is in its epilogue.
//
// Warp roles (576 threads): warps 0-7 epilogue group of slot 0, warps 8-15 of slot 1 (warp w owns TMEM lanes
// 32*(w%4).. and the column half (w/4)%2 of every 64-column chunk), warp 16 weight producer (+ TMEM alloc), warp 17
// MMA issuer.  Weights: pre-tiled bf16 images, [N rows][32 k] per stage (64-byte swizzle, K-major), streamed L2 ->
// smem by cp.async.bulk through an mbarrier ring.  PE(xyz) is written into the slot's chunk 0.
//
// Two variants of both kernels (template parameter CG2):
//  * cta_group::1 (training mode with operand saves, or objects that do not own a multiple of 256 rows): M = 128 MMAs per CTA,
//    5 stages of 16 KB, every stage fetched from L2 once per 2-CTA cluster (half per CTA, multicast); encoding_viewdir runs as
//    two accumulating steps (y part, then PE(viewdir) written into chunk 0).
//  * cta_group::2 (frozen weights: the default): ONE M = 256 MMA spans the CTA pair; each CTA holds its 128-row A operand and its
//    half of every stage (8 stages of 8 KB); the leader CTA's MMA warp issues for both SMs and collects both CTAs' epilogue
//    arrivals, the peer's MMA warp relays its stage completions; in the forward encoding_viewdir is one step whose last stage
//    multiplies a per-slot PE(viewdir) tile.  Same arithmetic, bit-identical sigma / rgb (tests/test_gpu_bf16.py).
#include "common.cuh"
#include "decoder.h"
#include "tc_ptx.cuh"
#include "rb_rows.cuh"
#include <algorithm>
#include <stdlib.h>
#include <utility>
#include <vector>

namespace snb {
namespace tc2 {
using namespace tc;

constexpr int kThreads = 576;
constexpr int kCluster = 2;               // CTAs per cluster: every weight stage is fetched from L2 ONCE per cluster (each CTA loads
                                          // 1/kCluster of it and multicasts it to all): L2 -> SM weight traffic / kCluster
constexpr uint16_t kClusterMask = (uint16_t)((1u << kCluster) - 1u);
constexpr int kRing = 5;
constexpr uint32_t kStageBytes = 16384;   // [256 n][32 k] bf16
// cta_group::2 variant (CG2): one M = 256 MMA spans the CTA pair, each CTA holds ITS half of every weight stage ([128 n][32 k],
// 8 KB), so the ring is twice as deep in the same shared memory and the tensor core reads 4 KB (A) + 4 KB (B) per instruction
// per SM instead of 4 + 8: the epilogue's operand stores get half of the shared-memory bandwidth instead of a quarter.
constexpr int kRing2 = 8;                 // (10 stages measured no faster: 39 188 vs 39 164 cycles per forward tile pair)
constexpr uint32_t kStageBytes2 = 8192;
constexpr int kRingMax = 10;              // barrier layout (both variants)
static_assert(kRing * kStageBytes >= kRing2 * kStageBytes2, "ring footprint");
constexpr int kMaxSteps = 13;
constexpr int kMaxLat = 4;                // shape_blocks + texture_blocks <= 4 (every shipped config: 3 + 1)

constexpr uint32_t SM_RING = 8 * kChunkBytes;                    // A chunks [slot][4]
constexpr uint32_t SM_PEV = SM_RING + kRing2 * kStageBytes2;      // CG2 forward: PE(viewdir) A tile per slot, [128][32] bf16, 64-byte swizzle
constexpr uint32_t kPevBytes = 8192;
static_assert(SM_PEV + 2 * kPevBytes <= SM_RING + kRing * kStageBytes, "the PE(viewdir) tiles live inside the ring footprint");
constexpr uint32_t SM_TAB = SM_RING + kRing * kStageBytes;
constexpr uint32_t TAB_BIAS = 0;                                 // tile-end scratch: [slot][128][4] floats (the column halves' partial heads / d xyz)
constexpr uint32_t TAB_LAT = TAB_BIAS + 4 * 1024;                // fwd: [128][16] bf16 all-ones A tile (4 KB); bwd: [slot][kMaxLat][256] latent column sums
constexpr uint32_t kBiasStageRowBytes = 32;                       // bias stage: [N rows][16 k] bf16, 32-byte swizzle
constexpr uint32_t TAB_WSIG = TAB_LAT + 2 * kMaxLat * 1024;      // [256]
constexpr uint32_t TAB_W2 = TAB_WSIG + 1024;                     // [3][128]
constexpr uint32_t TAB_BYTES = TAB_W2 + 1536;
constexpr uint32_t SM_BARS = SM_TAB + TAB_BYTES;
constexpr uint32_t SM_TOTAL = SM_BARS + 256;
constexpr uint32_t SM_ALLOC = SM_TOTAL + 1024;                   // + alignment slack
static_assert(SM_ALLOC <= 232448, "shared memory budget");

enum Epi : int { F_RELU = 0, F_SIGMA = 1, F_PEV = 2, F_RGB = 3, B_MASK = 4, B_VD = 5, B_EV = 6, B_XYZ = 7, F_NONE = 8 };
constexpr int BAR_WFULL = 0, BAR_WEMPTY = kRingMax, BAR_READY = 2 * kRingMax, BAR_ACC = 2 * kRingMax + 2;   // 24 barriers = 192 B
constexpr uint32_t kTmemSlotOff = 240;    // inside the 256-byte barrier block

struct Step {
  uint32_t w_off;            // byte offset of the step's first weight stage in the packed buffer
  uint16_t n_stages, n_out;  // K / 32, N
  int8_t epi, mask_slot, latent_slot, bias_row, dbg_idx, accumulate, produce_a, colsum;
  int8_t bias_stage;         // 0 none; 1 static image right after the step's weight stages; 2 per-object image of latent_slot (fwd only)
  int8_t save_chunks;        // training mode: number of 16 KB A-operand chunks of this step kept for the weight-gradient kernels (0 = none)
  int8_t tail_pev;           // 1: the step's LAST weight stage multiplies the slot's PE(viewdir) tile instead of the next chunk half
  uint8_t pad_[1];
  uint32_t save_off;         // ... and their byte offset inside the tile's save block
};

struct Program {
  int n_steps, n_mask_slots;
  int pev;                   // 1: encoding_viewdir is ONE step (y columns + PE(viewdir) columns); the epilogue groups keep PE(viewdir) of
                             // their tile in the slot's PEV tile (written with the tile's PE(xyz))
  uint32_t save_tile_bytes;  // size of one tile's save block (training mode)
  Step s[kMaxSteps];
};

struct Params {
  const float* xyz; const float* viewdir;
  int64_t M, rows_per_obj, B;
  const uint8_t* packed;
  const uint8_t* eimg;          // fwd: per-object effective-bias stage images [(Bs+Bt)][B][256 x 32 B] (latent.cu)
  const float* wsig; const float* bsig; const float* w2; const float* b2;
  uint32_t* masks;              // [tile][slot][8 words][128 rows]
  float* sigma; float* rgb; float* dbg;
  const float* sigma_in; const float* g_sigma; const float* g_rgb;
  float* g_xyz; float* g_viewdir; float* g_zlat;   // g_zlat [(Bs+Bt)][B][256], accumulated with atomics
  int r0_mask_slot, n_latent;
  const int64_t* m_dev;   // optional: the number of rows actually present (<= M), read on the device -- the fused render compacts
                          // the samples of rays that miss the box on the GPU and never learns the count on the host
  const int32_t* tile_start;   // optional (batched render): B + 1 ascending even tile offsets, object b owns tiles [tile_start[b], tile_start[b+1])
  const int32_t* live;         // optional, backward: the 256-row super tiles to run, ascending (decoder.h: DeviceRows) ...
  const int32_t* n_live;       // ... and their count, on the device
  rb::RowSrc rs;               // forward, batched render (K1): rs.rays8 != NULL -> the epilogue warps compute their rows' sample
                               // coordinates from the rays (32 B per ray + 4 B of jitter per row) instead of reading xyz / viewdir
  uint8_t* save;      // training mode (weight gradients wanted): [tile][Program::save_tile_bytes] copies of every step's A operand
  long long* trace;   // timing experiments only: CTA 0 writes clock64 stamps [pair][step][slot][4] = READY seen, MMAs issued, ACC seen, published
  Program prog;
};

// K-major, 64-byte-swizzled operand tile: rows 64 B apart, 8-row atoms 512 B apart (SBO), descriptor version 1.
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}

// K-major, 32-byte-swizzled tile of K = 16: rows 32 B apart, 8-row atoms 256 B apart (SBO).  Used for the bias stage (B) and
// the all-ones A tile, both invariant under the swizzle's exchange of a row's two 16-byte units.
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(256u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;
  return d;
}

struct Smem {
  uint8_t* base;
  uint32_t base_u32;
  __device__ uint8_t* chunk(uint32_t slot, int c) const { return base + (slot * 4u + (uint32_t)c) * kChunkBytes; }
  __device__ uint32_t chunk_u32(uint32_t slot, int c) const { return base_u32 + (slot * 4u + (uint32_t)c) * kChunkBytes; }
  __device__ uint32_t stage_u32(uint32_t s) const { return base_u32 + SM_RING + s * kStageBytes; }
  __device__ uint32_t stage2_u32(uint32_t s) const { return base_u32 + SM_RING + s * kStageBytes2; }
  __device__ uint8_t* pev(uint32_t slot) const { return base + SM_PEV + slot * kPevBytes; }
  __device__ uint32_t pev_u32(uint32_t slot) const { return base_u32 + SM_PEV + slot * kPevBytes; }
  __device__ float* tab(uint32_t off) const { return reinterpret_cast<float*>(base + SM_TAB + off); }
  __device__ uint32_t bar(int i) const { return base_u32 + SM_BARS + 8u * i; }
};

struct EpiCtx {
  uint32_t lane, hh, row, lane_field, tmem, slot;
  int64_t grow;
  bool valid;
};

__device__ __forceinline__ uint32_t mask_word(const uint32_t* mask_tile, int slot, int word, uint32_t row) {
  return __ldg(mask_tile + ((size_t)slot * 8 + word) * 128 + row);
}

__device__ __forceinline__ void store_row32(uint8_t* chunk, uint32_t row, uint32_t hh, const uint32_t (&pk)[16]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    uint4 q = make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
    *reinterpret_cast<uint4*>(chunk + swz(row, hh * 4 + u)) = q;
  }
}

// 16 columns (two 16-byte units, `unit0` and `unit0 + 1`) of one row
__device__ __forceinline__ void store_row16(uint8_t* chunk, uint32_t row, uint32_t unit0, const uint32_t (&pk)[8]) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    uint4 q = make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
    *reinterpret_cast<uint4*>(chunk + swz(row, unit0 + u)) = q;
  }
}

__device__ __forceinline__ void group_bar(uint32_t slot) { asm volatile("bar.sync %0, 256;" ::"r"(slot + 1) : "memory"); }

// ---- cluster-scope barrier helpers (CG2: the leader CTA's MMA warp waits for arrivals from BOTH CTAs of the pair)
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// this thread's smem writes (generic proxy) and TMEM reads are done: make them visible to the tensor core and tell the MMA warp
// (CG2: the MMA warp of the pair's leader CTA, through its cluster-mapped READY barrier `ready_leader`)
template <bool CG2>
__device__ __forceinline__ void publish(const Smem& sm, uint32_t slot, uint32_t lane, uint32_t ready_leader) {
  tc_fence_before();
  fence_async_smem();
  __syncwarp();
  if (lane == 0) {
    if (CG2) mbar_arrive_cluster(ready_leader);
    else mbar_arrive(sm.bar(BAR_READY + slot));
  }
}

// ------------------------------------------------------------------------------------------ producer / MMA roles
// Both roles run WARP-UNIFORMLY (all 32 lanes execute the loops; one elected lane issues the async instruction inside the
// asm block).  With the instructions inside an `if (lane == 0)` region nvcc keeps descriptors in vector registers and wraps
// every UTCHMMA / UBLKCP in an ELECT + 7 x R2UR + BRA.U.ANY waterfall: ~65 dependent instructions per two MMAs, which made
// the MMA issuer itself the bottleneck (580 cycles per 256-cycle stage, profiles/r1_trace_v2_first.txt).
__device__ __forceinline__ void bulk_g2s_elect(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "{\n"
      ".reg .pred e;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%3], %2;\n"
      "@e cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
      "}" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Weight stage shared by the cluster: this CTA expects the WHOLE stage on its own full barrier, fetches its 1/kCluster part and
// multicasts it to the same smem offset (and the same barrier offset) of every CTA of the cluster.
__device__ __forceinline__ void bulk_g2s_multicast_elect(uint32_t dst, const void* src, uint32_t part_bytes, uint32_t total_bytes,
                                                         uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "{\n"
      ".reg .pred e;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%4], %3;\n"
      "@e cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%4], %5;\n"
      "}" ::"r"(dst), "l"(src), "r"(part_bytes), "r"(total_bytes), "r"(bar), "h"(cta_mask) : "memory");
}
// smem -> global bulk copy of an operand tile (training mode), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n cp.async.bulk.commit_group;"
               ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_elect(uint32_t bar) {
  asm volatile(
      "{\n"
      ".reg .pred e;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "@e mbarrier.arrive.shared::cta.b64 _, [%0];\n"
      "}" ::"r"(bar) : "memory");
}
// two K=16 MMAs of one 32-k weight stage (A and B advance by 32 bytes = 2 descriptor units), then release the stage
__device__ __forceinline__ void umma_stage_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate,
                                                 uint32_t empty_bar) {
  asm volatile(
      "{\n"
      ".reg .pred e, p, t;\n"
      ".reg .b64 a1, b1;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.eq.b32 t, 0, 0;\n"
      "add.s64 a1, %1, 2;\n"
      "add.s64 b1, %2, 2;\n"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, t;\n"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;\n"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(empty_bar), "h"(kClusterMask) : "memory");
}
// one accumulating K=16 MMA (the bias stage: ones x [bias_hi, bias_mid, bias_lo, 0...]), then release the stage
__device__ __forceinline__ void umma_bias_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t empty_bar) {
  asm volatile(
      "{\n"
      ".reg .pred e, t;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "setp.eq.b32 t, 0, 0;\n"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, t;\n"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%4], %5;\n"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(empty_bar), "h"(kClusterMask) : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n"
      ".reg .pred e;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
      "}" ::"r"(bar) : "memory");
}

__device__ __forceinline__ int64_t rows_present(const Params& p) { return p.m_dev ? __ldg(p.m_dev) : p.M; }

// object that owns a tile: uniform rows per object, or (batched render) a search in the ascending tile offsets (B + 1 ints in L1)
__device__ __forceinline__ int64_t obj_of_tile(const Params& p, int64_t tile) {
  if (p.tile_start == nullptr) return (tile * kTileM) / p.rows_per_obj;
  int lo = 0, hi = (int)p.B;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((int64_t)__ldg(p.tile_start + mid) <= tile) lo = mid; else hi = mid;
  }
  return lo;
}

// ---- cta_group::2 forms: issued by the leader CTA only; A = [128 rows][K] in EACH CTA (same smem offset), B = each CTA's half of
// the N rows, D = 128 lanes x N columns in each CTA's TMEM; commits multicast to the same barrier offset in both CTAs.
__device__ __forceinline__ void umma2_stage_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate,
                                                  uint32_t empty_bar) {
  asm volatile(
      "{\n"
      ".reg .pred e, p, t;\n"
      ".reg .b64 a1, b1;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.eq.b32 t, 0, 0;\n"
      "add.s64 a1, %1, 2;\n"
      "add.s64 b1, %2, 2;\n"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], a1, b1, %3, t;\n"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], %6;\n"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(empty_bar), "h"(kClusterMask) : "memory");
}
__device__ __forceinline__ void umma2_bias_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t empty_bar) {
  asm volatile(
      "{\n"
      ".reg .pred e, t;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "setp.eq.b32 t, 0, 0;\n"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, t;\n"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%4], %5;\n"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(empty_bar), "h"(kClusterMask) : "memory");
}
__device__ __forceinline__ void umma2_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n"
      ".reg .pred e;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n"
      "}" ::"r"(bar), "h"(kClusterMask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster_elect(uint32_t cluster_addr) {
  asm volatile(
      "{\n"
      ".reg .pred e;\n"
      "elect.sync _|e, 0xffffffff;\n"
      "@e mbarrier.arrive.shared::cluster.b64 _, [%0];\n"
      "}" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// Tile owned by (cluster-uniform pair index pair0, CTA rank, slot).  CG1: every CTA owns a pair of consecutive tiles.  CG2: a slot
// is one 256-row super tile of the cluster and the CTA's rank picks its 128-row half (so that both halves share the B operand,
// including the per-object bias stage: the host only selects CG2 when objects own multiples of 256 rows).
template <bool CG2>
__device__ __forceinline__ int64_t tile_index(int64_t pair0, uint32_t crank, uint32_t slot) {
  return CG2 ? 2 * pair0 + 2 * (int64_t)slot + crank : 2 * (pair0 + crank) + slot;
}


// (A variant in which slot 1 ran a few steps BEHIND slot 0, so that one slot's short steps and tile boundary fall next to the other
// slot's 256 x 256 layers, was measured: no gain -- the tensor pipe is in order, a short step's MMAs still queue behind the other
// slot's long step and the long step's epilogue is then covered by only the short step's MMAs -- and its generic item iterator
// cost the MMA warp its warp-uniform code: +9 % cycles per tile pair.  profiles/r1_trace_cg2.md.)
template <bool CG2>
__device__ __forceinline__ void producer_loop(const Params& p, const Smem& sm, int64_t n_pairs) {
  constexpr uint32_t RING = CG2 ? kRing2 : kRing;
  uint32_t stage = 0, ph = 0;
  const int64_t n_tiles = (rows_present(p) + kTileM - 1) / kTileM;
  const uint32_t crank = cluster_ctarank();
  // every CTA of a cluster runs the same number of iterations (a CTA past the last pair still streams its share of the weights)
  for (int64_t pair0 = (int64_t)blockIdx.x - crank; pair0 < n_pairs; pair0 += gridDim.x) {
    for (int si = 0; si < p.prog.n_steps; ++si) {
      const Step& st = p.prog.s[si];
      const uint32_t bytes = (uint32_t)st.n_out * 64u, part = bytes / kCluster;
      for (uint32_t slot = 0; slot < 2; ++slot) {
        const uint8_t* src = p.packed + st.w_off + crank * part;
        for (int j = 0; j < st.n_stages; ++j) {
          mbar_wait(sm.bar(BAR_WEMPTY + stage), ph ^ 1u);   // released by the MMA warps of ALL CTAs of the cluster
          if (CG2) bulk_g2s_elect(sm.stage2_u32(stage), src, part, sm.bar(BAR_WFULL + stage));   // this CTA's half of the N rows
          else bulk_g2s_multicast_elect(sm.stage_u32(stage) + crank * part, src, part, bytes, sm.bar(BAR_WFULL + stage), kClusterMask);
          src += bytes;
          if (++stage == RING) { stage = 0; ph ^= 1u; }
        }
        if (st.bias_stage) {   // CTA-local (not multicast): static image after the weight stages, or this tile's object's image
          const uint8_t* bsrc = p.packed + st.w_off + (uint32_t)st.n_stages * bytes;
          if (st.bias_stage == 2) {
            const int64_t tile = tile_index<CG2>(pair0, CG2 ? 0u : crank, slot);   // CG2: the super tile's object
            const int64_t obj = tile < n_tiles ? obj_of_tile(p, tile) : 0;
            bsrc = p.eimg + ((size_t)st.latent_slot * p.B + obj) * (256u * kBiasStageRowBytes);
          }
          mbar_wait(sm.bar(BAR_WEMPTY + stage), ph ^ 1u);
          if (CG2) {
            const uint32_t half = (uint32_t)st.n_out / 2u * kBiasStageRowBytes;
            bulk_g2s_elect(sm.stage2_u32(stage), bsrc + crank * half, half, sm.bar(BAR_WFULL + stage));
          } else {
            bulk_g2s_elect(sm.stage_u32(stage), bsrc, (uint32_t)st.n_out * kBiasStageRowBytes, sm.bar(BAR_WFULL + stage));
          }
          if (++stage == RING) { stage = 0; ph ^= 1u; }
        }
      }
    }
  }
}

// CG2, non-leader CTA: its half of every weight stage lands in ITS shared memory on ITS full barrier; this warp forwards each
// completion to the leader's full barrier (count 2: the leader's own expect_tx arrival + this one), in ring order.
__device__ __forceinline__ void relay_loop(const Params& p, const Smem& sm, int64_t n_pairs) {
  uint32_t stage = 0, ph = 0;
  const uint32_t full0_leader = mapa_u32(sm.bar(BAR_WFULL), 0u);
  for (int64_t pair0 = (int64_t)blockIdx.x - 1; pair0 < n_pairs; pair0 += gridDim.x) {
    for (int si = 0; si < p.prog.n_steps; ++si) {
      const Step& st = p.prog.s[si];
      const int n = (int)st.n_stages + (st.bias_stage ? 1 : 0);
      for (int k = 0; k < 2 * n; ++k) {   // both slots
        mbar_wait(sm.bar(BAR_WFULL + stage), ph);
        mbar_arrive_cluster_elect(full0_leader + 8u * stage);
        if (++stage == (uint32_t)kRing2) { stage = 0; ph ^= 1u; }
      }
    }
  }
}

template <bool CG2>
__device__ __forceinline__ void mma_loop(const Params& p, const Smem& sm, int64_t n_pairs, uint32_t tmem_base) {
  constexpr uint32_t RING = CG2 ? kRing2 : kRing;
  uint32_t stage = 0, ph = 0, ready_ph = 0;
  const uint64_t ones_desc = umma_desc_sw32(sm.base_u32 + SM_TAB + TAB_LAT);
  const bool trace = p.trace != nullptr && blockIdx.x == 0;
  int64_t tr = 0;
  const uint32_t crank_m = cluster_ctarank();
  const int64_t n_tiles_m = (rows_present(p) + kTileM - 1) / kTileM;
  const uint32_t lane_m = threadIdx.x & 31u;
  for (int64_t pair0 = (int64_t)blockIdx.x - crank_m; pair0 < n_pairs; pair0 += gridDim.x) {
    for (int si = 0; si < p.prog.n_steps; ++si) {
      const Step& st = p.prog.s[si];
      const uint32_t idesc = umma_idesc(CG2 ? 256 : 128, st.n_out);
      const int n_stages = st.n_stages;
#pragma unroll
      for (uint32_t slot = 0; slot < 2; ++slot, tr += 4) {
        mbar_wait(sm.bar(BAR_READY + slot), (ready_ph >> slot) & 1u);   // A operand written, accumulator drained (CG2: in both CTAs)
        ready_ph ^= 1u << slot;
        tc_fence_after();
        if (trace) p.trace[tr] = clock64();
        const uint32_t d_tmem = tmem_base + slot * 256u;
        uint64_t a_desc = umma_desc(sm.chunk_u32(slot, 0));
        uint32_t acc = (uint32_t)st.accumulate;
        bool saving = false;
        if (!CG2 && p.save != nullptr && st.save_chunks > 0) {   // training mode: keep this step's A operand for the weight-gradient kernels
          const int64_t tile = tile_index<false>(pair0, crank_m, slot);
          saving = tile < n_tiles_m;
          if (saving && lane_m == 0)
            bulk_s2g(p.save + (size_t)tile * p.prog.save_tile_bytes + st.save_off, sm.chunk_u32(slot, 0), (uint32_t)st.save_chunks * kChunkBytes);
        }
        for (int j = 0; j < n_stages; ++j) {
          mbar_wait(sm.bar(BAR_WFULL + stage), ph);
          tc_fence_after();
          if (CG2) {
            const uint64_t a_use = (st.tail_pev && j == n_stages - 1) ? umma_desc_sw64(sm.pev_u32(slot)) : a_desc;
            umma2_stage_elect(d_tmem, a_use, umma_desc_sw64(sm.stage2_u32(stage)), idesc, acc, sm.bar(BAR_WEMPTY + stage));
          } else umma_stage_elect(d_tmem, a_desc, umma_desc_sw64(sm.stage_u32(stage)), idesc, acc, sm.bar(BAR_WEMPTY + stage));
          acc = 1u;
          a_desc += (j & 1) ? (uint64_t)((kChunkBytes - 64u) >> 4) : (uint64_t)(64u >> 4);   // next 32-k half of the chunk / next chunk
          if (++stage == RING) { stage = 0; ph ^= 1u; }
        }
        if (st.bias_stage) {
          mbar_wait(sm.bar(BAR_WFULL + stage), ph);
          tc_fence_after();
          if (CG2) umma2_bias_elect(d_tmem, ones_desc, umma_desc_sw32(sm.stage2_u32(stage)), idesc, sm.bar(BAR_WEMPTY + stage));
          else umma_bias_elect(d_tmem, ones_desc, umma_desc_sw32(sm.stage_u32(stage)), idesc, sm.bar(BAR_WEMPTY + stage));
          if (++stage == RING) { stage = 0; ph ^= 1u; }
        }
        if (saving) {   // the epilogue overwrites the chunks after BAR_ACC: the bulk store must have read them by then
          if (lane_m == 0) bulk_wait_read_all();
          __syncwarp();
        }
        if (CG2) umma2_commit_elect(sm.bar(BAR_ACC + slot));
        else umma_commit_elect(sm.bar(BAR_ACC + slot));
        if (trace) p.trace[tr + 1] = clock64();
      }
    }
  }
  if (!CG2 && p.save != nullptr && lane_m == 0) bulk_wait_all();
}

template <bool CG2>
__device__ __forceinline__ void kernel_prologue(Smem& sm, uint32_t tid, uint32_t warp, uint32_t& tmem_base) {
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm.base + SM_BARS + kTmemSlotOff);
  if (tid == 0) {
    if (CG2) {
      // full: the CTA's own expect_tx arrival (+ on the leader: the peer's relayed completion); empty / acc: ONE commit of the
      // leader's MMA warp, multicast to both CTAs; ready (leader only): 8 epilogue warps of each CTA
      const uint32_t full_count = cluster_ctarank() == 0 ? 2u : 1u;
      for (int i = 0; i < kRing2; ++i) { mbar_init(sm.bar(BAR_WFULL + i), full_count); mbar_init(sm.bar(BAR_WEMPTY + i), 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(sm.bar(BAR_READY + i), 16); mbar_init(sm.bar(BAR_ACC + i), 1); }
    } else {
      for (int i = 0; i < kRing; ++i) { mbar_init(sm.bar(BAR_WFULL + i), 1); mbar_init(sm.bar(BAR_WEMPTY + i), kCluster); }
      for (int i = 0; i < 2; ++i) { mbar_init(sm.bar(BAR_READY + i), 8); mbar_init(sm.bar(BAR_ACC + i), 1); }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (CG2) {
    __syncthreads();
    cluster_sync_all();   // both CTAs of the pair are resident before the paired TMEM allocation
    if (warp == 16) tmem_alloc2(smem_u32(tmem_slot), 512);
  } else {
    if (warp == 16) tmem_alloc(smem_u32(tmem_slot), 512);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // every CTA's barriers are initialised before a peer multicasts data / arrivals into them
  tc_fence_after();
  tmem_base = *tmem_slot;
}

__device__ __forceinline__ void smem_base(Smem& sm, uint8_t* smem_raw) {
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
  sm.base = smem_raw + pad;
  sm.base_u32 = raw + pad;
}

// ------------------------------------------------------------------------------------------ forward epilogue
// 16 accumulator columns of this thread's row: (+bias, sign bits, heads) -> bf16 -> two 16-byte units of the slot's A chunk.
// Returns the 16 SIGN bits (1 = negative pre-activation), element i at bit (15 - i).
template <int EPI, bool DBG>
__device__ __forceinline__ uint32_t fwd_half(const Params& p, const Smem& sm, const Step& st, const EpiCtx& e,
                                             const uint32_t (&r)[16], int c, int h, float& sig_acc, float (&rgb_acc)[3]) {
  const float* wsig_s = sm.tab(TAB_WSIG);
  const float* w2_s = sm.tab(TAB_W2);
  const int col0 = c * 64 + (int)e.hh * 32 + h * 16;
  uint32_t pk[8], mm[2] = {0u, 0u};   // two independent 8-element funnel-shift chains
#pragma unroll
  for (int i4 = 0; i4 < 4; ++i4) {
    float v[4] = {__uint_as_float(r[4 * i4]), __uint_as_float(r[4 * i4 + 1]), __uint_as_float(r[4 * i4 + 2]),
                  __uint_as_float(r[4 * i4 + 3])};   // the bias is already in the accumulator (bias stage)
    if (EPI != F_SIGMA) {
#pragma unroll
      for (int u = 0; u < 4; ++u) mm[i4 >> 1] = __funnelshift_l(__float_as_uint(v[u]), mm[i4 >> 1], 1);
    }
    if (EPI == F_SIGMA) {
      const float4 ws = *reinterpret_cast<const float4*>(wsig_s + col0 + 4 * i4);
      sig_acc += v[0] * ws.x + v[1] * ws.y + v[2] * ws.z + v[3] * ws.w;
    }
    if (EPI == F_RGB) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float4 ww = *reinterpret_cast<const float4*>(w2_s + k * 128 + col0 + 4 * i4);
        rgb_acc[k] += fmaxf(v[0], 0.f) * ww.x + fmaxf(v[1], 0.f) * ww.y + fmaxf(v[2], 0.f) * ww.z + fmaxf(v[3], 0.f) * ww.w;
      }
    }
    if (DBG) {
      if (e.valid && st.dbg_idx >= 0) {
        float* d = p.dbg + ((size_t)st.dbg_idx * p.M + e.grow) * 256 + col0 + 4 * i4;
#pragma unroll
        for (int u = 0; u < 4; ++u) d[u] = (EPI == F_SIGMA) ? v[u] : fmaxf(v[u], 0.f);
      }
    }
    if (EPI == F_SIGMA) {
      pk[2 * i4] = pack_bf16(v[0], v[1]);
      pk[2 * i4 + 1] = pack_bf16(v[2], v[3]);
    } else {   // F_RELU; F_RGB only keeps it in training mode (rgb.2's input for the weight-gradient kernels)
      pk[2 * i4] = pack_bf16_relu(v[0], v[1]);
      pk[2 * i4 + 1] = pack_bf16_relu(v[2], v[3]);
    }
  }
  if (EPI != F_RGB || p.save != nullptr) store_row16(sm.chunk(e.slot, c), e.row, e.hh * 4u + (uint32_t)h * 2u, pk);
  return ((mm[0] & 0xffu) << 8) | (mm[1] & 0xffu);
}

// One layer's epilogue for this thread's row: TMEM -> (+bias, ReLU, mask bits) -> bf16 -> the slot's A chunks.  The
// accumulator is read in 16-column pieces into two register sets: while one set is consumed the other one's tcgen05.ld is
// in flight (tcgen05.wait::ld waits for every outstanding load, so exactly one is kept outstanding across each compute).
template <int EPI, bool DBG>
__device__ __forceinline__ void fwd_epilogue(const Params& p, const Smem& sm, const Step& st, const EpiCtx& e,
                                             uint32_t* mask_tile, bool tile_ok, float& sig_acc, float (&rgb_acc)[3]) {
  constexpr int NC = (EPI == F_RGB) ? 2 : 4;
  const uint32_t t0 = e.tmem + e.hh * 32u + e.lane_field;
  uint32_t ra[16], rb[16];
  tmem_ld16_issue(t0, ra);
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    tmem_ld_wait();
    tmem_ld16_issue(t0 + (uint32_t)c * 64u + 16u, rb);
    const uint32_t s_lo = fwd_half<EPI, DBG>(p, sm, st, e, ra, c, 0, sig_acc, rgb_acc);
    tmem_ld_wait();
    if (c + 1 < NC) tmem_ld16_issue(t0 + (uint32_t)(c + 1) * 64u, ra);
    const uint32_t s_hi = fwd_half<EPI, DBG>(p, sm, st, e, rb, c, 1, sig_acc, rgb_acc);
    if (EPI != F_SIGMA) {
      if (tile_ok) mask_tile[((size_t)st.mask_slot * 8 + c * 2 + e.hh) * 128 + e.row] = ~((s_lo << 16) | s_hi);
    }
  }
}

// PE(viewdir) (deg 4: 27 columns, zero-padded to 32) of this thread's row into the slot's PEV tile: [128 rows][32 k] bf16, K-major,
// 64-byte swizzle (rows 64 B apart, 16-byte unit u of row r at (u ^ ((r >> 1) & 3))), the layout umma_desc_sw64 describes.
// The hh == 0 thread of a row writes columns 0-15, the hh == 1 thread columns 16-31.
__device__ __forceinline__ void write_pev_row(uint8_t* pev, uint32_t row, uint32_t hh, const float d[3]) {
  float s[4][3], c[4][3];
  trig_ladder<4>(d, s, c);
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a) v[a] = d[a];
#pragma unroll
  for (int f = 0; f < 4; ++f)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      v[3 + 3 * f + a] = s[f][a];
      v[15 + 3 * f + a] = c[f][a];
    }
  uint32_t pk[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) pk[i] = hh ? pack_bf16(v[16 + 2 * i], v[17 + 2 * i]) : pack_bf16(v[2 * i], v[2 * i + 1]);
#pragma unroll
  for (uint32_t u = 0; u < 2; ++u) {
    const uint32_t unit = 2u * hh + u;
    *reinterpret_cast<uint4*>(pev + row * 64u + ((unit ^ ((row >> 1) & 3u)) << 4)) = make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
  }
}

// ------------------------------------------------------------------------------------------ forward kernel
template <bool DBG, bool CG2, bool K1 = false>
__global__ void __launch_bounds__(kThreads, 1) tc2_fwd_kernel(const __grid_constant__ Params p) {
  extern __shared__ uint8_t smem_raw[];
  Smem sm;
  smem_base(sm, smem_raw);
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  {  // static tables
    uint32_t* ones = reinterpret_cast<uint32_t*>(sm.tab(TAB_LAT));   // [128][16] bf16 1.0: the A operand of every bias stage
    for (int i = tid; i < 1024; i += kThreads) ones[i] = 0x3F803F80u;
    fence_async_smem();
    float* wsig_s = sm.tab(TAB_WSIG);
    for (int i = tid; i < 256; i += kThreads) wsig_s[i] = __ldg(p.wsig + i);
    float* w2_s = sm.tab(TAB_W2);
    for (int i = tid; i < 384; i += kThreads) w2_s[i] = __ldg(p.w2 + i);
  }
  uint32_t tmem_base;
  kernel_prologue<CG2>(sm, tid, warp, tmem_base);
  const int64_t M_eff = rows_present(p);
  const int64_t n_tiles = (M_eff + kTileM - 1) / kTileM;
  const int64_t n_pairs = (n_tiles + 1) / 2;

  if (warp == 16) {
    producer_loop<CG2>(p, sm, n_pairs);
  } else if (warp == 17) {
    if (CG2 && cluster_ctarank() != 0) relay_loop(p, sm, n_pairs);
    else mma_loop<CG2>(p, sm, n_pairs, tmem_base);
  } else {
    const uint32_t slot = warp >> 3, gw = warp & 7u, gtid = tid & 255u;
    EpiCtx e;
    e.lane = lane; e.hh = gw >> 2; e.row = (gw & 3u) * 32u + lane; e.lane_field = ((gw & 3u) * 32u) << 16;
    e.tmem = tmem_base + slot * 256u; e.slot = slot;
    // tile-end scratch outside the A chunks (so the next tile can start before it is read): the hh == 1 half of every row
    // leaves its partial sigma / rgb heads here, the hh == 0 half adds its own and stores.  [128][4] floats per slot.
    float* part = sm.tab(TAB_BIAS) + slot * 512u;
    const int nslots = p.prog.n_mask_slots;
    uint32_t acc_cnt = 0;
    const uint32_t crank = cluster_ctarank();
    const int64_t pair_first = (int64_t)blockIdx.x - crank;
    float x[3] = {0.f, 0.f, 0.f}, dir[3] = {0.f, 0.f, 1.f};
    const uint32_t ready_leader = CG2 ? mapa_u32(sm.bar(BAR_READY + slot), 0u) : 0u;
    // K1 (batched render, opt-in: SNB_BATCH_FUSED_SAMPLER): a row's coordinates come from its ray.  Two dependent stages, issued one
    // decoder step apart: (1) row -> (object, ray, sample) through tile_start / counts / order, kept as two ints; (2) rays8 + jitter
    // -> the stratified sample (renderer.py:27-41, :111-114) in the reference's op order (rb::sample_point).  A tile's 128 rows are 2
    // rays at S = 64, so the ray loads are warp-uniform.  Measured: bit-identical outputs, forward kernel +3 % (the epilogue warps are
    // the critical resource at the tile boundary), see DESIGN.md row N1.
    const float rs_fstep = K1 ? (float)(1.0 / (double)p.rs.S) : 0.f;
    auto row_lookup = [&](int64_t p0, int32_t& gi32, int32_t& kb) {
      int64_t r = tile_index<CG2>(p0, crank, slot) * kTileM + e.row;
      if (r >= M_eff) r = M_eff - 1;
      const int b = (int)obj_of_tile(p, r / kTileM);
      const rb::ObjCounts c = p.rs.counts[b];
      int64_t ray; int k;
      rb::row_source(c, p.rs.order + (int64_t)b * p.rs.N, r - c.row_start, p.rs.S, &ray, &k);
      gi32 = (int32_t)((int64_t)b * p.rs.N + ray);
      kb = k | (b << 8);
    };
    auto coords_from_ray = [&](int32_t gi32, int32_t kb, float (&xo)[3], float (&dro)[3]) {
      const int k = kb & 255, b = kb >> 8;
      const int64_t gi = gi32;
      const rb::SamplePt sp = rb::sample_point(p.rs.rays8 + 8 * gi, __ldg(p.rs.z_steps + k), __ldg(p.rs.jitter + gi * p.rs.S + k), rs_fstep,
                                               __ldg(p.rs.box + 4 * b));
#pragma unroll
      for (int a = 0; a < 3; ++a) { xo[a] = sp.x[a]; dro[a] = sp.d[a]; }
    };
    auto load_coords = [&](int64_t p0, float (&xo)[3], float (&dro)[3]) {   // clamped: tiles past the end redo row M-1, never stored
      int64_t r = tile_index<CG2>(p0, crank, slot) * kTileM + e.row;
      if (r >= M_eff) r = M_eff - 1;
      xo[0] = __ldg(p.xyz + 3 * r); xo[1] = __ldg(p.xyz + 3 * r + 1); xo[2] = __ldg(p.xyz + 3 * r + 2);
      dro[0] = __ldg(p.viewdir + 3 * r); dro[1] = __ldg(p.viewdir + 3 * r + 1); dro[2] = __ldg(p.viewdir + 3 * r + 2);
    };
    constexpr bool k1 = K1;   // compile-time: the default kernel carries none of the K1 code (it sits at the 96-register cap)
    if (pair_first < n_pairs) {   // first tile of this CTA: PE(xyz) -> chunk 0
      if constexpr (k1) { int32_t g0, kb0; row_lookup(pair_first, g0, kb0); coords_from_ray(g0, kb0, x, dir); }
      else load_coords(pair_first, x, dir);
      write_pe_row<10>(sm.chunk(slot, 0), e.row, e.hh, x);
      publish<CG2>(sm, slot, lane, ready_leader);
      if (CG2 && p.prog.pev) write_pev_row(sm.pev(slot), e.row, e.hh, dir);   // needed at encoding_viewdir only: ordered by the next publish
    }
    for (int64_t pair0 = pair_first; pair0 < n_pairs; pair0 += gridDim.x) {
      const int64_t tile = tile_index<CG2>(pair0, crank, slot);
      const bool tile_ok = tile < n_tiles;
      const bool has_next = pair0 + (int64_t)gridDim.x < n_pairs;   // cluster-uniform
      e.grow = tile * kTileM + e.row;
      e.valid = tile_ok && e.grow < M_eff;
      uint32_t* mask_tile = p.masks + (size_t)(tile_ok ? tile : 0) * nslots * 8 * 128;
      float sig_acc = 0.f, rgb_acc[3] = {0.f, 0.f, 0.f};
      float xn[3] = {0.f, 0.f, 0.f}, dn[3] = {0.f, 0.f, 1.f};
      int32_t nx_gi = 0, nx_kb = 0;
      for (int si = 0; si < p.prog.n_steps; ++si) {
        const Step& st = p.prog.s[si];
        const bool last = si + 1 == p.prog.n_steps;
        if constexpr (k1) {
          if (has_next && si + 2 == p.prog.n_steps) row_lookup(pair0 + gridDim.x, nx_gi, nx_kb);   // stage 1, one step ahead
        }
        if (last && has_next) {   // the global latency hides behind rgb.0's MMAs
          if constexpr (k1) coords_from_ray(nx_gi, nx_kb, xn, dn);
          else load_coords(pair0 + gridDim.x, xn, dn);
        }
        // (computing PE(xn) here as well was measured SLOWER: 16 more live registers spill in the rgb-head epilogue)
        mbar_wait(sm.bar(BAR_ACC + slot), acc_cnt & 1u);
        acc_cnt++;
        tc_fence_after();
        if (p.trace && blockIdx.x == 0 && gtid == 0) p.trace[(((pair0 / gridDim.x) * p.prog.n_steps + si) * 2 + slot) * 4 + 2] = clock64();
        if (st.epi == F_RELU) fwd_epilogue<F_RELU, DBG>(p, sm, st, e, mask_tile, tile_ok, sig_acc, rgb_acc);
        else if (st.epi == F_SIGMA) fwd_epilogue<F_SIGMA, DBG>(p, sm, st, e, mask_tile, tile_ok, sig_acc, rgb_acc);
        else if (st.epi == F_PEV) write_pe_row<4>(sm.chunk(slot, 0), e.row, e.hh, dir);   // accumulator untouched: the next step adds to it
        else if (st.epi == F_RGB) fwd_epilogue<F_RGB, DBG>(p, sm, st, e, mask_tile, tile_ok, sig_acc, rgb_acc);
        // F_NONE (training mode's last step): no MMAs, no epilogue -- the MMA warp only copies rgb.2's input out of the A chunks
        if (!last) publish<CG2>(sm, slot, lane, ready_leader);
        else if (has_next) {   // rgb.0's MMAs are complete and its accumulator is drained: hand the NEXT tile's PE(xyz) to the MMA warp
          write_pe_row<10>(sm.chunk(slot, 0), e.row, e.hh, xn);   // before the tile-end bookkeeping below
          publish<CG2>(sm, slot, lane, ready_leader);
          // PE(viewdir) of the next tile, OFF the boundary's critical chain: it is only read by the next tile's encoding_viewdir MMAs,
          // which the MMA warp issues after this warp's next publish (fence + arrive); this tile's MMAs are all complete
          if (CG2 && p.prog.pev) write_pev_row(sm.pev(slot), e.row, e.hh, dn);
        } else tc_fence_before();
        if (p.trace && blockIdx.x == 0 && gtid == 0) p.trace[(((pair0 / gridDim.x) * p.prog.n_steps + si) * 2 + slot) * 4 + 3] = clock64();
      }
      // tile end: combine the two column halves of the sigma / rgb heads
      if (e.hh == 1) *reinterpret_cast<float4*>(part + 4 * e.row) = make_float4(sig_acc, rgb_acc[0], rgb_acc[1], rgb_acc[2]);
      group_bar(slot);
      if (e.hh == 0 && e.valid) {
        const float4 o = *reinterpret_cast<const float4*>(part + 4 * e.row);
        const float sp = sig_acc + o.x + __ldg(p.bsig);
        p.sigma[e.grow] = sp > 20.f ? sp : log1pf(expf(sp));   // nn.Softplus(): beta 1, threshold 20
        p.rgb[3 * e.grow] = rgb_acc[0] + o.y + __ldg(p.b2);
        p.rgb[3 * e.grow + 1] = rgb_acc[1] + o.z + __ldg(p.b2 + 1);
        p.rgb[3 * e.grow + 2] = rgb_acc[2] + o.w + __ldg(p.b2 + 2);
      }
      // `part` is rewritten one tile later, after every warp of the group has passed (at least) the next tile's first publish
#pragma unroll
      for (int a = 0; a < 3; ++a) { x[a] = xn[a]; dir[a] = dn[a]; }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while a peer can still multicast into its shared memory / barriers
  if (warp == 16) { if (CG2) tmem_dealloc2(tmem_base, 512); else tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------------------------------ backward epilogue
// acc = gradient w.r.t. the layer's input; mask it by the producing layer's ReLU bits and hand it on as the next A operand.
// EV: add the sigma-head gradient first, no mask.  16-column pieces, two register sets (see fwd_epilogue).
template <bool EV, bool MASK, int H>
__device__ __forceinline__ void bwd_half(const Smem& sm, const EpiCtx& e, const uint32_t (&r)[16], int c, const uint32_t (&msh)[8], float gsp) {
  const float* wsig_s = sm.tab(TAB_WSIG);
  const int col0 = c * 64 + (int)e.hh * 32 + H * 16;
  uint32_t pk[8];
#pragma unroll
  for (int i4 = 0; i4 < 4; ++i4) {
    float v[4] = {__uint_as_float(r[4 * i4]), __uint_as_float(r[4 * i4 + 1]), __uint_as_float(r[4 * i4 + 2]), __uint_as_float(r[4 * i4 + 3])};
    if (EV) {
      const float4 ws = *reinterpret_cast<const float4*>(wsig_s + col0 + 4 * i4);
      v[0] += gsp * ws.x; v[1] += gsp * ws.y; v[2] += gsp * ws.z; v[3] += gsp * ws.w;
    }
    pk[2 * i4] = pack_bf16(v[0], v[1]);
    pk[2 * i4 + 1] = pack_bf16(v[2], v[3]);
  }
  if (MASK) {   // ReLU mask on the packed pairs: one prmt + one and per pair (tc_ptx.cuh: mask_pair)
    pk[0] &= mask_pair<H * 16 + 0>(msh); pk[1] &= mask_pair<H * 16 + 2>(msh); pk[2] &= mask_pair<H * 16 + 4>(msh);
    pk[3] &= mask_pair<H * 16 + 6>(msh); pk[4] &= mask_pair<H * 16 + 8>(msh); pk[5] &= mask_pair<H * 16 + 10>(msh);
    pk[6] &= mask_pair<H * 16 + 12>(msh); pk[7] &= mask_pair<H * 16 + 14>(msh);
  }
  store_row16(sm.chunk(e.slot, c), e.row, e.hh * 4u + (uint32_t)H * 2u, pk);
}

template <bool EV, bool MASK>
__device__ __forceinline__ void bwd_epilogue(const Smem& sm, const EpiCtx& e, const uint32_t (&mw)[4], float gsp) {
  const uint32_t t0 = e.tmem + e.hh * 32u + e.lane_field;
  uint32_t ra[16], rb[16];
  tmem_ld16_issue(t0, ra);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t msh[8];
    if (MASK) mask_shifts(mw[c], msh);
    tmem_ld_wait();
    tmem_ld16_issue(t0 + (uint32_t)c * 64u + 16u, rb);
    bwd_half<EV, MASK, 0>(sm, e, ra, c, msh, gsp);
    tmem_ld_wait();
    if (c + 1 < 4) tmem_ld16_issue(t0 + (uint32_t)(c + 1) * 64u, ra);
    bwd_half<EV, MASK, 1>(sm, e, rb, c, msh, gsp);
  }
}

// Column sums over the 128 rows of the slot's A operand (4 chunks x 64 bf16 columns, 128-byte swizzled), run by the slot's
// epilogue warps WHILE the step's MMAs execute (the warps would otherwise spin on the accumulator barrier), so the latent
// gradient reduction is off the MMA -> epilogue -> MMA critical path.  Warp gw owns the 32 columns [32 gw, 32 gw + 32): one
// conflict-free LDS.128 covers 8 rows x 4 units (quarter-warps read rows r and r + 4, whose swizzles differ in bit 2);
// fp32 accumulation, then a 3-step transposing butterfly over the 8 lanes that share a unit.  `colsum` [256] is private to the
// slot's group and each column to one lane: plain read-modify-write.  Latent gradient: sum_samples d loss / d (x + z) =
// W^T (column sums of the layer's pre-activation gradient); the W^T fold runs once per object in latent.cu.
// (A legacy mma.sync ones^T x tile version was 10x fewer instructions but its HMMAs queue behind the in-flight tcgen05 MMAs
// of BOTH slots: +3600 cycles per step, profiles/r1_trace_v9_v10.md.)
__device__ __forceinline__ void colsum_a_operand(const Smem& sm, uint32_t slot, uint32_t gw, uint32_t lane, float* colsum) {
  const uint32_t c = gw >> 1, unit = (gw & 1u) * 4u + (lane & 3u);
  const uint32_t rsub = ((lane >> 3) & 3u) + 4u * ((lane >> 2) & 1u);
  const uint8_t* base = sm.chunk(slot, (int)c);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll 4
  for (uint32_t it = 0; it < 16; ++it) {
    const uint4 q = *reinterpret_cast<const uint4*>(base + swz(it * 8u + rsub, unit));
    acc[0] += __uint_as_float(q.x << 16); acc[1] += __uint_as_float(q.x & 0xffff0000u);
    acc[2] += __uint_as_float(q.y << 16); acc[3] += __uint_as_float(q.y & 0xffff0000u);
    acc[4] += __uint_as_float(q.z << 16); acc[5] += __uint_as_float(q.z & 0xffff0000u);
    acc[6] += __uint_as_float(q.w << 16); acc[7] += __uint_as_float(q.w & 0xffff0000u);
  }
#pragma unroll
  for (int o = 4; o >= 1; o >>= 1) {   // lane bits 4, 3, 2 <-> value index bits 2, 1, 0
    const bool upper = (lane & (uint32_t)(4 * o)) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float keep = upper ? acc[i + o] : acc[i];
      const float send = upper ? acc[i] : acc[i + o];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4 * o);
    }
  }
  const uint32_t idx = ((lane >> 4) & 1u) * 4u + ((lane >> 3) & 1u) * 2u + ((lane >> 2) & 1u);
  colsum[c * 64u + unit * 8u + idx] += acc[0];
}

// ------------------------------------------------------------------------------------------ backward kernel
template <bool CG2>
__global__ void __launch_bounds__(kThreads, 1) tc2_bwd_kernel(const __grid_constant__ Params p) {
  extern __shared__ uint8_t smem_raw[];
  Smem sm;
  smem_base(sm, smem_raw);
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  {
    float* colsum0 = sm.tab(TAB_LAT);
    for (uint32_t i = tid; i < 2 * kMaxLat * 256; i += kThreads) colsum0[i] = 0.f;
    float* wsig_s = sm.tab(TAB_WSIG);
    for (int i = tid; i < 256; i += kThreads) wsig_s[i] = __ldg(p.wsig + i);
    float* w2_s = sm.tab(TAB_W2);
    for (int i = tid; i < 384; i += kThreads) w2_s[i] = __ldg(p.w2 + i);
  }
  uint32_t tmem_base;
  kernel_prologue<CG2>(sm, tid, warp, tmem_base);
  const int64_t M_eff = rows_present(p);
  const int64_t n_tiles = (M_eff + kTileM - 1) / kTileM;
  // work list: super tile q of the persistent loop is live[q] (every role of a cluster walks the same list), or q without a list
  const int64_t n_pairs = p.live ? (int64_t)__ldg(p.n_live) : (n_tiles + 1) / 2;

  if (warp == 16) {
    producer_loop<CG2>(p, sm, n_pairs);
  } else if (warp == 17) {
    if (CG2 && cluster_ctarank() != 0) relay_loop(p, sm, n_pairs);
    else mma_loop<CG2>(p, sm, n_pairs, tmem_base);
  } else {
    const uint32_t slot = warp >> 3, gw = warp & 7u, gtid = tid & 255u;
    EpiCtx e;
    e.lane = lane; e.hh = gw >> 2; e.row = (gw & 3u) * 32u + lane; e.lane_field = ((gw & 3u) * 32u) << 16;
    e.tmem = tmem_base + slot * 256u; e.slot = slot;
    const uint32_t crank = cluster_ctarank();
    // tile_index with the list: this thread's 128-row half of list entry q (pair index p0 + its slot / rank); past the list's end
    // n_tiles (never processed, never stored)
    auto work_tile = [&](int64_t p0) -> int64_t {
      if (!p.live) return tile_index<CG2>(p0, crank, slot);
      const int64_t q = p0 + (CG2 ? slot : crank);
      return q < n_pairs ? 2 * (int64_t)__ldg(p.live + q) + (CG2 ? crank : slot) : n_tiles;
    };
    float* colsum = sm.tab(TAB_LAT) + slot * kMaxLat * 256;
    // tile-end scratch outside the A chunks: the hh == 1 half of every row leaves its partial d xyz here.  [128][4] floats per slot.
    float* part = sm.tab(TAB_BIAS) + slot * 512u;
    const float* w2_s = sm.tab(TAB_W2);
    const int nslots = p.prog.n_mask_slots;
    uint32_t acc_cnt = 0;
    const int64_t pair_first = (int64_t)blockIdx.x - crank;
    // upstream gradients of one tile row: d softplus-input of sigma, d rgb, and the rgb.0 ReLU mask words of this thread's columns
    const uint32_t ready_leader = CG2 ? mapa_u32(sm.bar(BAR_READY + slot), 0u) : 0u;
    auto load_upstream = [&](int64_t t, float& gsp_o, float (&g3o)[3], uint32_t (&mwo)[2]) {
      const bool ok = t < n_tiles;
      const int64_t r = t * kTileM + e.row;
      const bool valid = ok && r < M_eff;
      const int64_t cr = valid ? r : M_eff - 1;
      const float gsg = valid ? __ldg(p.g_sigma + r) : 0.f;
      gsp_o = gsg * (-expm1f(-__ldg(p.sigma_in + cr)));   // d softplus = 1 - exp(-softplus)
#pragma unroll
      for (int k = 0; k < 3; ++k) g3o[k] = valid ? __ldg(p.g_rgb + 3 * r + k) : 0.f;
      const uint32_t* mt = p.masks + (size_t)(ok ? t : 0) * nslots * 8 * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) mwo[c] = mask_word(mt, p.r0_mask_slot, c * 2 + (int)e.hh, e.row);
    };
    // d pre-activation of rgb.0 = (g_rgb W2) * mask -> A chunks 0,1 (128 columns)
    auto prologue = [&](const float (&g3)[3], const uint32_t (&mw2)[2]) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int col0 = c * 64 + (int)e.hh * 32;
        const uint32_t mw = mw2[c];
        uint32_t pk[16];
#pragma unroll
        for (int i4 = 0; i4 < 8; ++i4) {
          const float4 w0 = *reinterpret_cast<const float4*>(w2_s + col0 + 4 * i4);
          const float4 w1 = *reinterpret_cast<const float4*>(w2_s + 128 + col0 + 4 * i4);
          const float4 w2 = *reinterpret_cast<const float4*>(w2_s + 256 + col0 + 4 * i4);
          float v[4] = {g3[0] * w0.x + g3[1] * w1.x + g3[2] * w2.x, g3[0] * w0.y + g3[1] * w1.y + g3[2] * w2.y,
                        g3[0] * w0.z + g3[1] * w1.z + g3[2] * w2.z, g3[0] * w0.w + g3[1] * w1.w + g3[2] * w2.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) if (!mask_bit(mw, 4 * i4 + u)) v[u] = 0.f;
          pk[2 * i4] = pack_bf16(v[0], v[1]);
          pk[2 * i4 + 1] = pack_bf16(v[2], v[3]);
        }
        store_row32(sm.chunk(slot, c), e.row, e.hh, pk);
      }
    };
    float gsp = 0.f;
    if (pair_first < n_pairs) {   // first tile of this CTA
      float g3[3]; uint32_t mw2[2];
      load_upstream(work_tile(pair_first), gsp, g3, mw2);
      prologue(g3, mw2);
      publish<CG2>(sm, slot, lane, ready_leader);
    }
    int64_t tile = work_tile(pair_first);
    for (int64_t pair0 = pair_first; pair0 < n_pairs; pair0 += gridDim.x) {
      const int64_t next = work_tile(pair0 + gridDim.x);   // this slot's next tile: one list lookup per tile
      const bool tile_ok = tile < n_tiles;
      const bool has_next = pair0 + (int64_t)gridDim.x < n_pairs;   // cluster-uniform
      e.grow = tile * kTileM + e.row;
      e.valid = tile_ok && e.grow < M_eff;
      const int64_t crow = e.valid ? e.grow : M_eff - 1;
      const int64_t obj = tile_ok ? obj_of_tile(p, tile) : 0;
      const uint32_t* mask_tile = p.masks + (size_t)(tile_ok ? tile : 0) * nslots * 8 * 128;
      float gsp_n = 0.f, g3n[3] = {0.f, 0.f, 0.f}, gx[3] = {0.f, 0.f, 0.f};
      uint32_t mwn[2] = {0u, 0u};
      for (int si = 0; si < p.prog.n_steps; ++si) {
        const Step& st = p.prog.s[si];
        uint32_t mw[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        if (st.epi == B_MASK && st.mask_slot >= 0) {   // fetched before the wait: the L2 latency hides behind the layer's MMAs
#pragma unroll
          for (int c = 0; c < 4; ++c) mw[c] = mask_word(mask_tile, st.mask_slot, c * 2 + (int)e.hh, e.row);
        }
        const bool last = si + 1 == p.prog.n_steps;
        if (last && has_next) load_upstream(next, gsp_n, g3n, mwn);   // global latency hides behind the last MMAs
#ifndef SNB_EXP_NO_COLSUM   // (timing experiment builds only: upper bound of what the column-sum pass costs; wrong latent gradients)
        if (st.colsum) {   // column sums of this step's A operand (published by the whole group last step), while its MMAs run
          group_bar(slot);
          colsum_a_operand(sm, slot, gw, lane, colsum + st.latent_slot * 256);
        }
#endif
        mbar_wait(sm.bar(BAR_ACC + slot), acc_cnt & 1u);
        acc_cnt++;
        tc_fence_after();
#ifndef SNB_EXP_NO_COLSUM
        if (st.colsum) group_bar(slot);   // every warp is done reading the chunks this step's epilogue overwrites
#endif
        if (p.trace && blockIdx.x == 0 && gtid == 0) p.trace[(((pair0 / gridDim.x) * p.prog.n_steps + si) * 2 + slot) * 4 + 2] = clock64();
        if (st.epi == B_XYZ) {
          // acc = d PE(xyz) (64 columns): fold to d xyz.  g_x = g_0 + sum_f 2^f (g_sin,f cos_f - g_cos,f sin_f)
          uint32_t r[32];
          tmem_ld32(e.tmem + e.hh * 32u + e.lane_field, r);
          const float x[3] = {__ldg(p.xyz + 3 * crow), __ldg(p.xyz + 3 * crow + 1), __ldg(p.xyz + 3 * crow + 2)};
          float s[10][3], c[10][3];
          trig_ladder<10>(x, s, c);
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
          for (int a = 0; a < 3; ++a) gx[a] = g[a];
        } else if (st.epi == B_VD) {
          // acc columns 0..26 = d PE(viewdir): fold to d viewdir (deg 4)
          if (e.hh == 0) {
            uint32_t r[32];
            tmem_ld32(e.tmem + e.lane_field, r);
            const float d[3] = {__ldg(p.viewdir + 3 * crow), __ldg(p.viewdir + 3 * crow + 1), __ldg(p.viewdir + 3 * crow + 2)};
            float s[4][3], c[4][3];
            trig_ladder<4>(d, s, c);
            float g[3] = {0.f, 0.f, 0.f};
#pragma unroll
            for (int i = 0; i < 27; ++i) {
              const float gv = __uint_as_float(r[i]);
              if (i < 3) g[i] += gv;
              else if (i < 15) { const int f = (i - 3) / 3, a = (i - 3) % 3; g[a] += gv * (float)(1 << f) * c[f][a]; }
              else { const int f = (i - 15) / 3, a = (i - 15) % 3; g[a] -= gv * (float)(1 << f) * s[f][a]; }
            }
            if (e.valid && p.g_viewdir) { p.g_viewdir[3 * e.grow] = g[0]; p.g_viewdir[3 * e.grow + 1] = g[1]; p.g_viewdir[3 * e.grow + 2] = g[2]; }
          }
        } else if (st.epi == B_EV) {
          bwd_epilogue<true, false>(sm, e, mw, gsp);
        } else if (st.produce_a) {
          bwd_epilogue<false, true>(sm, e, mw, gsp);
        }
        if (!last) publish<CG2>(sm, slot, lane, ready_leader);
        else if (has_next) {   // the last MMAs are complete and their accumulator is drained: hand the NEXT tile's first operand over
          prologue(g3n, mwn);  // before the tile-end bookkeeping below
          publish<CG2>(sm, slot, lane, ready_leader);
        } else tc_fence_before();
        if (p.trace && blockIdx.x == 0 && gtid == 0) p.trace[(((pair0 / gridDim.x) * p.prog.n_steps + si) * 2 + slot) * 4 + 3] = clock64();
      }
      // ---- tile end: d xyz, and flush the latent column sums when this slot's next tile belongs to another object
      const bool flush = tile_ok && (next >= n_tiles || obj_of_tile(p, next) != obj);
      if (p.g_xyz != nullptr && e.hh == 1) *reinterpret_cast<float4*>(part + 4 * e.row) = make_float4(gx[0], gx[1], gx[2], 0.f);
      group_bar(slot);
      if (p.g_xyz != nullptr && e.hh == 0 && e.valid) {
        const float4 o = *reinterpret_cast<const float4*>(part + 4 * e.row);
        p.g_xyz[3 * e.grow] = gx[0] + o.x;
        p.g_xyz[3 * e.grow + 1] = gx[1] + o.y;
        p.g_xyz[3 * e.grow + 2] = gx[2] + o.z;
      }
      gsp = gsp_n;
      if (flush) {
        for (int sl = 0; sl < p.n_latent; ++sl) {
          const float v = colsum[sl * 256 + gtid];
          if (v != 0.f) atomicAdd(p.g_zlat + ((size_t)sl * p.B + obj) * 256 + gtid, v);
          colsum[sl * 256 + gtid] = 0.f;
        }
        group_bar(slot);
      }
      tile = next;
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while a peer can still multicast into its shared memory / barriers
  if (warp == 16) { if (CG2) tmem_dealloc2(tmem_base, 512); else tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------------------------------ weight packing
struct PackJob {
  const float* src; int ld; int transposed; int n_valid; int n_pad; int k0; int k_limit; uint32_t dst_off;
  int bias;   // 1: src is a bias vector (n_valid entries); dst is a bias stage [n_pad][16 k] (see bias_stage_row)
};

constexpr int kJobsPerLaunch = 64;
struct PackJobs { int n; PackJob j[kJobsPerLaunch]; };

// one block per stage image: dst[n][k] (64B-swizzled rows of 32 bf16) = src'(n, k0 + k), zero outside the valid range
__global__ void __launch_bounds__(256) pack2_kernel(const __grid_constant__ PackJobs jobs, uint8_t* __restrict__ packed) {
  const PackJob& jb = jobs.j[blockIdx.x];
  if (jb.bias) {
    for (int n = threadIdx.x; n < jb.n_pad; n += blockDim.x)
      bias_stage_row(packed + jb.dst_off + (uint32_t)n * kBiasStageRowBytes, n < jb.n_valid ? jb.src[n] : 0.f);
    return;
  }
  for (int e = threadIdx.x; e < jb.n_pad * 32; e += blockDim.x) {
    int n, k;
    if (jb.transposed) { k = e / jb.n_pad; n = e % jb.n_pad; }  // consecutive threads walk the contiguous source dimension
    else { n = e / 32; k = e % 32; }
    const int kg = jb.k0 + k;
    float v = 0.f;
    if (n < jb.n_valid && kg < jb.k_limit) v = jb.transposed ? jb.src[(size_t)kg * jb.ld + n] : jb.src[(size_t)n * jb.ld + kg];
    const uint32_t off = jb.dst_off + (uint32_t)n * 64u + ((((uint32_t)k >> 3) ^ (((uint32_t)n >> 1) & 3u)) << 4) + ((uint32_t)k & 7u) * 2u;
    *reinterpret_cast<__nv_bfloat16*>(packed + off) = __float2bfloat16_rn(v);
  }
}

}  // namespace tc2

// ------------------------------------------------------------------------------------------ host side
using namespace tc2;

bool tc2_supported(const snb_handle_s* h) {
  const snb_arch& a = h->arch;
  return a.arch == SNB_ARCH_CODENERF && a.W == 256 && a.num_xyz_freq == 10 && a.num_dir_freq == 4 &&
         a.shape_blocks + a.texture_blocks <= kMaxLat;
}

struct Tc2Plan {
  tc2::Program fwd, fwd_train, fwd_merged, bwd_full, bwd_noxyz;
  std::vector<tc2::PackJob> jobs;
  uint32_t total_bytes = 0;
  int r0_slot = 0;
};

// src'(n, k): n < n_valid rows, k < k_limit columns of the (possibly transposed) fp32 matrix; n_stages stages of 32 k
static void add_stages(Tc2Plan& pl, const float* src, int ld, bool transposed, int n_valid, int n_pad, int k_limit, int n_stages,
                       uint32_t* first_off) {
  *first_off = pl.total_bytes;
  for (int c = 0; c < n_stages; ++c) {
    tc2::PackJob j;
    j.src = src; j.ld = ld; j.transposed = transposed ? 1 : 0; j.n_valid = n_valid; j.n_pad = n_pad; j.k0 = c * 32;
    j.k_limit = k_limit; j.dst_off = pl.total_bytes; j.bias = 0;
    pl.jobs.push_back(j);
    pl.total_bytes += (uint32_t)n_pad * 64u;
  }
}

// static bias stage of a step: must directly follow the step's weight stages in the packed image
static void add_bias_stage(Tc2Plan& pl, tc2::Step& s, const float* bias, int n_valid, int n_pad) {
  tc2::PackJob j{};
  j.src = bias; j.n_valid = n_valid; j.n_pad = n_pad; j.dst_off = pl.total_bytes; j.bias = 1;
  pl.jobs.push_back(j);
  pl.total_bytes += (uint32_t)n_pad * tc2::kBiasStageRowBytes;
  s.bias_stage = 1;
}

static tc2::Step mk(int epi, int n_out, int n_stages, int mask_slot, int latent_slot, int bias_row, int dbg_idx) {
  tc2::Step s{};
  s.epi = (int8_t)epi; s.n_out = (uint16_t)n_out; s.n_stages = (uint16_t)n_stages; s.mask_slot = (int8_t)mask_slot;
  s.latent_slot = (int8_t)latent_slot; s.bias_row = (int8_t)bias_row; s.dbg_idx = (int8_t)dbg_idx;
  s.accumulate = 0; s.produce_a = 1; s.colsum = 0; s.bias_stage = 0;
  return s;
}

static Tc2Plan build_plan2(const snb_handle_s* h) {
  Tc2Plan pl;
  const int Bs = h->arch.shape_blocks, Bt = h->arch.texture_blocks, W = 256, dv = h->d_dir(), dx = h->d_xyz();
  const auto& ly = h->layers;
  const int slot_vv = Bs + 1, slot_r = Bs + Bt + 2;
  pl.r0_slot = slot_r;
  auto push = [](tc2::Program& pr, const tc2::Step& s) { pr.s[pr.n_steps++] = s; };
  {  // ---------------- forward
    tc2::Program& f = pl.fwd;
    f.n_steps = 0; f.n_mask_slots = Bs + Bt + 3;
    tc2::Step s = mk(F_RELU, 256, 2, 0, -1, 0, 0);                                         // encoding_xyz: K = 64 (63 valid)
    add_stages(pl, ly[h->iX].w, dx, false, 256, 256, dx, 2, &s.w_off);
    add_bias_stage(pl, s, ly[h->iX].b, 256, 256);
    push(f, s);
    for (int j = 1; j <= Bs; ++j) {
      s = mk(F_RELU, 256, 8, j, j - 1, -1, j);                                             // shape_layer_j, effective bias slot j-1
      add_stages(pl, ly[h->iS(j)].w, W, false, 256, 256, W, 8, &s.w_off);
      s.bias_stage = 2;
      push(f, s);
    }
    s = mk(F_SIGMA, 256, 8, -1, -1, 1, Bs + 1);                                            // encoding_shape (+ sigma head)
    add_stages(pl, ly[h->iES].w, W, false, 256, 256, W, 8, &s.w_off);
    add_bias_stage(pl, s, ly[h->iES].b, 256, 256);
    push(f, s);
    s = mk(F_PEV, 256, 8, -1, -1, -1, -1);                                                 // encoding_viewdir, y columns
    add_stages(pl, ly[h->iEV].w, W + dv, false, 256, 256, W, 8, &s.w_off);
    push(f, s);
    s = mk(F_RELU, 256, 2, slot_vv, -1, 2, Bs + 2);                                        // + PE(viewdir) columns [W, W+dv)
    s.accumulate = 1;
    add_stages(pl, ly[h->iEV].w + W, W + dv, false, 256, 256, dv, 2, &s.w_off);
    add_bias_stage(pl, s, ly[h->iEV].b, 256, 256);
    push(f, s);
    for (int j = 1; j <= Bt; ++j) {
      s = mk(F_RELU, 256, 8, slot_vv + j, Bs + j - 1, -1, Bs + 2 + j);
      add_stages(pl, ly[h->iT(j)].w, W, false, 256, 256, W, 8, &s.w_off);
      s.bias_stage = 2;
      push(f, s);
    }
    s = mk(F_RGB, 128, 8, slot_r, -1, 3, Bs + Bt + 3);                                     // rgb.0 (+ rgb.2 head)
    s.produce_a = 0;
    add_stages(pl, ly[h->iR0].w, W, false, 128, 128, W, 8, &s.w_off);
    add_bias_stage(pl, s, ly[h->iR0].b, 128, 128);
    push(f, s);
    // save layout (training mode): every step's A operand = that layer's input, K/64 chunks, in program order
    uint32_t off = 0;
    for (int i = 0; i < f.n_steps; ++i) {
      f.s[i].save_chunks = (int8_t)((f.s[i].n_stages + 1) / 2);
      f.s[i].save_off = off;
      off += (uint32_t)f.s[i].save_chunks * kChunkBytes;
    }
    pl.fwd_train = f;
    tc2::Step sv = mk(F_NONE, 128, 0, -1, -1, -1, -1);   // rgb.2's input: ReLU(rgb.0) left in chunks 0,1 by the F_RGB epilogue
    sv.produce_a = 0; sv.w_off = 0; sv.save_chunks = 2; sv.save_off = off;
    off += 2 * kChunkBytes;
    push(pl.fwd_train, sv);
    pl.fwd_train.save_tile_bytes = off;
    f.save_tile_bytes = 0;
  }
  {  // ---------------- backward (B operand = W^T: n = input unit, k = output unit)
    for (int full = 0; full < 2; ++full) {
      tc2::Program& b = full ? pl.bwd_full : pl.bwd_noxyz;
      b.n_steps = 0; b.n_mask_slots = Bs + Bt + 3;
      tc2::Step s = mk(B_MASK, 256, 4, slot_vv + Bt, -1, -1, -1);                          // through rgb.0 -> d T_Bt, mask of T_Bt
      add_stages(pl, ly[h->iR0].w, W, true, 256, 256, 128, 4, &s.w_off);
      push(b, s);
      for (int j = Bt; j >= 1; --j) {                                                      // through texture_layer_j
        s = mk(B_MASK, 256, 8, slot_vv + j - 1, Bs + j - 1, -1, -1);
        s.colsum = 1;
        add_stages(pl, ly[h->iT(j)].w, W, true, 256, 256, W, 8, &s.w_off);
        push(b, s);
      }
      if (full) {                                                                          // d PE(viewdir) = g_ev W_dir
        s = mk(B_VD, 64, 8, -1, -1, -1, -1);
        s.produce_a = 0;
        add_stages(pl, ly[h->iEV].w + W, W + dv, true, dv, 64, W, 8, &s.w_off);
        push(b, s);
      }
      s = mk(B_EV, 256, 8, -1, -1, -1, -1);                                                // through encoding_viewdir (y columns)
      add_stages(pl, ly[h->iEV].w, W + dv, true, 256, 256, W, 8, &s.w_off);
      push(b, s);
      s = mk(B_MASK, 256, 8, Bs, -1, -1, -1);                                              // through encoding_shape, mask of H_Bs
      add_stages(pl, ly[h->iES].w, W, true, 256, 256, W, 8, &s.w_off);
      push(b, s);
      for (int j = Bs; j >= 1; --j) {                                                      // through shape_layer_j
        s = mk(B_MASK, 256, 8, j - 1, j - 1, -1, -1);
        s.colsum = 1;
        if (!full && j == 1) {   // without pose gradients only the column sums of this step's A operand are needed: no MMAs
          s.produce_a = 0; s.n_stages = 0; s.w_off = 0;
        } else {
          add_stages(pl, ly[h->iS(j)].w, W, true, 256, 256, W, 8, &s.w_off);
        }
        push(b, s);
      }
      if (full) {
        s = mk(B_XYZ, 64, 8, -1, -1, -1, -1);                                              // through encoding_xyz -> d PE(xyz)
        s.produce_a = 0;
        add_stages(pl, ly[h->iX].w, dx, true, dx, 64, W, 8, &s.w_off);
        push(b, s);
      }
      // save layout (training mode uses the full program): every step's A operand = d pre-activation of the layer it goes
      // through; the B_VD step shares encoding_viewdir's with B_EV
      uint32_t off = 0;
      for (int i = 0; i < b.n_steps; ++i) {
        b.s[i].save_chunks = b.s[i].epi == B_VD ? 0 : (int8_t)((b.s[i].n_stages + 1) / 2);
        if (!full && b.s[i].n_stages == 0) b.s[i].save_chunks = 0;
        b.s[i].save_off = off;
        off += (uint32_t)b.s[i].save_chunks * kChunkBytes;
      }
      b.save_tile_bytes = off;
    }
  }
  {  // ---------------- forward, cta_group::2 kernels: encoding_viewdir as ONE step.  The y columns (8 stages) are followed by ONE 32-k
     // stage of the PE(viewdir) columns, multiplied with the slot's PEV tile: one commit -> epilogue round trip less per tile
     // (~2 000 idle tensor-pipe cycles per tile pair, profiles/r1_trace_cg2.md).  Its stages are a second copy at the image's end.
    const tc2::Program& f = pl.fwd;
    tc2::Program& g = pl.fwd_merged;
    g = tc2::Program{};
    g.n_mask_slots = f.n_mask_slots; g.pev = 1; g.save_tile_bytes = 0;
    for (int i = 0; i < f.n_steps; ++i) {
      if (i == Bs + 3) continue;                 // the separate PE(viewdir) step
      if (i != Bs + 2) { push(g, f.s[i]); continue; }
      tc2::Step s = mk(F_RELU, 256, 9, slot_vv, -1, 2, Bs + 2);
      s.tail_pev = 1;
      uint32_t unused;
      add_stages(pl, ly[h->iEV].w, W + dv, false, 256, 256, W, 8, &s.w_off);
      add_stages(pl, ly[h->iEV].w + W, W + dv, false, 256, 256, dv, 1, &unused);   // directly behind the y stages
      add_bias_stage(pl, s, ly[h->iEV].b, 256, 256);
      push(g, s);
    }
  }
  return pl;
}

// The step programs depend on the architecture only (the pack jobs also carry the weight pointers: tc2_pack_weights rebuilds):
// built once per handle, every launch reads them from the cache.
static const Tc2Plan& cached_plan2(const snb_handle_s* h) {
  if (!h->tc2_programs) h->tc2_programs = std::make_shared<Tc2Plan>(build_plan2(h));
  return *static_cast<const Tc2Plan*>(h->tc2_programs.get());
}

size_t tc2_packed_bytes(const snb_handle_s* h) {
  if (!tc2_supported(h)) return 0;
  return cached_plan2(h).total_bytes + 1024;
}

int tc2_pack_weights(const snb_handle_s* h, void* packed, cudaStream_t st) {
  Tc2Plan pl = build_plan2(h);
  for (size_t i = 0; i < pl.jobs.size(); i += kJobsPerLaunch) {
    tc2::PackJobs jb;
    jb.n = (int)std::min<size_t>(kJobsPerLaunch, pl.jobs.size() - i);
    for (int k = 0; k < jb.n; ++k) jb.j[k] = pl.jobs[i + k];
    pack2_kernel<<<jb.n, 256, 0, st>>>(jb, (uint8_t*)packed);
    SNB_LAUNCH_CHECK();
  }
  return 0;
}


static void fill_common2(tc2::Params& p, const snb_handle_s* h, const void* packed2, const float* xyz, const float* viewdir, int64_t M,
                         int64_t B, const uint8_t* eimg, uint32_t* masks) {
  p = tc2::Params{};
  p.xyz = xyz; p.viewdir = viewdir; p.M = M; p.B = B; p.rows_per_obj = M / B;
  p.packed = (const uint8_t*)packed2; p.eimg = eimg; p.masks = masks;
  p.wsig = h->layers[h->iSG].w; p.bsig = h->layers[h->iSG].b;
  p.w2 = h->layers[h->iR2].w; p.b2 = h->layers[h->iR2].b;
  p.n_latent = h->arch.shape_blocks + h->arch.texture_blocks;
  p.trace = h->trace;
}

// Grid = a whole number of clusters, at most as many as can be co-resident (persistent kernel, 1 CTA per SM; clusters cannot
// span GPCs, so a GPC with an odd SM count leaves one SM idle), at most one CTA per tile pair (rounded up to a full cluster).
template <typename K>
static int tc2_grid(K kernel, int64_t M) {
  // co-resident CTAs per device: the same answer for every kernel variant of this file (same block size / shared memory); cached
  // per device, written at most once per (thread, device) -- host threads driving different GPUs never share an entry
  static thread_local int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); dev = 0; }
  int& max_ctas = cached[dev];
  if (max_ctas == 0) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(sm_count() / kCluster * kCluster), 1, 1);
    cfg.blockDim = dim3(tc2::kThreads, 1, 1);
    cfg.dynamicSmemBytes = SM_ALLOC;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = kCluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n <= 0) { cudaGetLastError(); n = sm_count() / kCluster; }
    max_ctas = n * kCluster;
    if (max_ctas > sm_count()) max_ctas = sm_count() / kCluster * kCluster;
  }
  const int64_t pairs = ((M + kTileM - 1) / kTileM + 1) / 2;
  const int64_t want = (pairs + kCluster - 1) / kCluster * kCluster;
  return (int)(want < max_ctas ? want : max_ctas);
}

// cta_group::2 kernels: frozen weights only (no operand saves), and every 256-row super tile inside one object (the pair's two
// tiles share the B operand, hence the per-object bias stage).  SNB_TC_CG2=0 selects the cta_group::1 kernels.
static bool tc2_use_cg2(const snb_handle_s* h, const tc2::Params& p) {
  static const int env = [] { const char* e = getenv("SNB_TC_CG2"); return e ? atoi(e) : 1; }();
  const int want = h->cg2_mode < 0 ? env : h->cg2_mode;
  return want != 0 && p.save == nullptr && p.dbg == nullptr && (p.B == 1 || p.tile_start != nullptr || p.rows_per_obj % 256 == 0);
}

// opt-in shared-memory size of every kernel variant, once per device
static int tc2_init_device() {
  static std::atomic<bool> done[64];   // setting the attribute twice is harmless: the flag only saves the calls
  int dev = 0;
  SNB_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && done[dev].load(std::memory_order_acquire)) return 0;
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2_fwd_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_ALLOC));
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2_fwd_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_ALLOC));
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2_fwd_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_ALLOC));
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2_fwd_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_ALLOC));
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_ALLOC));
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_ALLOC));
  if (dev >= 0 && dev < 64) done[dev].store(true, std::memory_order_release);
  return 0;
}

template <typename K>
static cudaError_t tc2_launch(K kernel, int grid, cudaStream_t st, const tc2::Params& p) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid, 1, 1);
  cfg.blockDim = dim3(tc2::kThreads, 1, 1);
  cfg.dynamicSmemBytes = SM_ALLOC;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = kCluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

int tc2_launch_fwd(const snb_handle_s* h, const void* packed2, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const uint8_t* eimg, uint32_t* masks, float* sigma, float* rgb, float* dbg, uint8_t* save, cudaStream_t st,
                   const int64_t* m_dev, const int32_t* tile_start, const rb::RowSrc* rs) {
  const Tc2Plan& pl = cached_plan2(h);
  tc2::Params p;
  fill_common2(p, h, packed2, xyz, viewdir, M, B, eimg, masks);
  p.sigma = sigma; p.rgb = rgb; p.dbg = dbg;
  p.save = save;
  p.m_dev = m_dev;
  p.tile_start = tile_start;
  if (rs) p.rs = *rs;
  const bool cg2 = tc2_use_cg2(h, p);
  SNB_REQUIRE(rs == nullptr || (cg2 && !dbg && !save), "tc2 forward: the fused sampler runs on the cta_group::2 kernels (frozen weights)");
  p.prog = save ? pl.fwd_train : ((cg2 && !dbg) ? pl.fwd_merged : pl.fwd);
  if (tc2_init_device()) return 1;
  if (dbg) {
    SNB_CHECK_CUDA(tc2_launch(tc2_fwd_kernel<true, false>, tc2_grid(tc2_fwd_kernel<true, false>, M), st, p));
  } else if (cg2 && p.rs.rays8 != nullptr) {
    SNB_CHECK_CUDA(tc2_launch(tc2_fwd_kernel<false, true, true>, tc2_grid(tc2_fwd_kernel<false, true, true>, M), st, p));
  } else if (cg2) {
    SNB_CHECK_CUDA(tc2_launch(tc2_fwd_kernel<false, true>, tc2_grid(tc2_fwd_kernel<false, true>, M), st, p));
  } else {
    SNB_CHECK_CUDA(tc2_launch(tc2_fwd_kernel<false, false>, tc2_grid(tc2_fwd_kernel<false, false>, M), st, p));
  }
  return 0;
}

int tc2_launch_bwd(const snb_handle_s* h, const void* packed2, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                   const uint32_t* masks, const float* sigma, const float* g_sigma, const float* g_rgb, float* g_xyz,
                   float* g_viewdir, float* g_zlat, uint8_t* save, cudaStream_t st, const int64_t* m_dev, const int32_t* tile_start,
                   const int32_t* live, const int32_t* n_live) {
  const Tc2Plan& pl = cached_plan2(h);
  tc2::Params p;
  fill_common2(p, h, packed2, xyz, viewdir, M, B, nullptr, const_cast<uint32_t*>(masks));
  p.sigma_in = sigma; p.g_sigma = g_sigma; p.g_rgb = g_rgb; p.g_xyz = g_xyz; p.g_viewdir = g_viewdir; p.g_zlat = g_zlat;
  p.r0_mask_slot = pl.r0_slot;
  p.save = save;
  p.m_dev = m_dev;
  p.tile_start = tile_start;
  p.live = live; p.n_live = n_live;
  SNB_REQUIRE(save == nullptr || g_xyz != nullptr, "tc2 backward: training mode runs the full program (g_xyz scratch required)");
  p.prog = g_xyz ? pl.bwd_full : pl.bwd_noxyz;
  if (tc2_init_device()) return 1;
  if (tc2_use_cg2(h, p)) {
    SNB_CHECK_CUDA(tc2_launch(tc2_bwd_kernel<true>, tc2_grid(tc2_bwd_kernel<true>, M), st, p));
  } else {
    SNB_CHECK_CUDA(tc2_launch(tc2_bwd_kernel<false>, tc2_grid(tc2_bwd_kernel<false>, M), st, p));
  }
  return 0;
}

// =====================================================================================================================
// Weight gradients (training mode, SNB_PREC_BF16_TRAIN): dW_l = sum_samples dY_l^T X_l on the tensor core.
// The forward / backward kernels above left every layer's input X_l and pre-activation gradient dY_l in HBM as the very
// shared-memory operand images they used (128-sample tiles, 16 KB chunks of [128 samples][64 features] bf16, 128-byte
// swizzle).  Read with samples as the K dimension those bytes are exactly tcgen05's canonical MN-MAJOR 128B-swizzled layout
// (64 contiguous features per 128-byte row, 8-sample atoms of 1024 B), so no transposition is needed: per 16 samples one
// MMA  D[128 out][N in] += dY^T[128 out][16] . X^T[N in][16]  with both operands MN-major.  D (two 128-row halves x 256
// columns fp32) fills TMEM; one CTA owns (layer, tile range), accumulates over its tiles and adds its partial dW to global
// memory with atomics.  HBM-bound: 2 x (dy_chunks + x_chunks) x 8 KB per 64 samples.  Bias gradients = column sums of dY,
// taken by the epilogue warps from the same shared-memory pieces while the MMAs run.
// =====================================================================================================================
namespace tc2 {

constexpr int kWThreads = 192;            // warp 0 producer, warp 1 MMA issuer (+ TMEM alloc), warps 2..5 colsum + epilogue
constexpr int kWStages = 3;
constexpr uint32_t kWPiece = 8192;        // half a chunk: [64 samples][64 features]
constexpr uint32_t kWStageBytes = 8 * kWPiece;
constexpr uint32_t SMW_BARS = kWStages * kWStageBytes;
constexpr uint32_t SMW_ALLOC = SMW_BARS + 256 + 1024;
constexpr int kMaxWJobs = 16;

struct WJob {
  uint32_t dy_off, x_off;        // byte offsets inside the backward / forward tile save blocks
  int32_t dy_chunks, x_chunks;   // 64-feature chunks of dY (2 or 4) and of X (1 or 4)
  int32_t n_out, n_in;           // valid rows / columns of dW
  float* gw; int32_t ld, col0;   // dW (out, ld) row-major, this job's columns start at col0
  float* gb;                     // bias gradient (n_out) or NULL
};
struct WParams {
  const uint8_t* fsave; const uint8_t* bsave;
  uint32_t f_tile_bytes, b_tile_bytes;
  int64_t n_tiles;
  const int64_t* m_dev;   // optional device-side row count (see Params::m_dev)
  int32_t n_jobs, splits;
  WJob jobs[kMaxWJobs];
};

// MN-major, 128-byte-swizzled operand: 64 features per 128-byte row, consecutive samples 128 B apart, 8-sample atoms 1024 B
// apart (SBO), next 64-feature group one piece further (LBO).
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(kWPiece >> 4) << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__global__ void __launch_bounds__(kWThreads, 1) tc2_wgrad_kernel(const __grid_constant__ WParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
  uint8_t* base = smem_raw + pad;
  const uint32_t base_u32 = raw + pad;
  auto bar = [&](int i) { return base_u32 + SMW_BARS + 8u * (uint32_t)i; };   // full[0..2], empty[3..5], done[6]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base + SMW_BARS + 128);
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const WJob& jb = p.jobs[blockIdx.x / p.splits];
  const int split = blockIdx.x % p.splits;
  if (tid == 0) {
    for (int i = 0; i < kWStages; ++i) { mbar_init(bar(i), 1); mbar_init(bar(kWStages + i), 1 + 4); }
    mbar_init(bar(2 * kWStages), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_pieces = jb.dy_chunks + jb.x_chunks;
  const int64_t n_tiles = p.m_dev ? (__ldg(p.m_dev) + kTileM - 1) / kTileM : p.n_tiles;
  const int64_t my_tiles = n_tiles > split ? (n_tiles - split + p.splits - 1) / p.splits : 0;
  const int64_t n_iters = my_tiles * 2;   // half tiles

  if (warp == 0) {
    // ---------------------------------------------------------------- producer: one 64-sample half tile per stage
    uint32_t stage = 0, ph = 0;
    for (int64_t it = 0; it < n_iters; ++it) {
      const int64_t tile = split + (it >> 1) * p.splits;
      const uint32_t ht = (uint32_t)(it & 1);
      mbar_wait(bar(kWStages + stage), ph ^ 1u);
      if (lane == 0) {
        mbar_expect_tx(bar(stage), (uint32_t)n_pieces * kWPiece);
        const uint8_t* dy = p.bsave + (size_t)tile * p.b_tile_bytes + jb.dy_off + ht * kWPiece;
        const uint8_t* xx = p.fsave + (size_t)tile * p.f_tile_bytes + jb.x_off + ht * kWPiece;
        const uint32_t dst = base_u32 + stage * kWStageBytes;
        for (int c = 0; c < jb.dy_chunks; ++c) bulk_g2s(dst + (uint32_t)c * kWPiece, dy + (size_t)c * kChunkBytes, kWPiece, bar(stage));
        for (int c = 0; c < jb.x_chunks; ++c)
          bulk_g2s(dst + (uint32_t)(jb.dy_chunks + c) * kWPiece, xx + (size_t)c * kChunkBytes, kWPiece, bar(stage));
      }
      __syncwarp();
      if (++stage == (uint32_t)kWStages) { stage = 0; ph ^= 1u; }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t n_cols = (uint32_t)jb.x_chunks * 64u;
    const uint32_t idesc = umma_idesc(128, n_cols) | (1u << 15) | (1u << 16);   // A and B MN-major
    const int n_halves = jb.dy_chunks / 2;
    uint32_t stage = 0, ph = 0;
    for (int64_t it = 0; it < n_iters; ++it) {
      mbar_wait(bar(stage), ph);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t sb = base_u32 + stage * kWStageBytes;
        for (int ks = 0; ks < 4; ++ks) {          // 16 samples per MMA: two 8-sample atoms
          const uint64_t b_desc = umma_desc_mn(sb + (uint32_t)jb.dy_chunks * kWPiece + (uint32_t)ks * 2048u);
          for (int hf = 0; hf < n_halves; ++hf) {
            const uint64_t a_desc = umma_desc_mn(sb + (uint32_t)(2 * hf) * kWPiece + (uint32_t)ks * 2048u);
            umma_bf16(tmem_base + (uint32_t)hf * 256u, a_desc, b_desc, idesc, (it > 0 || ks > 0) ? 1u : 0u);
          }
        }
        umma_commit(bar(kWStages + stage));
      }
      __syncwarp();
      if (++stage == (uint32_t)kWStages) { stage = 0; ph ^= 1u; }
    }
    if (lane == 0) umma_commit(bar(2 * kWStages));
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- bias column sums during the loop, then the epilogue
    const uint32_t w4 = warp - 2;                 // 0..3: dY piece this warp sums
    float acc[2][8];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[a][i] = 0.f;
    const uint32_t rsub = ((lane >> 3) & 3u) + 4u * ((lane >> 2) & 1u);
    const bool do_sum = jb.gb != nullptr && (int)w4 < jb.dy_chunks;
    uint32_t stage = 0, ph = 0;
    for (int64_t it = 0; it < n_iters; ++it) {
      mbar_wait(bar(stage), ph);
      if (do_sum) {
        const uint8_t* piece = base + stage * kWStageBytes + w4 * kWPiece;
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          const uint32_t unit = (uint32_t)a * 4u + (lane & 3u);
#pragma unroll 4
          for (uint32_t g = 0; g < 8; ++g) {
            const uint4 q = *reinterpret_cast<const uint4*>(piece + swz(g * 8u + rsub, unit));
            acc[a][0] += __uint_as_float(q.x << 16); acc[a][1] += __uint_as_float(q.x & 0xffff0000u);
            acc[a][2] += __uint_as_float(q.y << 16); acc[a][3] += __uint_as_float(q.y & 0xffff0000u);
            acc[a][4] += __uint_as_float(q.z << 16); acc[a][5] += __uint_as_float(q.z & 0xffff0000u);
            acc[a][6] += __uint_as_float(q.w << 16); acc[a][7] += __uint_as_float(q.w & 0xffff0000u);
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(kWStages + stage));
      if (++stage == (uint32_t)kWStages) { stage = 0; ph ^= 1u; }
    }
    if (do_sum) {
#pragma unroll
      for (int a = 0; a < 2; ++a) {
#pragma unroll
        for (int o = 4; o >= 1; o >>= 1) {
          const bool upper = (lane & (uint32_t)(4 * o)) != 0;
#pragma unroll
          for (int i = 0; i < o; ++i) {
            const float keep = upper ? acc[a][i + o] : acc[a][i];
            const float send = upper ? acc[a][i] : acc[a][i + o];
            acc[a][i] = keep + __shfl_xor_sync(0xffffffffu, send, 4 * o);
          }
        }
        const uint32_t idx = ((lane >> 4) & 1u) * 4u + ((lane >> 3) & 1u) * 2u + ((lane >> 2) & 1u);
        const int col = (int)(w4 * 64u + ((uint32_t)a * 4u + (lane & 3u)) * 8u + idx);
        if (col < jb.n_out && n_iters > 0) atomicAdd(jb.gb + col, acc[a][0]);
      }
    }
    // epilogue: this warp owns TMEM lanes 32 (warp % 4) ..: rows of dW
    mbar_wait(bar(2 * kWStages), 0u);
    tc_fence_after();
    if (n_iters > 0) {
      const uint32_t q4 = warp & 3u;
      const int n_halves = jb.dy_chunks / 2, n_cols = jb.x_chunks * 64;
      for (int hf = 0; hf < n_halves; ++hf) {
        const int row = hf * 128 + (int)(q4 * 32u + lane);
        for (int c0 = 0; c0 < n_cols; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(tmem_base + (uint32_t)hf * 256u + (uint32_t)c0 + ((q4 * 32u) << 16), r);
          if (row < jb.n_out) {
            float* dst = jb.gw + (size_t)row * jb.ld + jb.col0 + c0;
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c0 + i < jb.n_in) atomicAdd(dst + i, __uint_as_float(r[i]));
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// dW_layer[o][i] += sum_obj s[slot][obj][o] * z[slot][obj][i]: the per-object latent vector z is part of the consuming
// layer's input (x + z), but the tensor-core path only saw x (z was folded into the bias).  grid (slots, W), block W.
struct OuterJobs { int n; float* gw[kMaxLat]; };
__global__ void __launch_bounds__(256) wgrad_latent_outer_kernel(const __grid_constant__ OuterJobs J, int64_t B, int W,
                                                                const float* __restrict__ s, const float* __restrict__ z) {
  const int slot = blockIdx.x, o = blockIdx.y, i = threadIdx.x;
  if (i >= W) return;
  float acc = 0.f;
  for (int64_t b = 0; b < B; ++b) acc = fmaf(s[((size_t)slot * B + b) * W + o], z[((size_t)slot * B + b) * W + i], acc);
  J.gw[slot][(size_t)o * W + i] += acc;
}

// sigma head and rgb.2 on CUDA cores from the saved operand images: y = encoding_shape output (4 chunks), h = ReLU(rgb.0) (2 chunks)
//   d w_sigma[i] = sum_s gsp[s] y[s][i],  d b_sigma = sum_s gsp[s];  d W2[k][j] = sum_s g_rgb[s][k] h[s][j],  d b2[k] = sum_s g_rgb[s][k]
// Thread t owns one 16-byte unit (8 columns) u = t % 32 and the 16 rows of row group t / 32 of every tile: a warp reads one whole
// 512-byte sample row per step (16-byte loads, independent across the 16 rows), partial sums stay in registers across tiles.
__global__ void __launch_bounds__(256) wgrad_heads_kernel(const uint8_t* __restrict__ fsave, uint32_t f_tile_bytes, uint32_t y_off,
                                                         uint32_t h_off, int64_t n_tiles, int64_t M, const int64_t* __restrict__ m_dev,
                                                         const float* __restrict__ sigma,
                                                         const float* __restrict__ g_sigma, const float* __restrict__ g_rgb,
                                                         float* __restrict__ gw_sig, float* __restrict__ gb_sig,
                                                         float* __restrict__ gw2, float* __restrict__ gb2) {
  __shared__ float gs[128], g3[3][128];
  if (m_dev) { M = __ldg(m_dev); n_tiles = (M + kTileM - 1) / kTileM; }
  __shared__ float red[8][4][256];   // [row group][sigma | rgb k][column]
  const uint32_t t = threadIdx.x, u = t & 31u, rg = t >> 5;
  const uint32_t chunk = u >> 3, unit = u & 7u;
  float a_sig[8], a2[3][8], a_b = 0.f, a_b2[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 8; ++i) { a_sig[i] = 0.f; a2[0][i] = 0.f; a2[1][i] = 0.f; a2[2][i] = 0.f; }
  auto fma8 = [](float (&acc)[8], float w, const uint4& q) {
    acc[0] = fmaf(w, __uint_as_float(q.x << 16), acc[0]); acc[1] = fmaf(w, __uint_as_float(q.x & 0xffff0000u), acc[1]);
    acc[2] = fmaf(w, __uint_as_float(q.y << 16), acc[2]); acc[3] = fmaf(w, __uint_as_float(q.y & 0xffff0000u), acc[3]);
    acc[4] = fmaf(w, __uint_as_float(q.z << 16), acc[4]); acc[5] = fmaf(w, __uint_as_float(q.z & 0xffff0000u), acc[5]);
    acc[6] = fmaf(w, __uint_as_float(q.w << 16), acc[6]); acc[7] = fmaf(w, __uint_as_float(q.w & 0xffff0000u), acc[7]);
  };
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    __syncthreads();
    if (t < 128) {
      const int64_t r = tile * 128 + t;
      const bool ok = r < M;
      gs[t] = ok ? __ldg(g_sigma + r) * (-expm1f(-__ldg(sigma + r))) : 0.f;
      g3[0][t] = ok ? __ldg(g_rgb + 3 * r) : 0.f; g3[1][t] = ok ? __ldg(g_rgb + 3 * r + 1) : 0.f; g3[2][t] = ok ? __ldg(g_rgb + 3 * r + 2) : 0.f;
    }
    __syncthreads();
    const uint8_t* ty = fsave + (size_t)tile * f_tile_bytes + y_off + (size_t)chunk * kChunkBytes;
    const uint8_t* th = fsave + (size_t)tile * f_tile_bytes + h_off + (size_t)chunk * kChunkBytes;
#pragma unroll 4
    for (uint32_t k = 0; k < 16; ++k) {
      const uint32_t srow = rg * 16u + k;
      const uint4 qy = __ldg(reinterpret_cast<const uint4*>(ty + swz(srow, unit)));
      fma8(a_sig, gs[srow], qy);
      if (chunk < 2) {
        const uint4 qh = __ldg(reinterpret_cast<const uint4*>(th + swz(srow, unit)));
        fma8(a2[0], g3[0][srow], qh); fma8(a2[1], g3[1][srow], qh); fma8(a2[2], g3[2][srow], qh);
      }
      if (u == 0) { a_b += gs[srow]; a_b2[0] += g3[0][srow]; a_b2[1] += g3[1][srow]; a_b2[2] += g3[2][srow]; }
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint32_t col = chunk * 64u + unit * 8u + (uint32_t)i;
    red[rg][0][col] = a_sig[i];
    if (chunk < 2) { red[rg][1][col] = a2[0][i]; red[rg][2][col] = a2[1][i]; red[rg][3][col] = a2[2][i]; }
  }
  __syncthreads();
  {
    float v = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) v += red[g][0][t];
    atomicAdd(gw_sig + t, v);
    if (t < 128) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        float w = 0.f;
#pragma unroll
        for (int g = 0; g < 8; ++g) w += red[g][1 + k][t];
        atomicAdd(gw2 + k * 128 + t, w);
      }
    }
  }
  if (u == 0) {   // one lane per row group
    atomicAdd(gb_sig, a_b);
    atomicAdd(gb2, a_b2[0]); atomicAdd(gb2 + 1, a_b2[1]); atomicAdd(gb2 + 2, a_b2[2]);
  }
}

// latent layers (per object): d pre = dz * [z > 0];  d W_lat[o][k] += sum_b dpre[b][o] latent[b][k];  d b_lat[o] += sum_b dpre[b][o].
// grid (slots, W), block D.  (The fp32 back end's generic sgemm takes ~70 us per layer for these 8-row GEMMs.)
struct LatWJobs { int n, n_shape; float* gw[kMaxLat]; float* gb[kMaxLat]; };
__global__ void __launch_bounds__(1024) wgrad_latent_layers_kernel(const __grid_constant__ LatWJobs J, int64_t B, int W, int D,
                                                                  const float* __restrict__ zlat, const float* __restrict__ dz,
                                                                  const float* __restrict__ shape_latent,
                                                                  const float* __restrict__ texture_latent) {
  const int slot = blockIdx.x, o = blockIdx.y, k = threadIdx.x;
  if (k >= D) return;
  const float* lat = slot < J.n_shape ? shape_latent : texture_latent;
  float acc = 0.f, accb = 0.f;
  for (int64_t b = 0; b < B; ++b) {
    const size_t zi = ((size_t)slot * B + b) * W + o;
    const float dp = zlat[zi] > 0.f ? dz[zi] : 0.f;
    acc = fmaf(dp, lat[b * D + k], acc);
    accb += dp;
  }
  J.gw[slot][(size_t)o * D + k] += acc;
  if (k == 0) J.gb[slot][o] += accb;
}

}  // namespace tc2

size_t tc2_fwd_save_bytes(const snb_handle_s* h, int64_t M) {
  return (size_t)((M + kTileM - 1) / kTileM) * cached_plan2(h).fwd_train.save_tile_bytes;
}
size_t tc2_bwd_save_bytes(const snb_handle_s* h, int64_t M) {
  return (size_t)((M + kTileM - 1) / kTileM) * cached_plan2(h).bwd_full.save_tile_bytes;
}

// All weight / bias gradients of the decoder layers that run on the tensor core, the two heads, and the z (x) s outer products
// of the latent-consuming layers.  g_weights: canonical order (2 per layer), already zeroed.  s_lat: the per-object column sums
// [(Bs+Bt)][B][256] the backward kernel produced; zlat: the forward's per-object latent activations.
int tc2_launch_wgrad(const snb_handle_s* h, int64_t M, int64_t B, const uint8_t* fsave, const uint8_t* bsave, const float* sigma,
                     const float* g_sigma, const float* g_rgb, const float* s_lat, const float* zlat, float* const* gw,
                     cudaStream_t st, const int64_t* m_dev) {
  const Tc2Plan& pl = cached_plan2(h);
  const tc2::Program& F = pl.fwd_train;
  const tc2::Program& Bp = pl.bwd_full;
  const int Bs = h->arch.shape_blocks, Bt = h->arch.texture_blocks, W = 256, dv = h->d_dir(), dx = h->d_xyz();
  // forward step indices: 0 X | 1..Bs S_j | Bs+1 ES | Bs+2 EVy | Bs+3 EVdir | Bs+4.. T_j | Bs+Bt+4 R0 | Bs+Bt+5 rgb.2 input
  // backward (full) step indices: 0 R0 | 1..Bt T_j (j = Bt..1) | Bt+1 VD | Bt+2 EV | Bt+3 ES | Bt+4.. S_j (j = Bs..1) | Bs+Bt+4 XYZ
  auto fX = [&](int step) { return F.s[step].save_off; };
  auto bY = [&](int step) { return Bp.s[step].save_off; };
  tc2::WParams p{};
  p.fsave = fsave; p.bsave = bsave; p.f_tile_bytes = F.save_tile_bytes; p.b_tile_bytes = Bp.save_tile_bytes;
  p.n_tiles = (M + kTileM - 1) / kTileM;
  p.m_dev = m_dev;
  int nj = 0;
  auto add = [&](int layer, int col0, int ld, uint32_t dy_off, int dy_chunks, int n_out, uint32_t x_off, int x_chunks, int n_in, bool bias) {
    tc2::WJob& j = p.jobs[nj++];
    j.dy_off = dy_off; j.dy_chunks = dy_chunks; j.n_out = n_out; j.x_off = x_off; j.x_chunks = x_chunks; j.n_in = n_in;
    j.gw = gw[2 * layer]; j.ld = ld; j.col0 = col0; j.gb = bias ? gw[2 * layer + 1] : nullptr;
  };
  add(h->iX, 0, dx, bY(Bs + Bt + 4), 4, W, fX(0), 1, dx, true);
  for (int j = 1; j <= Bs; ++j) add(h->iS(j), 0, W, bY(Bt + 4 + (Bs - j)), 4, W, fX(j), 4, W, true);
  add(h->iES, 0, W, bY(Bt + 3), 4, W, fX(Bs + 1), 4, W, true);
  add(h->iEV, 0, W + dv, bY(Bt + 2), 4, W, fX(Bs + 2), 4, W, true);
  add(h->iEV, W, W + dv, bY(Bt + 2), 4, W, fX(Bs + 3), 1, dv, false);
  for (int j = 1; j <= Bt; ++j) add(h->iT(j), 0, W, bY(1 + (Bt - j)), 4, W, fX(Bs + 3 + j), 4, W, true);
  add(h->iR0, 0, W, bY(0), 2, W / 2, fX(Bs + Bt + 4), 4, W, true);
  SNB_REQUIRE(nj <= tc2::kMaxWJobs, "wgrad: too many jobs");
  p.n_jobs = nj;
  const int sms = sm_count();
  int splits = sms / nj;
  if (splits < 1) splits = 1;
  if ((int64_t)splits > p.n_tiles) splits = (int)p.n_tiles;
  p.splits = splits;
  SNB_CHECK_CUDA(cudaFuncSetAttribute(tc2::tc2_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc2::SMW_ALLOC));
  tc2::tc2_wgrad_kernel<<<nj * splits, tc2::kWThreads, tc2::SMW_ALLOC, st>>>(p);
  SNB_LAUNCH_CHECK();
  // z (x) s outer products of the latent-consuming layers
  tc2::OuterJobs oj{};
  oj.n = Bs + Bt;
  for (int j = 1; j <= Bs + Bt; ++j) oj.gw[j - 1] = gw[2 * (j <= Bs ? h->iS(j) : h->iT(j - Bs))];
  tc2::wgrad_latent_outer_kernel<<<dim3((unsigned)(Bs + Bt), (unsigned)W), 256, 0, st>>>(oj, B, W, s_lat, zlat);
  SNB_LAUNCH_CHECK();
  // heads
  const int64_t nt = p.n_tiles;
  const int grid = (int)(nt < 4 * sms ? nt : 4 * sms);
  tc2::wgrad_heads_kernel<<<grid, 256, 0, st>>>(fsave, F.save_tile_bytes, fX(Bs + 2), fX(Bs + Bt + 5), nt, M, m_dev, sigma, g_sigma, g_rgb,
                                               gw[2 * h->iSG], gw[2 * h->iSG + 1], gw[2 * h->iR2], gw[2 * h->iR2 + 1]);
  SNB_LAUNCH_CHECK();
  return 0;
}

// weight / bias gradients of the per-object latent layers from dz = d loss / d z (the folded column sums)
int tc2_launch_latent_wgrad(const snb_handle_s* h, int64_t B, const float* zlat, const float* dz, const float* shape_latent,
                            const float* texture_latent, float* const* gw, cudaStream_t st) {
  const int Bs = h->arch.shape_blocks, Bt = h->arch.texture_blocks, W = h->arch.W, D = h->arch.latent_dim;
  SNB_REQUIRE(D <= 1024, "latent wgrad: latent_dim > 1024");
  tc2::LatWJobs J{};
  J.n = Bs + Bt; J.n_shape = Bs;
  for (int j = 1; j <= Bs + Bt; ++j) {
    const int li = j <= Bs ? h->iSL(j) : h->iTL(j - Bs);
    J.gw[j - 1] = gw[2 * li]; J.gb[j - 1] = gw[2 * li + 1];
  }
  tc2::wgrad_latent_layers_kernel<<<dim3((unsigned)(Bs + Bt), (unsigned)W), (unsigned)((D + 31) / 32 * 32), 0, st>>>(
      J, B, W, D, zlat, dz, shape_latent, texture_latent);
  SNB_LAUNCH_CHECK();
  return 0;
}

}  // namespace snb
