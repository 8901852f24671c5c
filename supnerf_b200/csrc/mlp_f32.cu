// K2 / K2b, SNB_PREC_FP32 back end: the latent-conditioned decoder MLP in true fp32 (FFMA), layer by
// layer, with the positional encoding, ReLU masks, latent column sums and weight gradients as small
// fused kernels around one strided SGEMM.  This is the 1e-5 parity mode; the throughput mode is the
// tcgen05 kernel in mlp_tc.cu.  Restructurings (exact, SURVEY §8(a')3): the latent layers are
// evaluated once per object and enter as a per-object row offset of the next GEMM's A operand; the
// `cat([y, PE(viewdir)])` layer is two GEMMs accumulating into one output.
#include "common.cuh"
#include "decoder.h"
#include "sgemm.cuh"
#include <math.h>

namespace snb {

// ---- positional encoding (model_codenerf.py:4-10) -------------------------------------------------
__global__ void pe_fwd_kernel(const float* __restrict__ x, int64_t M, int deg, float* __restrict__ out, int ld) {
  const int64_t n = M * 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / 3;
    const int a = (int)(i - m * 3);
    const float v = x[i];
    float* o = out + m * ld;
    o[a] = v;
    float sc = 1.f;
    for (int f = 0; f < deg; ++f) {
      const float y = sc * v;  // exact: power of two
      o[3 + 3 * f + a] = sinf(y);
      o[3 + 3 * deg + 3 * f + a] = cosf(y);
      sc *= 2.f;
    }
  }
}

// g_x = g_0 + sum_f 2^f (g_sin,f cos(2^f x) - g_cos,f sin(2^f x))
__global__ void pe_bwd_kernel(const float* __restrict__ g_pe, int ld, const float* __restrict__ x, int64_t M, int deg,
                              float* __restrict__ g_x) {
  const int64_t n = M * 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / 3;
    const int a = (int)(i - m * 3);
    const float v = x[i];
    const float* gp = g_pe + m * ld;
    float acc = gp[a], sc = 1.f;
    for (int f = 0; f < deg; ++f) {
      const float y = sc * v;
      acc += sc * (gp[3 + 3 * f + a] * cosf(y) - gp[3 + 3 * deg + 3 * f + a] * sinf(y));
      sc *= 2.f;
    }
    g_x[i] = acc;
  }
}

// nn.Softplus() defaults: beta 1, threshold 20 (model_codenerf.py:30)
__global__ void softplus_kernel(float* __restrict__ x, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    x[i] = v > 20.f ? v : log1pf(expf(v));
  }
}

// d softplus / d pre = sigmoid(pre) = 1 - exp(-softplus(pre)); above the threshold it is 1 (1 - e^-20 rounds to 1).
__global__ void softplus_bwd_kernel(const float* __restrict__ sigma, const float* __restrict__ g_sigma,
                                    float* __restrict__ g_pre, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    g_pre[i] = g_sigma[i] * (-expm1f(-sigma[i]));
}

// In place: optionally accumulate the per-object column sums of g (BEFORE masking), then g *= (h > 0).
// grid.x = objects * chunks_per_obj, block = 256 threads, each thread owns columns c, c+256, ...
__global__ void __launch_bounds__(256) mask_colsum_kernel(float* __restrict__ g, const float* __restrict__ h, int ld,
                                                         int width, int64_t rows_per_obj, int chunks_per_obj,
                                                         int rows_per_chunk, float* __restrict__ colsum) {
  const int64_t obj = blockIdx.x / chunks_per_obj;
  const int chunk = blockIdx.x % chunks_per_obj;
  const int64_t r0 = obj * rows_per_obj + (int64_t)chunk * rows_per_chunk;
  int64_t r1 = r0 + rows_per_chunk;
  const int64_t rend = (obj + 1) * rows_per_obj;
  if (r1 > rend) r1 = rend;
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    double s = 0.0;  // these sums cancel heavily (latent / bias gradients): keep the per-chunk partial exact
    for (int64_t r = r0; r < r1; ++r) {
      const float v = g[r * ld + c];
      s += (double)v;
      if (h != nullptr && !(h[r * ld + c] > 0.f)) g[r * ld + c] = 0.f;
    }
    if (colsum != nullptr) atomicAdd(colsum + obj * width + c, (float)s);
  }
}

// bias gradient: out[c] += sum_rows g[r][c]
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ g, int ld, int width, int64_t rows,
                                                    int rows_per_block, float* __restrict__ out) {
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    double s = 0.0;
    for (int64_t r = r0; r < r1; ++r) s += (double)g[r * ld + c];
    atomicAdd(out + c, (float)s);
  }
}

__global__ void fill_kernel(float* __restrict__ p, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

static inline int ew_grid(int64_t n) {
  int64_t b = ceil_div(n, 256);
  int64_t cap = (int64_t)sm_count() * 8;
  if (b > cap) b = cap;
  return (int)(b > 0 ? b : 1);
}

struct Bump {
  float* base;
  int64_t used = 0;
  float* take(int64_t n) {
    float* r = base ? base + used : nullptr;
    used += (n + 3) & ~int64_t(3);
    return r;
  }
};

static inline int64_t al4(int64_t n) { return (n + 3) & ~int64_t(3); }

// ---- workspace layout (CodeNeRF family) ---------------------------------------------------------------
struct F32Layout {
  int W, Bs, Bt, dx, dv, ldx, ldv;
  int64_t total;
  float *X0, *V, *E, *VV, *R;
  float* H[17];   // H[0..Bs]
  float* T[17];   // T[1..Bt]  (T[0] = VV)
  float* ZS[17];  // ZS[1..Bs]  (B, W)
  float* ZT[17];  // ZT[1..Bt]
};

static F32Layout make_layout(const snb_handle_s* h, int64_t M, int64_t B, float* ws) {
  F32Layout L;
  L.W = h->arch.W; L.Bs = h->arch.shape_blocks; L.Bt = h->arch.texture_blocks;
  L.dx = h->d_xyz(); L.dv = h->d_dir();
  L.ldx = (L.dx + 3) & ~3; L.ldv = (L.dv + 3) & ~3;
  Bump b{ws};
  L.X0 = b.take(M * L.ldx);
  L.V = b.take(M * L.ldv);
  for (int j = 0; j <= L.Bs; ++j) L.H[j] = b.take(M * L.W);
  L.E = b.take(M * L.W);
  L.VV = b.take(M * L.W);
  L.T[0] = L.VV;
  for (int j = 1; j <= L.Bt; ++j) L.T[j] = b.take(M * L.W);
  L.R = b.take(M * (L.W / 2));
  for (int j = 1; j <= L.Bs; ++j) L.ZS[j] = b.take(B * L.W);
  for (int j = 1; j <= L.Bt; ++j) L.ZT[j] = b.take(B * L.W);
  L.total = b.used;
  return L;
}

struct AutoRFLayout;
static size_t autorf_workspace_floats(const snb_handle_s* h, int64_t M, int64_t B);
static size_t autorf_bwd_scratch_floats(const snb_handle_s* h, int64_t M, int64_t B);
static int autorf_forward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B, const float* shape_latent,
                          const float* texture_latent, float* sigma, float* rgb, float* ws, cudaStream_t st);
static int autorf_backward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B, const float* shape_latent,
                           const float* texture_latent, const float* sigma, const float* g_sigma, const float* g_rgb, const float* ws,
                           float* scratch, float* g_xyz, float* g_viewdir, float* g_shape_latent, float* g_texture_latent,
                           float* const* gw, cudaStream_t st);

size_t f32_workspace_floats(const snb_handle_s* h, int64_t M, int64_t B) {
  if (h->arch.arch == SNB_ARCH_AUTORF) return autorf_workspace_floats(h, M, B);
  return (size_t)make_layout(h, M, B, nullptr).total + 16;
}

size_t f32_bwd_scratch_floats(const snb_handle_s* h, int64_t M, int64_t B) {
  if (h->arch.arch == SNB_ARCH_AUTORF) return autorf_bwd_scratch_floats(h, M, B);
  const int W = h->arch.W;
  const int ldx = (h->d_xyz() + 3) & ~3, ldv = (h->d_dir() + 3) & ~3;
  return (size_t)(2 * al4(M * W) + al4(M * (W / 2)) + al4(M * ldx) + al4(M * ldv) + al4(M) +
                  (h->arch.shape_blocks + h->arch.texture_blocks) * al4(B * W) + 16);
}

// Y = act((A [+ rowadd]) W^T + b [+ Y])
static int fwd_linear(const float* A, int lda, int64_t M, int K, const float* Wt, int ldw, const float* bias, int N,
                      float* Y, int ldy, int act, int accumulate, const float* rowadd, int64_t rpo, cudaStream_t st) {
  GemmArgs g{};
  g.A = A; g.sAi = lda; g.sAk = 1;
  g.B = Wt; g.sBk = 1; g.sBj = ldw;
  g.C = Y; g.ldc = ldy; g.M = M; g.N = N; g.K = K;
  g.a_add = rowadd; g.a_add_ld = K; g.a_rows_per_obj = rpo > 0 ? rpo : 1;
  g.bias = bias; g.accumulate = accumulate; g.act = act;
  return launch_sgemm(g, true, true, st);
}

// dX = dY W  (dY: M x N(out), W: (out, in) with row stride ldw, dX: M x K(in))
static int bwd_data(const float* dY, int ldy, int64_t M, int N_out, const float* Wt, int ldw, int K_in, float* dX,
                    int ldx, int accumulate, cudaStream_t st) {
  GemmArgs g{};
  g.A = dY; g.sAi = ldy; g.sAk = 1;
  g.B = Wt; g.sBk = ldw; g.sBj = 1;
  g.C = dX; g.ldc = ldx; g.M = M; g.N = K_in; g.K = N_out;
  g.accumulate = accumulate;
  return launch_sgemm(g, true, false, st);
}

// dW (out x in, row stride ldw) += dY^T (X [+ rowadd]);  db += colsum dY.  dW/db must be zeroed by the caller.
static int bwd_weight(const float* dY, int ldy, int64_t M, int N_out, const float* X, int ldx, int K_in, float* dW,
                      int ldw, float* db, const float* rowadd, int64_t rpo, cudaStream_t st) {
  if (dW != nullptr) {
    GemmArgs g{};
    g.A = dY; g.sAi = 1; g.sAk = ldy;
    g.B = X; g.sBk = ldx; g.sBj = 1;
    g.C = dW; g.ldc = ldw; g.M = N_out; g.N = K_in; g.K = M;
    g.b_add = rowadd; g.b_add_ld = K_in; g.b_rows_per_obj = rpo > 0 ? rpo : 1;
    g.k_split = 2048;
    if (launch_sgemm(g, false, false, st)) return 1;
  }
  if (db != nullptr && M > 0) {
    const int rpb = 2048;
    colsum_kernel<<<(unsigned)ceil_div(M, rpb), 256, 0, st>>>(dY, ldy, N_out, M, rpb, db);
    SNB_LAUNCH_CHECK();
  }
  return 0;
}

static int mask_colsum(float* g, const float* hmask, int ld, int width, int64_t M, int64_t B, float* colsum,
                       cudaStream_t st) {
  if (M == 0) return 0;
  const int64_t rpo = M / B;
  const int rows_per_chunk = 256;
  const int chunks = (int)ceil_div(rpo, rows_per_chunk);
  mask_colsum_kernel<<<(unsigned)(B * chunks), 256, 0, st>>>(g, hmask, ld, width, rpo, chunks, rows_per_chunk, colsum);
  SNB_LAUNCH_CHECK();
  return 0;
}

static int zero(float* p, int64_t n, cudaStream_t st) {
  if (n == 0 || p == nullptr) return 0;
  SNB_CHECK_CUDA(cudaMemsetAsync(p, 0, n * sizeof(float), st));
  return 0;
}

#define TRY(x) do { if ((x) != 0) return 1; } while (0)

int f32_forward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                const float* shape_latent, const float* texture_latent, float* sigma, float* rgb, float* ws,
                cudaStream_t st) {
  if (h->arch.arch == SNB_ARCH_AUTORF) return autorf_forward(h, xyz, viewdir, M, B, shape_latent, texture_latent, sigma, rgb, ws, st);
  SNB_REQUIRE(h->arch.arch == SNB_ARCH_CODENERF, "f32_forward: arch %d not handled here", h->arch.arch);
  F32Layout L = make_layout(h, M, B, ws);
  const int W = L.W, D = h->arch.latent_dim;
  const int64_t rpo = M / B;
  const auto& ly = h->layers;
  pe_fwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(xyz, M, h->arch.num_xyz_freq, L.X0, L.ldx);
  SNB_LAUNCH_CHECK();
  pe_fwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(viewdir, M, h->arch.num_dir_freq, L.V, L.ldv);
  SNB_LAUNCH_CHECK();
  // shape/texture_latent_layer_j once per object (model_codenerf.py:51,59): one launch; ZS[1..Bs], ZT[1..Bt] are contiguous
  TRY(latent_forward_fused(h, B, shape_latent, texture_latent, L.ZS[1], nullptr, st));
  (void)D;
  TRY(fwd_linear(L.X0, L.ldx, M, L.dx, ly[h->iX].w, L.dx, ly[h->iX].b, W, L.H[0], W, 1, 0, nullptr, 0, st));
  for (int j = 1; j <= L.Bs; ++j)
    TRY(fwd_linear(L.H[j - 1], W, M, W, ly[h->iS(j)].w, W, ly[h->iS(j)].b, W, L.H[j], W, 1, 0, L.ZS[j], rpo, st));
  TRY(fwd_linear(L.H[L.Bs], W, M, W, ly[h->iES].w, W, ly[h->iES].b, W, L.E, W, 0, 0, nullptr, 0, st));
  TRY(fwd_linear(L.E, W, M, W, ly[h->iSG].w, W, ly[h->iSG].b, 1, sigma, 1, 0, 0, nullptr, 0, st));
  softplus_kernel<<<ew_grid(M), 256, 0, st>>>(sigma, M);
  SNB_LAUNCH_CHECK();
  // encoding_viewdir on cat([E, PE(viewdir)]) (model_codenerf.py:56-57) as two accumulating GEMMs
  TRY(fwd_linear(L.E, W, M, W, ly[h->iEV].w, W + L.dv, nullptr, W, L.VV, W, 0, 0, nullptr, 0, st));
  TRY(fwd_linear(L.V, L.ldv, M, L.dv, ly[h->iEV].w + W, W + L.dv, ly[h->iEV].b, W, L.VV, W, 1, 1, nullptr, 0, st));
  for (int j = 1; j <= L.Bt; ++j)
    TRY(fwd_linear(L.T[j - 1], W, M, W, ly[h->iT(j)].w, W, ly[h->iT(j)].b, W, L.T[j], W, 1, 0, L.ZT[j], rpo, st));
  TRY(fwd_linear(L.T[L.Bt], W, M, W, ly[h->iR0].w, W, ly[h->iR0].b, W / 2, L.R, W / 2, 1, 0, nullptr, 0, st));
  TRY(fwd_linear(L.R, W / 2, M, W / 2, ly[h->iR2].w, W / 2, ly[h->iR2].b, 3, rgb, 3, 0, 0, nullptr, 0, st));
  return 0;
}

int f32_backward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                 const float* shape_latent, const float* texture_latent, const float* sigma, const float* g_sigma,
                 const float* g_rgb, const float* ws, float* scratch, float* g_xyz, float* g_viewdir,
                 float* g_shape_latent, float* g_texture_latent, float* const* gw, cudaStream_t st) {
  if (h->arch.arch == SNB_ARCH_AUTORF)
    return autorf_backward(h, xyz, viewdir, M, B, shape_latent, texture_latent, sigma, g_sigma, g_rgb, ws, scratch, g_xyz, g_viewdir,
                           g_shape_latent, g_texture_latent, gw, st);
  SNB_REQUIRE(h->arch.arch == SNB_ARCH_CODENERF, "f32_backward: arch %d not handled here", h->arch.arch);
  F32Layout L = make_layout(h, M, B, const_cast<float*>(ws));
  const int W = L.W, D = h->arch.latent_dim, W2 = W / 2;
  const int64_t rpo = M / B;
  const auto& ly = h->layers;
  Bump sb{scratch};
  float* dA = sb.take(M * W);
  float* dB = sb.take(M * W);
  float* dR = sb.take(M * W2);
  float* dX0 = sb.take(M * L.ldx);
  float* dV = sb.take(M * L.ldv);
  float* gsp = sb.take(M);
  float* dZ = sb.take((int64_t)(L.Bs + L.Bt) * al4(B * W));
  auto dZS = [&](int j) { return dZ + (int64_t)(j - 1) * al4(B * W); };
  auto dZT = [&](int j) { return dZ + (int64_t)(L.Bs + j - 1) * al4(B * W); };
  auto GW = [&](int layer) -> float* { return gw ? gw[2 * layer] : nullptr; };
  auto GB = [&](int layer) -> float* { return gw ? gw[2 * layer + 1] : nullptr; };
  if (gw) {
    for (size_t i = 0; i < ly.size(); ++i) {
      TRY(zero(gw[2 * i], (int64_t)ly[i].out * ly[i].in, st));
      TRY(zero(gw[2 * i + 1], ly[i].out, st));
    }
  }
  TRY(zero(dZ, (int64_t)(L.Bs + L.Bt) * al4(B * W), st));

  // rgb head: rgb = R W2^T + b2 ; R = relu(T_Bt W1^T + b1)
  TRY(bwd_weight(g_rgb, 3, M, 3, L.R, W2, W2, GW(h->iR2), W2, GB(h->iR2), nullptr, 0, st));
  TRY(bwd_data(g_rgb, 3, M, 3, ly[h->iR2].w, W2, W2, dR, W2, 0, st));
  TRY(mask_colsum(dR, L.R, W2, W2, M, B, nullptr, st));
  TRY(bwd_weight(dR, W2, M, W2, L.T[L.Bt], W, W, GW(h->iR0), W, GB(h->iR0), nullptr, 0, st));
  float* cur = dA;   // gradient w.r.t. the OUTPUT of the layer being unwound
  float* nxt = dB;
  TRY(bwd_data(dR, W2, M, W2, ly[h->iR0].w, W, W, cur, W, 0, st));
  // texture blocks: T_j = relu((T_{j-1} + ZT_j) Wj^T + bj)
  for (int j = L.Bt; j >= 1; --j) {
    TRY(mask_colsum(cur, L.T[j], W, W, M, B, nullptr, st));                       // -> grad of pre-activation
    TRY(bwd_weight(cur, W, M, W, L.T[j - 1], W, W, GW(h->iT(j)), W, GB(h->iT(j)), L.ZT[j], rpo, st));
    TRY(bwd_data(cur, W, M, W, ly[h->iT(j)].w, W, W, nxt, W, 0, st));             // grad of (T_{j-1} + ZT_j)
    TRY(mask_colsum(nxt, nullptr, W, W, M, B, dZT(j), st));                       // latent grad = per-object column sum
    float* t = cur; cur = nxt; nxt = t;
  }
  // encoding_viewdir: VV = relu([E, V] Wv^T + bv)
  TRY(mask_colsum(cur, L.VV, W, W, M, B, nullptr, st));
  TRY(bwd_weight(cur, W, M, W, L.E, W, W, GW(h->iEV), W + L.dv, GB(h->iEV), nullptr, 0, st));
  TRY(bwd_weight(cur, W, M, W, L.V, L.ldv, L.dv, gw ? GW(h->iEV) + W : nullptr, W + L.dv, nullptr, nullptr, 0, st));
  if (g_viewdir) TRY(bwd_data(cur, W, M, W, ly[h->iEV].w + W, W + L.dv, L.dv, dV, L.ldv, 0, st));
  TRY(bwd_data(cur, W, M, W, ly[h->iEV].w, W + L.dv, W, nxt, W, 0, st));          // dE (texture branch)
  { float* t = cur; cur = nxt; nxt = t; }
  // sigma head: sigma = softplus(E wσ + bσ)
  softplus_bwd_kernel<<<ew_grid(M), 256, 0, st>>>(sigma, g_sigma, gsp, M);
  SNB_LAUNCH_CHECK();
  TRY(bwd_weight(gsp, 1, M, 1, L.E, W, W, GW(h->iSG), W, GB(h->iSG), nullptr, 0, st));
  TRY(bwd_data(gsp, 1, M, 1, ly[h->iSG].w, W, W, cur, W, 1, st));                  // dE += gsp ⊗ wσ
  // encoding_shape (no activation)
  TRY(bwd_weight(cur, W, M, W, L.H[L.Bs], W, W, GW(h->iES), W, GB(h->iES), nullptr, 0, st));
  TRY(bwd_data(cur, W, M, W, ly[h->iES].w, W, W, nxt, W, 0, st));
  { float* t = cur; cur = nxt; nxt = t; }
  for (int j = L.Bs; j >= 1; --j) {
    TRY(mask_colsum(cur, L.H[j], W, W, M, B, nullptr, st));
    TRY(bwd_weight(cur, W, M, W, L.H[j - 1], W, W, GW(h->iS(j)), W, GB(h->iS(j)), L.ZS[j], rpo, st));
    TRY(bwd_data(cur, W, M, W, ly[h->iS(j)].w, W, W, nxt, W, 0, st));
    TRY(mask_colsum(nxt, nullptr, W, W, M, B, dZS(j), st));
    float* t = cur; cur = nxt; nxt = t;
  }
  // encoding_xyz
  TRY(mask_colsum(cur, L.H[0], W, W, M, B, nullptr, st));
  TRY(bwd_weight(cur, W, M, W, L.X0, L.ldx, L.dx, GW(h->iX), L.dx, GB(h->iX), nullptr, 0, st));
  if (g_xyz) {
    TRY(bwd_data(cur, W, M, W, ly[h->iX].w, L.dx, L.dx, dX0, L.ldx, 0, st));
    pe_bwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(dX0, L.ldx, xyz, M, h->arch.num_xyz_freq, g_xyz);
    SNB_LAUNCH_CHECK();
  }
  if (g_viewdir) {
    pe_bwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(dV, L.ldv, viewdir, M, h->arch.num_dir_freq, g_viewdir);
    SNB_LAUNCH_CHECK();
  }
  // latent layers (per object): ZS_j = relu(latent Wsl_j^T + b)
  if (g_shape_latent) TRY(zero(g_shape_latent, B * D, st));
  if (g_texture_latent) TRY(zero(g_texture_latent, B * D, st));
  for (int j = 1; j <= L.Bs; ++j) {
    TRY(mask_colsum(dZS(j), L.ZS[j], W, W, B, B, nullptr, st));
    TRY(bwd_weight(dZS(j), W, B, W, shape_latent, D, D, GW(h->iSL(j)), D, GB(h->iSL(j)), nullptr, 0, st));
    if (g_shape_latent) TRY(bwd_data(dZS(j), W, B, W, ly[h->iSL(j)].w, D, D, g_shape_latent, D, 1, st));
  }
  for (int j = 1; j <= L.Bt; ++j) {
    TRY(mask_colsum(dZT(j), L.ZT[j], W, W, B, B, nullptr, st));
    TRY(bwd_weight(dZT(j), W, B, W, texture_latent, D, D, GW(h->iTL(j)), D, GB(h->iTL(j)), nullptr, 0, st));
    if (g_texture_latent) TRY(bwd_data(dZT(j), W, B, W, ly[h->iTL(j)].w, D, D, g_texture_latent, D, 1, st));
  }
  return 0;
}


// =====================================================================================================================
// AutoRF decoder (SURVEY 8a7, model_autorf.py:156-186), fp32.  W = latent_dim = D.  With P = relu(encoding_xyz(PE(x))):
//   shape:    s_0 = shape_latent (per object);  s_{j+1} = relu(shape_layer_j((s_j + P) / 2)),  j = 0 .. Bs-2
//             sigma = softplus(sigma.0((s_{Bs-1} + P) / 2))
//   texture:  t_0 = texture_latent (per object); t_{j+1} = relu(texture_layer_j((t_j + P) / 2)), j = 0 .. Bt-3
//             t'  = relu(texture_layer_{Bt-2}([ (t_{Bt-2} + s_{Bs-1} + P) / 3, PE(d) ]))
//             rgb = sigmoid(rgb.0([ (t' + P) / 2, PE(d) ]))
// Every Linear input (the mixed tensors) is kept for the weight gradients; the `cat` layers are two accumulating GEMMs.
// Layers (handle order): 0 encoding_xyz | 1..Bs-1 shape_layer_j | iSG sigma.0 | iSG+1..iSG+Bt-2 texture_layer_j (plain) |
// iSG+Bt-1 texture_layer_{Bt-2} (D x (D + dv)) | iR0 rgb.0 (3 x (D + dv)).
// =====================================================================================================================
// out[m][c] = scale * (t0 + t1 [+ t2]);  a term with bcast != 0 is per object: row m / rows_per_obj of a (B, D) tensor
__global__ void mix_kernel(float* __restrict__ out, const float* __restrict__ t0, int b0, const float* __restrict__ t1, int b1,
                           const float* __restrict__ t2, int b2, int D, int64_t M, int64_t rpo, float scale) {
  const int64_t n = M * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / D;
    const int c = (int)(i - m * D);
    const int64_t o = m / rpo;
    float v = t0[(b0 ? o : m) * D + c] + t1[(b1 ? o : m) * D + c];
    if (t2 != nullptr) v += t2[(b2 ? o : m) * D + c];
    out[i] = v * scale;   // (a + b) / 2 == (a + b) * 0.5f exactly; / 3 is rounded like the reference's division below
  }
}
// out = (t0 + t1 + t2) / 3 with a true division (model_autorf.py:176)
__global__ void mix3_div_kernel(float* __restrict__ out, const float* __restrict__ t0, int b0, const float* __restrict__ t1, int b1,
                                const float* __restrict__ t2, int D, int64_t M, int64_t rpo) {
  const int64_t n = M * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / D;
    const int c = (int)(i - m * D);
    const int64_t o = m / rpo;
    out[i] = (t0[(b0 ? o : m) * D + c] + t1[(b1 ? o : m) * D + c] + t2[i]) / 3.f;
  }
}
__global__ void axpy_kernel(float* __restrict__ y, const float* __restrict__ x, int64_t n, float scale, int accumulate) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = (accumulate ? y[i] : 0.f) + scale * x[i];
}
__global__ void sigmoid_kernel(float* __restrict__ x, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    x[i] = 1.f / (1.f + expf(-x[i]));
}
__global__ void sigmoid_bwd_kernel(const float* __restrict__ y, const float* __restrict__ g, float* __restrict__ g_pre, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    g_pre[i] = g[i] * y[i] * (1.f - y[i]);
}

struct AutoRFLayout {
  int D, Bs, Bt, dx, dv, ldx, ldv;
  int64_t total;
  float *X0, *V, *P, *Asig, *C, *Tv, *Cr, *RGB;
  float* S[17];    // S[1..Bs-1]  (S[0] = the shape latent, per object)
  float* As[17];   // As[0..Bs-2] = (s_j + P) / 2
  float* T[17];    // T[1..Bt-2]  (T[0] = the texture latent)
  float* At[17];   // At[0..Bt-3]
};

static AutoRFLayout autorf_layout(const snb_handle_s* h, int64_t M, float* ws) {
  AutoRFLayout L;
  L.D = h->arch.latent_dim; L.Bs = h->arch.shape_blocks; L.Bt = h->arch.texture_blocks;
  L.dx = h->d_xyz(); L.dv = h->d_dir();
  L.ldx = (L.dx + 3) & ~3; L.ldv = (L.dv + 3) & ~3;
  Bump b{ws};
  L.X0 = b.take(M * L.ldx);
  L.V = b.take(M * L.ldv);
  L.P = b.take(M * L.D);
  for (int j = 1; j <= L.Bs - 1; ++j) L.S[j] = b.take(M * L.D);
  for (int j = 0; j <= L.Bs - 2; ++j) L.As[j] = b.take(M * L.D);
  L.Asig = b.take(M * L.D);
  for (int j = 1; j <= L.Bt - 2; ++j) L.T[j] = b.take(M * L.D);
  for (int j = 0; j <= L.Bt - 3; ++j) L.At[j] = b.take(M * L.D);
  L.C = b.take(M * L.D);
  L.Tv = b.take(M * L.D);
  L.Cr = b.take(M * L.D);
  L.RGB = b.take(M * 4);
  L.total = b.used;
  return L;
}

static size_t autorf_workspace_floats(const snb_handle_s* h, int64_t M, int64_t) { return (size_t)autorf_layout(h, M, nullptr).total + 16; }
static size_t autorf_bwd_scratch_floats(const snb_handle_s* h, int64_t M, int64_t) {
  const int D = h->arch.latent_dim, ldx = (h->d_xyz() + 3) & ~3, ldv = (h->d_dir() + 3) & ~3;
  return (size_t)(4 * al4(M * D) + al4(M * ldx) + al4(M * ldv) + al4(M) + al4(M * 4) + 16);
}

static int mix2(float* out, const float* a, bool a_obj, const float* P, int D, int64_t M, int64_t rpo, cudaStream_t st) {
  if (M == 0) return 0;
  mix_kernel<<<ew_grid(M * D), 256, 0, st>>>(out, a, a_obj ? 1 : 0, P, 0, nullptr, 0, D, M, rpo, 0.5f);
  SNB_LAUNCH_CHECK();
  return 0;
}
static int axpy(float* y, const float* x, int64_t n, float scale, bool accumulate, cudaStream_t st) {
  if (n == 0) return 0;
  axpy_kernel<<<ew_grid(n), 256, 0, st>>>(y, x, n, scale, accumulate ? 1 : 0);
  SNB_LAUNCH_CHECK();
  return 0;
}

static int autorf_forward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B, const float* shape_latent,
                          const float* texture_latent, float* sigma, float* rgb, float* ws, cudaStream_t st) {
  AutoRFLayout L = autorf_layout(h, M, ws);
  const int D = L.D, Bs = L.Bs, Bt = L.Bt, iSG = h->iSG, iTV = h->iSG + Bt - 1, iR0 = h->iR0;
  const int64_t rpo = M / B;
  const auto& ly = h->layers;
  if (M == 0) return 0;
  pe_fwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(xyz, M, h->arch.num_xyz_freq, L.X0, L.ldx);
  SNB_LAUNCH_CHECK();
  pe_fwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(viewdir, M, h->arch.num_dir_freq, L.V, L.ldv);
  SNB_LAUNCH_CHECK();
  TRY(fwd_linear(L.X0, L.ldx, M, L.dx, ly[0].w, L.dx, ly[0].b, D, L.P, D, 1, 0, nullptr, 0, st));
  // shape branch
  for (int j = 0; j <= Bs - 2; ++j) {
    TRY(mix2(L.As[j], j == 0 ? shape_latent : L.S[j], j == 0, L.P, D, M, rpo, st));
    TRY(fwd_linear(L.As[j], D, M, D, ly[1 + j].w, D, ly[1 + j].b, D, L.S[j + 1], D, 1, 0, nullptr, 0, st));
  }
  const float* s_last = Bs - 1 == 0 ? shape_latent : L.S[Bs - 1];
  const bool s_last_obj = Bs - 1 == 0;
  TRY(mix2(L.Asig, s_last, s_last_obj, L.P, D, M, rpo, st));
  TRY(fwd_linear(L.Asig, D, M, D, ly[iSG].w, D, ly[iSG].b, 1, sigma, 1, 0, 0, nullptr, 0, st));
  softplus_kernel<<<ew_grid(M), 256, 0, st>>>(sigma, M);
  SNB_LAUNCH_CHECK();
  // texture branch
  for (int j = 0; j <= Bt - 3; ++j) {
    TRY(mix2(L.At[j], j == 0 ? texture_latent : L.T[j], j == 0, L.P, D, M, rpo, st));
    TRY(fwd_linear(L.At[j], D, M, D, ly[iSG + 1 + j].w, D, ly[iSG + 1 + j].b, D, L.T[j + 1], D, 1, 0, nullptr, 0, st));
  }
  const float* t_last = Bt - 2 == 0 ? texture_latent : L.T[Bt - 2];
  mix3_div_kernel<<<ew_grid(M * D), 256, 0, st>>>(L.C, t_last, Bt - 2 == 0 ? 1 : 0, s_last, s_last_obj ? 1 : 0, L.P, D, M, rpo);
  SNB_LAUNCH_CHECK();
  TRY(fwd_linear(L.C, D, M, D, ly[iTV].w, D + L.dv, nullptr, D, L.Tv, D, 0, 0, nullptr, 0, st));
  TRY(fwd_linear(L.V, L.ldv, M, L.dv, ly[iTV].w + D, D + L.dv, ly[iTV].b, D, L.Tv, D, 1, 1, nullptr, 0, st));
  TRY(mix2(L.Cr, L.Tv, false, L.P, D, M, rpo, st));
  TRY(fwd_linear(L.Cr, D, M, D, ly[iR0].w, D + L.dv, nullptr, 3, rgb, 3, 0, 0, nullptr, 0, st));
  TRY(fwd_linear(L.V, L.ldv, M, L.dv, ly[iR0].w + D, D + L.dv, ly[iR0].b, 3, rgb, 3, 0, 1, nullptr, 0, st));
  sigmoid_kernel<<<ew_grid(M * 3), 256, 0, st>>>(rgb, M * 3);
  SNB_LAUNCH_CHECK();
  SNB_CHECK_CUDA(cudaMemcpyAsync(L.RGB, rgb, (size_t)M * 3 * sizeof(float), cudaMemcpyDeviceToDevice, st));   // sigmoid' needs the output
  return 0;
}

static int autorf_backward(const snb_handle_s* h, const float* xyz, const float* viewdir, int64_t M, int64_t B, const float* shape_latent,
                           const float* texture_latent, const float* sigma, const float* g_sigma, const float* g_rgb, const float* ws,
                           float* scratch, float* g_xyz, float* g_viewdir, float* g_shape_latent, float* g_texture_latent,
                           float* const* gw, cudaStream_t st) {
  AutoRFLayout L = autorf_layout(h, M, const_cast<float*>(ws));
  const int D = L.D, Bs = L.Bs, Bt = L.Bt, iSG = h->iSG, iTV = h->iSG + Bt - 1, iR0 = h->iR0;
  const auto& ly = h->layers;
  auto GW = [&](int layer) -> float* { return gw ? gw[2 * layer] : nullptr; };
  auto GB = [&](int layer) -> float* { return gw ? gw[2 * layer + 1] : nullptr; };
  if (gw)
    for (size_t i = 0; i < ly.size(); ++i) {
      TRY(zero(gw[2 * i], (int64_t)ly[i].out * ly[i].in, st));
      TRY(zero(gw[2 * i + 1], ly[i].out, st));
    }
  if (g_shape_latent) TRY(zero(g_shape_latent, B * D, st));
  if (g_texture_latent) TRY(zero(g_texture_latent, B * D, st));
  if (M == 0) return 0;
  Bump sb{scratch};
  float* cur = sb.take(M * D);    // gradient w.r.t. the output of the layer being unwound
  float* tmp = sb.take(M * D);    // gradient w.r.t. a Linear's (mixed) input
  float* gP = sb.take(M * D);     // accumulated gradient of P (it enters every mix)
  float* gS = sb.take(M * D);     // gradient of s_{Bs-1} (sigma head + the 3-way mix)
  float* dX0 = sb.take(M * L.ldx);
  float* dV = sb.take(M * L.ldv);
  float* gsp = sb.take(M);
  float* dpre = sb.take(M * 4);
  // rgb = sigmoid([Cr, V] Wr^T + br)
  sigmoid_bwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(L.RGB, g_rgb, dpre, M * 3);
  SNB_LAUNCH_CHECK();
  TRY(bwd_weight(dpre, 3, M, 3, L.Cr, D, D, GW(iR0), D + L.dv, GB(iR0), nullptr, 0, st));
  TRY(bwd_weight(dpre, 3, M, 3, L.V, L.ldv, L.dv, gw ? GW(iR0) + D : nullptr, D + L.dv, nullptr, nullptr, 0, st));
  if (g_viewdir) TRY(bwd_data(dpre, 3, M, 3, ly[iR0].w + D, D + L.dv, L.dv, dV, L.ldv, 0, st));
  TRY(bwd_data(dpre, 3, M, 3, ly[iR0].w, D + L.dv, D, tmp, D, 0, st));              // d Cr;  Cr = (Tv + P) / 2
  TRY(axpy(gP, tmp, M * D, 0.5f, false, st));
  TRY(axpy(cur, tmp, M * D, 0.5f, false, st));                                       // d Tv
  // Tv = relu([C, V] Wv^T + bv)
  TRY(mask_colsum(cur, L.Tv, D, D, M, B, nullptr, st));
  TRY(bwd_weight(cur, D, M, D, L.C, D, D, GW(iTV), D + L.dv, GB(iTV), nullptr, 0, st));
  TRY(bwd_weight(cur, D, M, D, L.V, L.ldv, L.dv, gw ? GW(iTV) + D : nullptr, D + L.dv, nullptr, nullptr, 0, st));
  if (g_viewdir) TRY(bwd_data(cur, D, M, D, ly[iTV].w + D, D + L.dv, L.dv, dV, L.ldv, 1, st));
  TRY(bwd_data(cur, D, M, D, ly[iTV].w, D + L.dv, D, tmp, D, 0, st));               // d C;  C = (t_{Bt-2} + s_{Bs-1} + P) / 3
  const float third = 1.f / 3.f;
  TRY(axpy(gP, tmp, M * D, third, true, st));
  TRY(axpy(gS, tmp, M * D, third, false, st));
  TRY(axpy(cur, tmp, M * D, third, false, st));                                      // d t_{Bt-2}
  // texture chain: t_{j+1} = relu(texture_layer_j(At_j)),  At_j = (t_j + P) / 2
  for (int j = Bt - 3; j >= 0; --j) {
    TRY(mask_colsum(cur, L.T[j + 1], D, D, M, B, nullptr, st));
    TRY(bwd_weight(cur, D, M, D, L.At[j], D, D, GW(iSG + 1 + j), D, GB(iSG + 1 + j), nullptr, 0, st));
    TRY(bwd_data(cur, D, M, D, ly[iSG + 1 + j].w, D, D, tmp, D, 0, st));
    TRY(axpy(gP, tmp, M * D, 0.5f, true, st));
    TRY(axpy(cur, tmp, M * D, 0.5f, false, st));                                     // d t_j
  }
  if (g_texture_latent) TRY(mask_colsum(cur, nullptr, D, D, M, B, g_texture_latent, st));   // t_0 = the latent: per-object column sums
  // sigma = softplus(sigma.0(Asig)),  Asig = (s_{Bs-1} + P) / 2
  softplus_bwd_kernel<<<ew_grid(M), 256, 0, st>>>(sigma, g_sigma, gsp, M);
  SNB_LAUNCH_CHECK();
  TRY(bwd_weight(gsp, 1, M, 1, L.Asig, D, D, GW(iSG), D, GB(iSG), nullptr, 0, st));
  TRY(bwd_data(gsp, 1, M, 1, ly[iSG].w, D, D, tmp, D, 0, st));
  TRY(axpy(gP, tmp, M * D, 0.5f, true, st));
  TRY(axpy(gS, tmp, M * D, 0.5f, true, st));
  // shape chain
  float* g = gS;
  for (int j = Bs - 2; j >= 0; --j) {
    TRY(mask_colsum(g, L.S[j + 1], D, D, M, B, nullptr, st));
    TRY(bwd_weight(g, D, M, D, L.As[j], D, D, GW(1 + j), D, GB(1 + j), nullptr, 0, st));
    TRY(bwd_data(g, D, M, D, ly[1 + j].w, D, D, tmp, D, 0, st));
    TRY(axpy(gP, tmp, M * D, 0.5f, true, st));
    TRY(axpy(cur, tmp, M * D, 0.5f, false, st));                                     // d s_j
    g = cur;
  }
  if (g_shape_latent) TRY(mask_colsum(g, nullptr, D, D, M, B, g_shape_latent, st));
  // P = relu(encoding_xyz(X0))
  TRY(mask_colsum(gP, L.P, D, D, M, B, nullptr, st));
  TRY(bwd_weight(gP, D, M, D, L.X0, L.ldx, L.dx, GW(0), L.dx, GB(0), nullptr, 0, st));
  if (g_xyz) {
    TRY(bwd_data(gP, D, M, D, ly[0].w, L.dx, L.dx, dX0, L.ldx, 0, st));
    pe_bwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(dX0, L.ldx, xyz, M, h->arch.num_xyz_freq, g_xyz);
    SNB_LAUNCH_CHECK();
  }
  if (g_viewdir) {
    pe_bwd_kernel<<<ew_grid(M * 3), 256, 0, st>>>(dV, L.ldv, viewdir, M, h->arch.num_dir_freq, g_viewdir);
    SNB_LAUNCH_CHECK();
  }
  (void)shape_latent; (void)texture_latent;
  return 0;
}

}  // namespace snb
