// Refine-iteration glue (SURVEY 8(f) rank 1), the parts around the render: pose parametrisation and the optimiser step of
// optimizer_nuscenes.py:684-699 and :757-769 / :1762-1769, one launch each instead of ~60 + ~15 elementwise launches.
//   pose  : rot_vec (axis-angle), trans_vec -> rot_mat2opt = Rodrigues(rot_vec) (what pytorch3d.transforms.axis_angle_to_matrix
//           evaluates), t2opt = trans_vec; with opt_cam_pose false (every shipped config) cam2opt = [R^T | -R^T t] (:695-697).
//           The same launch builds the shared sample vector of utils.sample_from_rays (utils.py:154-167) from the DETACHED
//           translation norm (utils.py:468-469), so nothing in an iteration needs the host.
//   AdamW : torch.optim.AdamW's update (decoupled weight decay, bias correction) on R independent rows (one per object) of up to 8
//           small tensors with their own learning rates, state on the device, each row with its own step counter and active byte.
// Scalar work: one thread does the 3x3 algebra in double, S threads the sample vector, one block per row the optimiser.
#include "common.cuh"
#include "../../include/supnerf_b200.h"
#include <math.h>

namespace snb {

struct Rod {   // R = I + a K + b K^2,  K = [v]x
  double th, a, b, da, db;   // da = a'(th) / th, db = b'(th) / th  (so that d a / d v_i = da * v_i)
};
__device__ __forceinline__ Rod rod_coeffs(const double v[3]) {
  Rod r;
  const double t2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
  r.th = sqrt(t2);
  if (r.th < 1e-4) {   // series: a = 1 - t^2/6, b = 1/2 - t^2/24
    r.a = 1.0 - t2 / 6.0; r.b = 0.5 - t2 / 24.0; r.da = -1.0 / 3.0 + t2 / 30.0; r.db = -1.0 / 12.0 + t2 / 180.0;
  } else {
    const double s = sin(r.th), c = cos(r.th);
    r.a = s / r.th; r.b = (1.0 - c) / t2;
    r.da = (r.th * c - s) / (t2 * r.th);                       // a'(th) / th
    r.db = (r.th * s - 2.0 * (1.0 - c)) / (t2 * t2);           // b'(th) / th
  }
  return r;
}
__device__ __forceinline__ void skew(const double v[3], double K[9]) {
  K[0] = 0; K[1] = -v[2]; K[2] = v[1]; K[3] = v[2]; K[4] = 0; K[5] = -v[0]; K[6] = -v[1]; K[7] = v[0]; K[8] = 0;
}
__device__ __forceinline__ void mat3(const double A[9], const double B[9], double C[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
__device__ __forceinline__ void rodrigues(const double v[3], const Rod& r, double R[9]) {
  double K[9], K2[9];
  skew(v, K); mat3(K, K, K2);
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0 ? 1.0 : 0.0) + r.a * K[i] + r.b * K2[i];
}

// One block per object.  Object b reads row int(it[b]) of its jitter table (B, T, S) -- `it` being its optimiser's device-side step
// counter, so a captured iteration needs neither an index_select nor a counter-increment launch.  z2 / jitter2 (optional): a second
// sample vector from the same pose and another draw (the per-iteration lidar-pixel evaluation, optimizer_nuscenes.py:759-769).
// Every table read is guarded: an active object whose counter lies outside [0, T) gets NaN in z / z2 and sets *err (if given); an
// inactive one reads row 0 instead and reports nothing (its render runs on placeholder inputs and is ignored).
__global__ void __launch_bounds__(1024) refine_pose_fwd_kernel(const float* __restrict__ rot_vec, const float* __restrict__ trans_vec,
                                                              int opt_cam_pose, const float* __restrict__ obj_diag, int S,
                                                              const float* __restrict__ jitter, const float* __restrict__ jitter2,
                                                              const float* __restrict__ it, int T, const uint8_t* __restrict__ active,
                                                              int* __restrict__ err, float* __restrict__ cam, float* __restrict__ z,
                                                              float* __restrict__ z2) {
  __shared__ double tn;
  const int b = blockIdx.x;
  rot_vec += 3 * b; trans_vec += 3 * b; cam += 12 * b;
  if (threadIdx.x == 0) {
    const double v[3] = {rot_vec[0], rot_vec[1], rot_vec[2]}, t[3] = {trans_vec[0], trans_vec[1], trans_vec[2]};
    double R[9];
    rodrigues(v, rod_coeffs(v), R);
    float c[12];
    if (opt_cam_pose) {
      for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) c[4 * i + j] = (float)R[3 * i + j]; c[4 * i + 3] = (float)t[i]; }
    } else {   // cam2opt = [R^T | -R^T t]
      for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) c[4 * i + j] = (float)R[3 * j + i];
        c[4 * i + 3] = (float)(-(R[i] * t[0] + R[3 + i] * t[1] + R[6 + i] * t[2]));
      }
    }
    for (int i = 0; i < 12; ++i) cam[i] = c[i];
    tn = sqrt((double)c[3] * c[3] + (double)c[7] * c[7] + (double)c[11] * c[11]);   // norm of the fp32 translation, in double
  }
  __syncthreads();
  // utils.py:468-469 + :154-167: near/far python floats (double), torch.linspace's fp32 formula, jitter scaled by (far-near)/(2S)
  const double half = (double)obj_diag[b] / 2.0, near = tn - half, far = tn + half, dist = (far - near) / (2.0 * S);
  const float start = (float)(near + dist), end = (float)(far - dist);
  const float step = S > 1 ? (end - start) / (float)(S - 1) : 0.f;
  const float scale = (float)((far - near) / (2.0 * S));
  const float c = it[b];
  const bool in_table = c >= 0.f && c < (float)T;    // false for NaN too
  const bool bad = !in_table && active[b] != 0;
  const int64_t row = (int64_t)b * T + (in_table ? (int64_t)c : 0);
  if (bad && err != nullptr && threadIdx.x == 0) *err = 1;
  for (int i = threadIdx.x; i < S; i += blockDim.x) {
    const float lin = i < S / 2 ? __fadd_rn(start, __fmul_rn(step, (float)i)) : __fsub_rn(end, __fmul_rn(step, (float)(S - 1 - i)));
    z[(int64_t)b * S + i] = bad ? __int_as_float(0x7fffffff) : __fadd_rn(lin, __fmul_rn(jitter[row * S + i], scale));
    if (z2 != nullptr) z2[(int64_t)b * S + i] = bad ? __int_as_float(0x7fffffff) : __fadd_rn(lin, __fmul_rn(jitter2[row * S + i], scale));
  }
}

__global__ void refine_pose_bwd_kernel(const float* __restrict__ rot_vec, const float* __restrict__ trans_vec, int opt_cam_pose,
                                       const float* __restrict__ g_cam, float* __restrict__ g_rot, float* __restrict__ g_trans) {
  if (threadIdx.x != 0) return;
  rot_vec += 3 * blockIdx.x; trans_vec += 3 * blockIdx.x; g_cam += 12 * blockIdx.x; g_rot += 3 * blockIdx.x; g_trans += 3 * blockIdx.x;   // one block per object
  const double v[3] = {rot_vec[0], rot_vec[1], rot_vec[2]}, t[3] = {trans_vec[0], trans_vec[1], trans_vec[2]};
  const Rod r = rod_coeffs(v);
  double R[9], K[9], K2[9];
  skew(v, K); mat3(K, K, K2);
  rodrigues(v, r, R);
  double G[12];
  for (int i = 0; i < 12; ++i) G[i] = g_cam[i];
  double GR[9], gt[3];   // d loss / d R, d loss / d t
  if (opt_cam_pose) {
    for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) GR[3 * i + j] = G[4 * i + j]; gt[i] = G[4 * i + 3]; }
  } else {
    // cam[i][j] = R[j][i];  cam[i][3] = -sum_k R[k][i] t[k]
    for (int k = 0; k < 3; ++k) {
      gt[k] = 0.0;
      for (int i = 0; i < 3; ++i) {
        GR[3 * k + i] = G[4 * i + k] - G[4 * i + 3] * t[k];
        gt[k] -= R[3 * k + i] * G[4 * i + 3];
      }
    }
  }
  // R = I + a K + b K^2:  d R / d v_i = da v_i K + a E_i + db v_i K^2 + b (E_i K + K E_i)
  double sK = 0.0, sK2 = 0.0;
  for (int i = 0; i < 9; ++i) { sK += GR[i] * K[i]; sK2 += GR[i] * K2[i]; }
  for (int i = 0; i < 3; ++i) {
    double e[3] = {0.0, 0.0, 0.0}, E[9], EK[9], KE[9];
    e[i] = 1.0;
    skew(e, E); mat3(E, K, EK); mat3(K, E, KE);
    double sE = 0.0, sEK = 0.0;
    for (int j = 0; j < 9; ++j) { sE += GR[j] * E[j]; sEK += GR[j] * (EK[j] + KE[j]); }
    g_rot[i] = (float)(r.da * v[i] * sK + r.a * sE + r.db * v[i] * sK2 + r.b * sEK);
    g_trans[i] = (float)gt[i];
  }
}

constexpr int kMaxAdamGroups = 8;
struct AdamGroups {
  int n_groups;
  float* p[kMaxAdamGroups]; const float* g[kMaxAdamGroups]; float* m[kMaxAdamGroups]; float* v[kMaxAdamGroups];
  int n[kMaxAdamGroups]; float lr[kMaxAdamGroups];   // n: elements of ONE row of the tensor (row r starts at r * n)
  float beta1, beta2, eps, weight_decay;
  float* step;             // device: steps taken so far, one counter per row (incremented here)
  const uint8_t* active;   // per row; an inactive row is left bit-for-bit unchanged
  // loss history (hist null = none): an active row r writes {loss3[r][0..2], loss_rgb2[r * rgb2_stride]} to hist[r][step[r]][0..3]
  const float* loss3; const float* loss_rgb2; int rgb2_stride; float* hist; int hist_rows;
};

// torch.optim.AdamW (amsgrad off, maximize off): p *= 1 - lr wd; m, v update; p -= lr / bc1 * m / (sqrt(v) / sqrt(bc2) + eps).
// One block per row; each row's bias corrections come from its own step counter.
__global__ void __launch_bounds__(1024) adamw_step_kernel(const __grid_constant__ AdamGroups A) {
  const int r = blockIdx.x;
  if (A.active[r] == 0) return;
  __shared__ float s_s;
  if (threadIdx.x == 0) s_s = A.step[r];
  __syncthreads();
  const float t = s_s + 1.f;
  const float bc1 = 1.f - powf(A.beta1, t), bc2s = sqrtf(1.f - powf(A.beta2, t));
  for (int gi = 0; gi < A.n_groups; ++gi) {
    const float lr = A.lr[gi], step_size = lr / bc1;
    const int64_t o = (int64_t)r * A.n[gi];
    float* __restrict__ P = A.p[gi] + o; const float* __restrict__ G = A.g[gi] + o;
    float* __restrict__ M = A.m[gi] + o; float* __restrict__ V = A.v[gi] + o;
    for (int i = threadIdx.x; i < A.n[gi]; i += blockDim.x) {
      const float g = G[i];
      float p = P[i] * (1.f - lr * A.weight_decay);
      const float m = A.beta1 * M[i] + (1.f - A.beta1) * g;
      const float v = A.beta2 * V[i] + (1.f - A.beta2) * g * g;
      M[i] = m; V[i] = v;
      p -= step_size * (m / (sqrtf(v) / bc2s + A.eps));
      P[i] = p;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const float s = s_s;
    if (A.hist != nullptr && s >= 0.f && s < (float)A.hist_rows) {
      float* h = A.hist + ((int64_t)r * A.hist_rows + (int64_t)s) * 4;
      h[0] = A.loss3[3 * r]; h[1] = A.loss3[3 * r + 1]; h[2] = A.loss3[3 * r + 2]; h[3] = A.loss_rgb2[(int64_t)r * A.rgb2_stride];
    }
    A.step[r] = t;
  }
}

}  // namespace snb

using namespace snb;

extern "C" int snb_refine_pose_slots_fwd(const float* rot_vec, const float* trans_vec, int32_t n_slots, int32_t opt_cam_pose,
                                         const float* obj_diag, int32_t n_samples, const float* jitter, const float* jitter2,
                                         const float* step_counters, int32_t table_rows, const uint8_t* active, int32_t* err_flag,
                                         float* cam, float* z, float* z2, void* stream) {
  SNB_REQUIRE(n_slots >= 1 && rot_vec && trans_vec && cam && z && jitter && obj_diag && step_counters && active && n_samples >= 1 &&
              table_rows >= 1, "refine_pose_slots_fwd: bad arguments");
  SNB_REQUIRE(z2 == nullptr || jitter2 != nullptr, "refine_pose_slots_fwd: z2 needs jitter2");
  SNB_REQUIRE(sm_count() > 0, "refine_pose_slots_fwd: no CUDA device (there is no CPU fallback)");
  const int threads = (n_samples + 31) / 32 * 32 < 1024 ? (n_samples + 31) / 32 * 32 : 1024;
  refine_pose_fwd_kernel<<<n_slots, threads, 0, (cudaStream_t)stream>>>(rot_vec, trans_vec, opt_cam_pose, obj_diag, n_samples, jitter, jitter2,
                                                                        step_counters, table_rows, active, err_flag, cam, z, z2);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_refine_pose_batch_bwd(const float* rot_vec, const float* trans_vec, int32_t n_objs, int32_t opt_cam_pose,
                                         const float* g_cam, float* g_rot, float* g_trans, void* stream) {
  SNB_REQUIRE(n_objs >= 1 && rot_vec && trans_vec && g_cam && g_rot && g_trans, "refine_pose_batch_bwd: bad arguments");
  SNB_REQUIRE(sm_count() > 0, "refine_pose_batch_bwd: no CUDA device (there is no CPU fallback)");
  refine_pose_bwd_kernel<<<n_objs, 32, 0, (cudaStream_t)stream>>>(rot_vec, trans_vec, opt_cam_pose, g_cam, g_rot, g_trans);
  SNB_LAUNCH_CHECK();
  return 0;
}

extern "C" int snb_adamw_step_rows(int32_t n_groups, float* const* params, const float* const* grads, float* const* exp_avg,
                                   float* const* exp_avg_sq, const int32_t* row_sizes, const float* lrs, float beta1, float beta2,
                                   float eps, float weight_decay, int32_t n_rows, float* steps, const uint8_t* active,
                                   const float* loss3, const float* loss_rgb2, int32_t loss_rgb2_stride, float* loss_history,
                                   int32_t history_rows, void* stream) {
  SNB_REQUIRE(n_groups >= 1 && n_groups <= kMaxAdamGroups, "adamw_step_rows: 1..%d tensors", kMaxAdamGroups);
  SNB_REQUIRE(n_rows >= 1, "adamw_step_rows: n_rows >= 1");
  SNB_REQUIRE(params && grads && exp_avg && exp_avg_sq && row_sizes && lrs && steps && active, "adamw_step_rows: null pointer");
  SNB_REQUIRE(loss_history == nullptr || (loss3 && loss_rgb2 && history_rows >= 1), "adamw_step_rows: the loss history needs its sources");
  SNB_REQUIRE(sm_count() > 0, "adamw_step_rows: no CUDA device (there is no CPU fallback)");
  AdamGroups A{};
  A.n_groups = n_groups;
  int widest = 1;
  for (int i = 0; i < n_groups; ++i) {
    SNB_REQUIRE(params[i] && grads[i] && exp_avg[i] && exp_avg_sq[i] && row_sizes[i] >= 0, "adamw_step_rows: bad tensor %d", i);
    A.p[i] = params[i]; A.g[i] = grads[i]; A.m[i] = exp_avg[i]; A.v[i] = exp_avg_sq[i]; A.n[i] = row_sizes[i]; A.lr[i] = lrs[i];
    widest = row_sizes[i] > widest ? row_sizes[i] : widest;
  }
  A.beta1 = beta1; A.beta2 = beta2; A.eps = eps; A.weight_decay = weight_decay;
  A.step = steps; A.active = active;
  A.loss3 = loss3; A.loss_rgb2 = loss_rgb2; A.rgb2_stride = loss_rgb2_stride; A.hist = loss_history; A.hist_rows = history_rows;
  const int threads = (widest + 31) / 32 * 32 < 1024 ? (widest + 31) / 32 * 32 : 1024;
  adamw_step_kernel<<<n_rows, threads, 0, (cudaStream_t)stream>>>(A);
  SNB_LAUNCH_CHECK();
  return 0;
}
