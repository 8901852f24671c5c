// C-ABI entry points that are not tied to one kernel file: error text, device info, the per-model
// handle, and the decoder MLP's entry points (argument checks; decoder.cu picks and runs the back end).
#include "common.cuh"
#include "decoder.h"
#include <stdarg.h>
#include <string.h>
#include <new>

namespace snb {

static thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return -1; }
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { cudaGetLastError(); return -1; }
    cached = n; cached_dev = dev;
  }
  return cached;
}

}  // namespace snb

using namespace snb;

extern "C" int snb_abi_version(void) { return SNB_ABI_VERSION; }
extern "C" uint64_t snb_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" const char* snb_last_error(void) { return g_err; }

extern "C" int snb_device_info(int* sms, int* major, int* minor) {
  int dev = 0;
  SNB_CHECK_CUDA(cudaGetDevice(&dev));
  int a = 0, b = 0, c = 0;
  SNB_CHECK_CUDA(cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev));
  SNB_CHECK_CUDA(cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMajor, dev));
  SNB_CHECK_CUDA(cudaDeviceGetAttribute(&c, cudaDevAttrComputeCapabilityMinor, dev));
  if (sms) *sms = a;
  if (major) *major = b;
  if (minor) *minor = c;
  return 0;
}

static int expected_layers(const snb_arch& a) {
  if (a.arch == SNB_ARCH_CODENERF) return 6 + 2 * a.shape_blocks + 2 * a.texture_blocks;
  return a.shape_blocks + a.texture_blocks + 1;
}

extern "C" int snb_create(snb_handle* out, const snb_arch* arch) {
  SNB_REQUIRE(out && arch, "snb_create: null argument");
  SNB_REQUIRE(arch->arch == SNB_ARCH_CODENERF || arch->arch == SNB_ARCH_AUTORF, "snb_create: unknown arch %d", arch->arch);
  SNB_REQUIRE(arch->shape_blocks >= 1 && arch->shape_blocks <= 16 && arch->texture_blocks >= 1 && arch->texture_blocks <= 16,
              "snb_create: blocks out of range");
  SNB_REQUIRE(arch->W >= 8 && arch->W % 8 == 0 && arch->latent_dim >= 1, "snb_create: W must be a positive multiple of 8");
  SNB_REQUIRE(arch->num_xyz_freq >= 0 && arch->num_xyz_freq <= 16 && arch->num_dir_freq >= 0 && arch->num_dir_freq <= 16,
              "snb_create: frequency count out of range");
  if (arch->arch == SNB_ARCH_AUTORF)
    SNB_REQUIRE(arch->texture_blocks >= 2 && arch->W == arch->latent_dim, "snb_create: AutoRF needs texture_blocks >= 2, W == latent_dim");
  snb_handle_s* h = new (std::nothrow) snb_handle_s();
  SNB_REQUIRE(h != nullptr, "snb_create: out of memory");
  h->arch = *arch;
  const int W = arch->W, D = arch->latent_dim, dx = 3 + 6 * arch->num_xyz_freq, dv = 3 + 6 * arch->num_dir_freq;
  auto add = [&](int o, int i) { snb_layer l; l.out = o; l.in = i; h->layers.push_back(l); };
  if (arch->arch == SNB_ARCH_CODENERF) {
    add(W, dx);
    for (int j = 0; j < arch->shape_blocks; ++j) { add(W, D); add(W, W); }
    h->iES = (int)h->layers.size(); add(W, W);
    h->iSG = (int)h->layers.size(); add(1, W);
    h->iEV = (int)h->layers.size(); add(W, W + dv);
    for (int j = 0; j < arch->texture_blocks; ++j) { add(W, D); add(W, W); }
    h->iR0 = (int)h->layers.size(); add(W / 2, W);
    h->iR2 = (int)h->layers.size(); add(3, W / 2);
  } else {
    add(D, dx);
    for (int j = 0; j < arch->shape_blocks - 1; ++j) add(D, D);
    h->iSG = (int)h->layers.size(); add(1, D);
    for (int j = 0; j < arch->texture_blocks - 2; ++j) add(D, D);
    add(D, D + dv);
    h->iR0 = (int)h->layers.size(); add(3, D + dv);
  }
  if ((int)h->layers.size() != expected_layers(*arch)) { delete h; SNB_REQUIRE(false, "snb_create: internal layer count"); }
  *out = h;
  return 0;
}

extern "C" int snb_destroy(snb_handle h) {
  delete h;
  return 0;
}

extern "C" int snb_num_weight_tensors(snb_handle h) { return h ? 2 * (int)h->layers.size() : -1; }

extern "C" int snb_layer_shape(snb_handle h, int layer, int* out_dim, int* in_dim) {
  SNB_REQUIRE(h && layer >= 0 && layer < (int)h->layers.size(), "snb_layer_shape: bad layer");
  if (out_dim) *out_dim = h->layers[layer].out;
  if (in_dim) *in_dim = h->layers[layer].in;
  return 0;
}

extern "C" int snb_set_weights(snb_handle h, const float* const* tensors, int32_t n) {
  SNB_REQUIRE(h && tensors, "snb_set_weights: null argument");
  SNB_REQUIRE(n == 2 * (int)h->layers.size(), "snb_set_weights: expected %d tensors, got %d", 2 * (int)h->layers.size(), n);
  for (size_t i = 0; i < h->layers.size(); ++i) {
    SNB_REQUIRE(tensors[2 * i] && tensors[2 * i + 1], "snb_set_weights: tensor %d is null", (int)(2 * i));
    h->layers[i].w = tensors[2 * i];
    h->layers[i].b = tensors[2 * i + 1];
  }
  h->weights_set = true;
  return 0;
}

extern "C" int snb_tc_set_debug(snb_handle h, float* acts) { SNB_REQUIRE(h, "snb_tc_set_debug: null handle"); h->dbg_acts = acts; return 0; }
extern "C" int snb_tc_set_trace(snb_handle h, long long* stamps) { SNB_REQUIRE(h, "snb_tc_set_trace: null handle"); h->trace = stamps; return 0; }
extern "C" int snb_tc_set_cg2(snb_handle h, int32_t mode) { SNB_REQUIRE(h, "snb_tc_set_cg2: null handle"); h->cg2_mode = mode; return 0; }
extern "C" int snb_kernel_timing_enable(snb_handle h, int32_t on) { SNB_REQUIRE(h, "snb_kernel_timing_enable: null handle"); decoder_timing_enable(h, on); return 0; }
extern "C" int snb_kernel_timing_read(snb_handle h, int32_t which, float* ms_host, int32_t max_n) {
  if (!h) return 0;
  return decoder_timing_read(h, which, ms_host, max_n);
}

extern "C" size_t snb_packed_bytes(snb_handle h) { return h ? decoder_packed_bytes(h) : 0; }

extern "C" int snb_pack_weights(snb_handle h, void* packed, void* stream) {
  SNB_REQUIRE(h && packed, "snb_pack_weights: null argument");
  SNB_REQUIRE(h->weights_set, "snb_pack_weights: call snb_set_weights first");
  return decoder_pack_weights(h, packed, (cudaStream_t)stream);
}

static int check_mlp_args(snb_handle h, int32_t precision, int64_t M, int64_t B) {
  SNB_REQUIRE(h != nullptr, "mlp: null handle");
  SNB_REQUIRE(h->weights_set, "mlp: weights not set");
  SNB_REQUIRE(precision == SNB_PREC_FP32 || precision == SNB_PREC_BF16 || precision == SNB_PREC_BF16_TRAIN || precision == SNB_PREC_FP32_TC,
              "mlp: unknown precision %d", precision);
  SNB_REQUIRE(M >= 0 && B >= 1 && M % B == 0, "mlp: n_rows (%lld) must be a multiple of n_objs (%lld)", (long long)M, (long long)B);
  SNB_REQUIRE(sm_count() > 0, "mlp: no CUDA device (there is no CPU fallback)");
  return 0;
}

extern "C" size_t snb_mlp_workspace_bytes(snb_handle h, int64_t M, int64_t B, int32_t precision) {
  return h ? decoder_workspace_bytes(h, precision, M, B) : 0;
}

extern "C" size_t snb_mlp_bwd_scratch_bytes(snb_handle h, int64_t M, int64_t B, int32_t precision) {
  return h ? decoder_scratch_bytes(h, precision, M, B) : 0;
}

extern "C" int snb_mlp_fwd(snb_handle h, int32_t precision, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                           const float* shape_latent, const float* texture_latent, float* sigma, float* rgb,
                           void* workspace, void* stream) {
  if (check_mlp_args(h, precision, M, B)) return 2;
  if (M == 0) return 0;
  SNB_REQUIRE(xyz && viewdir && shape_latent && texture_latent && sigma && rgb && workspace, "mlp_fwd: null pointer");
  return decoder_forward(h, precision, xyz, viewdir, M, B, shape_latent, texture_latent, sigma, rgb, workspace, (cudaStream_t)stream);
}

extern "C" int snb_mlp_bwd(snb_handle h, int32_t precision, const float* xyz, const float* viewdir, int64_t M, int64_t B,
                           const float* shape_latent, const float* texture_latent, const float* sigma,
                           const float* g_sigma, const float* g_rgb, const void* workspace, void* scratch, float* g_xyz,
                           float* g_viewdir, float* g_shape_latent, float* g_texture_latent, float* const* g_weights,
                           void* stream) {
  if (check_mlp_args(h, precision, M, B)) return 2;
  if (M == 0) return decoder_zero_grads(h, B, g_shape_latent, g_texture_latent, g_weights, (cudaStream_t)stream);   // no samples
  SNB_REQUIRE(xyz && viewdir && shape_latent && texture_latent && sigma && g_sigma && g_rgb && workspace && scratch,
              "mlp_bwd: null pointer");
  return decoder_backward(h, precision, xyz, viewdir, M, B, shape_latent, texture_latent, sigma, g_sigma, g_rgb, workspace, scratch,
                          g_xyz, g_viewdir, g_shape_latent, g_texture_latent, g_weights, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// Gradient all-reduce of the sharded modes (SURVEY 8b / 8e): ONE ncclAllReduce(sum, fp32) over the caller's flat buffer
// -- [d cam_pose (12) | d shapecode (D) | d texturecode (D) | loss] in the ray-sharded mode (2.1 KB), the flat weight-gradient
// buffer in the data-parallel mode -- on the caller's communicator and stream.  NCCL is not linked: the entry point is looked
// up in the libnccl the process already uses (torch's), so the library has no NCCL dependency of its own.
// ---------------------------------------------------------------------------------------------------------------------
#include <dlfcn.h>

namespace {
typedef int (*nccl_allreduce_fn)(const void*, void*, size_t, int /*ncclDataType_t*/, int /*ncclRedOp_t*/, void* /*ncclComm_t*/, cudaStream_t);
nccl_allreduce_fn find_nccl_allreduce() {
  static std::atomic<nccl_allreduce_fn> cached{nullptr};
  nccl_allreduce_fn f = cached.load(std::memory_order_acquire);
  if (f) return f;
  void* sym = dlsym(RTLD_DEFAULT, "ncclAllReduce");
  if (!sym) {
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the instance torch.distributed already loaded
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW);
    if (lib) sym = dlsym(lib, "ncclAllReduce");
  }
  f = reinterpret_cast<nccl_allreduce_fn>(sym);
  if (f) cached.store(f, std::memory_order_release);
  return f;
}
}  // namespace

extern "C" int snb_allreduce_grads(snb_handle h, void* nccl_comm, float* flat, size_t n, void* stream) {
  (void)h;   // the handle names the model the gradients belong to; the reduction itself is stateless
  SNB_REQUIRE(nccl_comm != nullptr && (flat != nullptr || n == 0), "snb_allreduce_grads: null communicator or buffer");
  if (n == 0) return 0;
  nccl_allreduce_fn f = find_nccl_allreduce();
  SNB_REQUIRE(f != nullptr, "snb_allreduce_grads: ncclAllReduce not found (libnccl.so.2 is not loaded in this process)");
  const int rc = f(flat, flat, n, /*ncclFloat32*/ 7, /*ncclSum*/ 0, nccl_comm, (cudaStream_t)stream);
  SNB_REQUIRE(rc == 0, "snb_allreduce_grads: ncclAllReduce failed with ncclResult_t %d", rc);
  return 0;
}
