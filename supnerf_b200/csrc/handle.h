// Per-model handle shared by the MLP back ends.
#pragma once
#include <memory>
#include <utility>
#include <vector>
#include "../../include/supnerf_b200.h"

struct snb_layer {
  const float* w = nullptr;  // (out, in) row-major fp32, borrowed
  const float* b = nullptr;  // (out)
  int out = 0, in = 0;
};

// byte offsets of the two-tile and split-precision images behind the one-tile bf16 image at 0, and the buffer size (0: not built yet)
struct snb_packed_layout { size_t two_tile = 0, split = 0, bytes = 0; };

struct snb_handle_s {
  snb_arch arch;
  std::vector<snb_layer> layers;  // canonical (state_dict) order
  bool weights_set = false;
  // bf16 back end
  const void* packed = nullptr;   // borrowed: caller-owned buffer filled by snb_pack_weights
  // per-handle caches of pure functions of the architecture (built on first use; a handle is used by one host thread at a time)
  mutable std::shared_ptr<void> tc2_programs;   // mlp_tc2.cu: the step programs of the two-tile kernels
  mutable snb_packed_layout packed_layout;      // decoder.cu: where each weight image sits in the packed buffer
  // test / tuning / measurement hooks, per handle (a handle is used by one host thread at a time; nothing here is process-global)
  float* dbg_acts = nullptr;                    // snb_tc_set_debug
  long long* trace = nullptr;                   // snb_tc_set_trace
  int cg2_mode = -1;                            // snb_tc_set_cg2 (-1: the SNB_TC_CG2 environment variable, default 1)
  bool timing_on = false;                       // snb_kernel_timing_enable
  std::vector<std::pair<void*, void*>> ev_fwd, ev_bwd;   // cudaEvent_t pairs around the tcgen05 kernels
  // CodeNeRF-family layer indices
  int iX = 0, iES = 0, iSG = 0, iEV = 0, iR0 = 0, iR2 = 0;
  int iSL(int j) const { return 1 + 2 * (j - 1); }       // shape_latent_layer_j, j = 1..Bs
  int iS(int j) const { return 2 + 2 * (j - 1); }        // shape_layer_j
  int iTL(int j) const { return iEV + 1 + 2 * (j - 1); } // texture_latent_layer_j
  int iT(int j) const { return iEV + 2 + 2 * (j - 1); }  // texture_layer_j
  int d_xyz() const { return 3 + 6 * arch.num_xyz_freq; }
  int d_dir() const { return 3 + 6 * arch.num_dir_freq; }
};
