// Shared pieces of the window-attention kernels: parameter block, relative-position-bias indexing, register
// re-balancing between warp-specialised roles.
#pragma once
#include "crf_host.h"
#include "crf_ptx.cuh"
#include "crf_window.cuh"

namespace crf {

struct AttnParams {
  WindowGeom gm;
  int B, C, nH;
  int hd;             // head_dim: 32, or 16 (tiles stay 32 wide, the upper half zero-filled)
  int total_windows;  // B * nW
  int npairs;
  const __nv_bfloat16* qk;   // (T, 2C)
  const __nv_bfloat16* vb;   // (T, C)
  const float* qk_bias;      // (2C)
  const float* table;        // ((2ws-1)^2, nH)
  float scale;
  const float* ext_mask;     // optional additive mask (nwm, N, N) f32 (N = ws^2), window index = global window % nwm; or nullptr
  int ext_mask_nw;
  int ext_replaces;          // 1: ext_mask REPLACES the closed-form shift mask (CRFBlock.forward's mask_matrix); 0: added on top
  // forward
  __nv_bfloat16* o;          // (T, C)
  float* lse;                // (B*nW, nH, 64)
  // backward
  const __nv_bfloat16* dout; // (T, C)
  __nv_bfloat16* dqk;        // (T, 2C)
  float* dv;                 // (T, C)
  int dv_acc;
  float* d_table;            // ((2ws-1)^2, nH)
  float* d_qk_bias;          // (2C)
  float rcp_nW, rcp_nWw;     // 1 / windows per image, 1 / windows per row (fast exact division in the kernels)
  int prof;                  // development: block (0,0) prints per-phase cycle counts (CRF_ATTN_PROF=1)
};

// register re-balancing between warp-specialised roles (whole warpgroups execute these)
template <int N>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }

int fill_attn_params(AttnParams& P, const crf_block_desc& d);

}  // namespace crf
