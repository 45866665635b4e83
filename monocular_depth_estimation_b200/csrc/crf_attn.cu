// Window-attention core: parameter block and the two stream-ordered launchers the block / layer orchestration and the
// stage-level C entry points (crf_attn_fwd / crf_attn_bwd) call.  The kernels live in crf_attn_async.cu.
#include <stdlib.h>

#include "crf_attn_common.cuh"

namespace crf {

int launch_attn_fwd_async(const AttnParams& P, const crf_block_desc& d, cudaStream_t st);
int launch_attn_bwd_async(const AttnParams& P, const crf_block_desc& d, cudaStream_t st);
int launch_attn_fwd_wide(const AttnParams& P, const crf_block_desc& d, cudaStream_t st);  // crf_attn_wide.cu
int launch_attn_bwd_wide(const AttnParams& P, const crf_block_desc& d, cudaStream_t st);

// head_dim 16 / 32: crf_attn_async.cu (pipelined).  head_dim 64 / 128: crf_attn_wide.cu (32-wide slices of a head,
// synchronous structure; verified on B200 through tools/hwcheck, profiles/r01_hwcheck.txt).
bool head_dim_supported(int hd) { return hd == 16 || hd == 32 || hd == 64 || hd == 128; }

int fill_attn_params(AttnParams& P, const crf_block_desc& d) {
  CRF_CHECK(d.num_heads > 0 && d.C % d.num_heads == 0 && head_dim_supported(d.C / d.num_heads),
            "attention core: head_dim must be 16, 32, 64 or 128 (C=%d, heads=%d)", d.C, d.num_heads);
  CRF_CHECK(d.window >= kMinWindow && d.window <= kMaxWindow, "attention core: window must be in [%d, %d] (got %d)",
            kMinWindow, kMaxWindow, d.window);
  CRF_CHECK(d.shift >= 0 && d.shift < d.window, "shift_size must in 0-window_size");
  P.gm = WindowGeom(d.H, d.W, d.window, d.shift);
  P.B = d.B;
  P.C = d.C;
  P.nH = d.num_heads;
  P.hd = d.C / d.num_heads;
  P.total_windows = d.B * P.gm.nW;
  P.npairs = (P.total_windows + 1) / 2;
  P.rcp_nW = 1.0f / static_cast<float>(P.gm.nW);
  P.rcp_nWw = 1.0f / static_cast<float>(P.gm.nWw);
  CRF_CHECK(P.total_windows < (1 << 22), "attention core: too many windows (%d)", P.total_windows);
  P.prof = getenv("CRF_ATTN_PROF") != nullptr;  // development: per-phase cycle counts of block (0,0)
  return 0;
}

int launch_attn_fwd(const crf_block_desc& d, const void* qk, const void* vb, const float* qk_bias, float scale,
                    const float* table, const float* ext_mask, int ext_mask_nw, void* o, float* lse, cudaStream_t st,
                    int ext_replaces) {
  AttnParams P{};
  if (fill_attn_params(P, d)) return 1;
  P.qk = reinterpret_cast<const __nv_bfloat16*>(qk);
  P.vb = reinterpret_cast<const __nv_bfloat16*>(vb);
  P.qk_bias = qk_bias;
  P.table = table;
  P.scale = scale;
  P.ext_mask = ext_mask_nw > 0 ? ext_mask : nullptr;
  P.ext_mask_nw = ext_mask_nw > 0 ? ext_mask_nw : 1;
  P.ext_replaces = (P.ext_mask != nullptr && ext_replaces) ? 1 : 0;
  P.o = reinterpret_cast<__nv_bfloat16*>(o);
  P.lse = lse;
  return P.hd > 32 ? launch_attn_fwd_wide(P, d, st) : launch_attn_fwd_async(P, d, st);
}

int launch_attn_bwd(const crf_block_desc& d, const void* qk, const void* vb, const float* qk_bias, float scale,
                    const float* table, const float* ext_mask, int ext_mask_nw, const float* lse, const void* dout,
                    void* dqk, float* dv, int dv_acc, float* d_table, float* d_qk_bias, cudaStream_t st, int ext_replaces) {
  AttnParams P{};
  if (fill_attn_params(P, d)) return 1;
  P.qk = reinterpret_cast<const __nv_bfloat16*>(qk);
  P.vb = reinterpret_cast<const __nv_bfloat16*>(vb);
  P.qk_bias = qk_bias;
  P.table = table;
  P.scale = scale;
  P.ext_mask = ext_mask_nw > 0 ? ext_mask : nullptr;
  P.ext_mask_nw = ext_mask_nw > 0 ? ext_mask_nw : 1;
  P.ext_replaces = (P.ext_mask != nullptr && ext_replaces) ? 1 : 0;
  P.lse = const_cast<float*>(lse);
  P.dout = reinterpret_cast<const __nv_bfloat16*>(dout);
  P.dqk = reinterpret_cast<__nv_bfloat16*>(dqk);
  P.dv = dv;
  P.dv_acc = dv_acc;
  P.d_table = d_table;
  P.d_qk_bias = d_qk_bias;
  return P.hd > 32 ? launch_attn_bwd_wide(P, d, st) : launch_attn_bwd_async(P, d, st);
}

}  // namespace crf
