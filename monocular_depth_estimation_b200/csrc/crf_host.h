// Host-side helpers shared by the translation units of libcrf_sm100.so: error reporting, device guard,
// TMA tensor-map creation through the driver entry point (no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/crf_sm100.h"

namespace crf {

int set_error(const char* fmt, ...);  // always returns 1
const char* get_error();

#define CRF_CHECK(cond, ...)                  \
  do {                                        \
    if (!(cond)) return crf::set_error(__VA_ARGS__); \
  } while (0)

#define CRF_CUDA(call)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (call);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return crf::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// Sets the device for the duration of a call and restores the previous one (entry points may be called from
// the autograd worker thread whose current device is not ours).
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    cur = dev;
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != cur) cudaSetDevice(prev);
  }
  int cur = -1;
};

// 2-D bf16 row-major tensor (rows, cols) -> tiled tensor map with 128-byte swizzle, box = (64 cols, box_rows).
int make_tmap_bf16(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
// 2-D fp32 row-major tensor (rows, cols) -> box = (32 cols, box_rows), 128-byte swizzle (epilogue tiles).
int make_tmap_f32(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);

int num_sms(int device);
bool head_dim_supported(int hd);  // 16, 32 (crf_attn_async.cu), 64, 128 (crf_attn_wide.cu)
void note_launch(int n = 1);

// Optional per-kernel timing (crf_timing_enable): CUDA events recorded on the launch stream around each kernel,
// aggregated per label together with the kernel's ALGORITHMIC flops and bytes.  Off by default (zero overhead).
class KernelTimer {
 public:
  KernelTimer(cudaStream_t st, double flops, double bytes, const char* fmt, ...);
  ~KernelTimer();
 private:
  cudaStream_t st_;
  cudaEvent_t e0_ = nullptr, e1_ = nullptr;
  double flops_, bytes_;
  char label_[96];
  bool on_ = false;
};
void timing_enable(bool on);
size_t timing_report(char* buf, size_t cap);   // kernel-launch counter exported as crf_kernel_launches()
long long launch_count();

// Kernel launch with the programmatic-stream-serialization attribute (PDL): the kernel may be scheduled while the
// previous kernel of the stream is still draining; every kernel launched through here begins with pdl_prologue()
// (crf_ptx.cuh), which waits for the previous grid before anything else runs.  cluster_x > 1 launches clusters of
// that many CTAs along x.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_cluster(unsigned cluster_x, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                      cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  return launch_pdl_cluster(1, kern, grid, block, smem, st, static_cast<Args&&>(args)...);
}

// ---- internal launchers (stream-ordered, no allocation) ----
// launch_gemm validates the arguments, picks the kernel with plan_gemm (crf_sched.h), builds the tensor maps with
// gemm_maps and launches the CTA-pair kernel (crf_gemm_pair.cu), the persistent kernel (crf_gemm_persist.cu) or the
// tiled kernel (crf_gemm.cu).
int launch_gemm(const crf_gemm_args& a, cudaStream_t st);
// TMA maps of one GEMM, in the kernels' parameter order.  Maps an epilogue does not use are copies of tmA (never read).
struct GemmMaps {
  CUtensorMap tmA, tmB, tmO0, tmO1, tmAux;
};
// Checks that the epilogue has its outputs and aux input and builds the maps: a K-major operand in boxes of 128 rows (A)
// or b_rows rows (B), an MN-major one in boxes of 64 K-rows, both twice as wide with split3; outputs and aux in boxes
// of 128 rows.
int gemm_maps(const crf_gemm_args& a, uint32_t b_rows, GemmMaps* m);
int launch_gemm_pair(const crf_gemm_args& a, const GemmMaps& m, cudaStream_t st);
int launch_gemm_persistent(const crf_gemm_args& a, const GemmMaps& m, cudaStream_t st);
// crf_precise.cu: the fp32 precision mode (crf_block_desc.precision == CRF_PREC_FP32)
size_t precise_saved_bytes(const crf_block_desc& d);
size_t precise_bwd_bytes(const crf_block_desc& d);
int block_fwd_precise(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, float* y, void* saved,
                      cudaStream_t st);
int block_bwd_precise(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, const float* dy,
                      const void* saved, float* dx, void* dx_bf16, float* dv, int dv_accumulate, const crf_block_grads* g,
                      void* ws, size_t ws_bytes, cudaStream_t st);
bool mlp_fused_supported(int C);                                      // crf_mlp_fused.cu: C = 128, 256
int launch_mlp_fused_fwd(const crf_mlp_args& m, cudaStream_t st);
int mlp_debug_prof(long long* out, int n);                            // CRF_MLP_PROF=1 timeline (debug)
size_t gemm_splitk_workspace_bytes(int M, int N, int K, int device, int* splits_out);
int launch_ln_fwd(const void* x, int x_dtype, int64_t sb, int64_t st_, int64_t sc, int B, int T_img, int C,
                  const float* gamma, const float* beta, float eps, void* xn, float* stats, float* x_copy,
                  cudaStream_t st);
int launch_ln_bwd(const float* g, const float* x, const float* stats, const float* gamma, const float* dres,
                  float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T, int C, cudaStream_t st);
// crf_dgrad_lnbwd.cu: input-gradient GEMM + LayerNorm backward of that input in one kernel (C = 128, 256)
bool dgrad_lnbwd_supported(int C, int K);
int launch_dgrad_lnbwd(const void* dY, const void* W, int K, const float* x, const float* stats, const float* gamma,
                       const float* dres, float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T, int C, int device,
                       cudaStream_t st);
// The closing LayerNorm of a decoder stage over (T, C) fp32 rows, T = B H W tokens.  shuffle_w = W > 0: the
// PixelShuffle(2) that follows is folded into the output store / the gradient load, y and g being (B, 2H, 2W, C/4)
// NHWC maps.
int launch_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                         float* stats, int T, int C, cudaStream_t st, int shuffle_w = 0);
int launch_layernorm_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                         void* dx_bf16, float* dgamma, float* dbeta, int T, int C, cudaStream_t st, int shuffle_w = 0);
int launch_depth_loss_fwd(const void* pred, int pred_dtype, const float* tgt, int n_img, int H, int W, float* sums,
                          float* G, cudaStream_t st);
int launch_depth_loss_bwd(const void* pred, int pred_dtype, const float* tgt, const float* G, const float* gout,
                          int n_img, int H, int W, void* dpred, cudaStream_t st);
int launch_pixel_shuffle_nhwc(const void* src, void* dst, int dtype, int B, int H, int W, int C, int inverse,
                              cudaStream_t st);
int launch_adam_step(const crf_adam_tensor* tensors, int n_tensors, int chunk_elems, double lr, double b1, double b2,
                     double eps, double wd, float* step, cudaStream_t st);
int launch_colsum_bf16(const void* g, float* out, int T, int N, cudaStream_t st);
// crf_bn.cu: training-mode BatchNorm + activation on channels-last bf16 maps (include/crf_sm100.h: crf_bn_fwd / _bwd)
size_t bn_workspace_bytes(int T, int C, int device);
int launch_bn_fwd(const void* x, void* y, const float* weight, const float* bias, float* running_mean,
                  float* running_var, long long* num_batches_tracked, float* save_mean, float* save_invstd, int T, int C,
                  float eps, float momentum, int act, void* ws, size_t ws_bytes, int* tickets, int device,
                  cudaStream_t st);
int launch_bn_bwd(const void* x, const void* dy, const float* weight, const float* bias, const float* save_mean,
                  const float* save_invstd, void* dx, float* dweight, float* dbias, int T, int C, int act, void* ws,
                  size_t ws_bytes, int* tickets, int device, cudaStream_t st);
int launch_cast_bf16(const float* src, void* dst, int64_t n, cudaStream_t st);
int launch_cast4_bf16(const float* const src[4], void* const dst[4], const long long n[4], cudaStream_t st);
int launch_convert_tokens(const void* src, int dtype, int64_t sb, int64_t st_, int64_t sc, int B, int T_img, int C,
                          void* dst_bf16, cudaStream_t st);
int launch_window_gather(const float* x, float* windows, int B, int H, int W, int C, int window, int shift,
                         cudaStream_t st);
int launch_window_scatter(const float* windows, float* x, int B, int H, int W, int C, int window, int shift,
                          cudaStream_t st);
int launch_shift_mask(float* mask, int H, int W, int window, int shift, cudaStream_t st);
int launch_attn_fwd(const crf_block_desc& d, const void* qk, const void* vb, const float* qk_bias, float scale,
                    const float* table, const float* ext_mask, int ext_mask_nw, void* o, float* lse, cudaStream_t st,
                    int ext_replaces = 0);
int launch_attn_bwd(const crf_block_desc& d, const void* qk, const void* vb, const float* qk_bias, float scale,
                    const float* table, const float* ext_mask, int ext_mask_nw, const float* lse, const void* dout,
                    void* dqk, float* dv, int dv_acc, float* d_table, float* d_qk_bias, cudaStream_t st,
                    int ext_replaces = 0);

}  // namespace crf
