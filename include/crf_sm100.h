/*
 * crf_sm100.h -- C ABI of libcrf_sm100.so: the NeWCRFs neural-window FC-CRF block, forward and backward,
 * as hand-written CUDA for sm_100a (B200).
 *
 * This is the drop-in boundary for ONE hot path of LuizGuzzo/Monocular_Depth_Estimation:
 *   src/newcrf_layers.py:30-59    window_partition / window_reverse
 *   src/newcrf_layers.py:110-149  WindowAttention.forward
 *   src/newcrf_layers.py:195-257  CRFBlock.forward
 *   src/newcrf_layers.py:323-363  BasicCRFLayer.forward  (shift mask at :332-350)
 * and the autograd backward of those functions (the reference has no explicit backward code).
 *
 * Conventions
 *   - plain C: pointers, sizes, POD structs; no C++ exceptions cross the boundary.
 *   - every function returns 0 on success, non-zero on error; crf_last_error() returns the message
 *     (thread-local).
 *   - every device buffer (inputs, outputs, saved-for-backward, workspace) is allocated by the caller; the
 *     library never allocates, frees or retains device memory between calls.
 *   - all work is enqueued on the caller's stream (a cudaStream_t passed as void*); no hidden syncs.
 *   - entry points are re-entrant (forward runs on the Python thread, backward on the autograd engine
 *     thread); the device ordinal is taken from the descriptor, not from thread-local CUDA state.
 *   - "tokens" are the B*H*W feature-map positions in natural (b, h, w) order; T = B*H*W.
 */
#ifndef CRF_SM100_H_
#define CRF_SM100_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRF_ABI_VERSION 4
enum { CRF_PREC_BF16 = 0, CRF_PREC_FP32 = 1 };

enum { CRF_DT_F32 = 0, CRF_DT_BF16 = 1 };

/* --------------------------------------------------------------------------------------------------------
 * Problem descriptor of one CRFBlock call (replaces the Python attributes CRFBlock.{dim,num_heads,
 * window_size,shift_size,H,W}, newcrf_layers.py:170-193, and the tensor metadata torch carries).
 * Strides are in ELEMENTS of the tensor's dtype.
 *   x : logical (B, H*W, C)      -- the reference passes a strided view of NCHW (newcrf_layers.py:426)
 *   v : logical (B, H, W, C)     -- strided view of NCHW (newcrf_layers.py:427)
 * ------------------------------------------------------------------------------------------------------ */
typedef struct crf_block_desc {
  int32_t B, H, W, C;
  int32_t num_heads;
  int32_t window;   /* 2..8 (the reference's default 7) */
  int32_t shift;    /* 0 or window/2 */
  int32_t training; /* 1: keep everything backward needs in `saved` */
  int32_t device;   /* CUDA device ordinal that owns every pointer */
  int32_t x_dtype;  /* CRF_DT_* */
  int32_t v_dtype;
  int32_t v_preconverted; /* 1: `v` already is the bf16 token-major copy produced by crf_convert_v */
  int64_t x_stride_b, x_stride_t, x_stride_c;
  int64_t v_stride_b, v_stride_h, v_stride_w, v_stride_c;
  int32_t precision;      /* CRF_PREC_BF16 (default): bf16 tensor-core operands and intermediates, rel 2e-2;
                           * CRF_PREC_FP32: split-operand tensor-core GEMMs + fp32 attention / intermediates, rel 1e-3
                           * (BASELINE.json's two tolerance tiers).  v_preconverted must be 0 in the fp32 mode. */
  int32_t reserved;
} crf_block_desc;

/* fp32 parameters of one CRFBlock, names as in the reference state_dict (SURVEY.md 8b). */
typedef struct crf_block_params {
  const float* norm1_w;  /* (C)      blocks.i.norm1.weight */
  const float* norm1_b;  /* (C)      */
  const float* qk_w;     /* (2C, C)  blocks.i.attn.qk.weight : first C rows -> q, last C rows -> k */
  const float* qk_b;     /* (2C)     */
  const float* rpb_table;/* ((2w-1)^2,nH), w = window: blocks.i.attn.relative_position_bias_table */
  const float* proj_w;   /* (C, C)   */
  const float* proj_b;   /* (C)      */
  const float* norm2_w;  /* (C)      */
  const float* norm2_b;  /* (C)      */
  const float* fc1_w;    /* (4C, C)  */
  const float* fc1_b;    /* (4C)     */
  const float* fc2_w;    /* (C, 4C)  */
  const float* fc2_b;    /* (C)      */
  float qk_scale;        /* head_dim^-0.5 unless overridden (newcrf_layers.py:83) */
  float ln_eps;          /* 1e-5 */
  const float* ext_mask; /* NULL: the shifted-window mask of BasicCRFLayer.forward (newcrf_layers.py:332-350), evaluated
                          * in closed form.  Otherwise an additive (ext_mask_windows, N, N) f32 mask, N = window^2, that REPLACES it
                          * (CRFBlock.forward's mask_matrix argument, :195,236): window w of every image uses
                          * ext_mask[w mod ext_mask_windows]. */
  int32_t ext_mask_windows;
  int32_t reserved;
} crf_block_params;

/* fp32 gradient outputs, same shapes as crf_block_params; the library ACCUMULATES (+=) into them, so the
 * caller zero-fills (or passes .grad buffers directly). */
typedef struct crf_block_grads {
  float* norm1_w; float* norm1_b;
  float* qk_w;    float* qk_b;
  float* rpb_table;
  float* proj_w;  float* proj_b;
  float* norm2_w; float* norm2_b;
  float* fc1_w;   float* fc1_b;
  float* fc2_w;   float* fc2_b;
} crf_block_grads;

const char* crf_last_error(void);
int crf_abi_version(void);
/* number of CUDA kernels this library has launched since it was loaded (bench.py's gpu_launches) */
long long crf_kernel_launches(void);
/* Per-kernel timing for bench.py's roofline: when enabled, every kernel launch is bracketed by CUDA events on its
 * own stream.  crf_timing_report synchronises them and writes a JSON array (one object per kernel label: launches,
 * total_ms, algorithmic flops and bytes per launch) into buf; returns the size needed.  Enabling clears old data. */
int crf_timing_enable(int on);
size_t crf_timing_report(char* buf, size_t cap);

/* Sizes (bytes) of the caller-allocated `saved` buffer (lives from forward to backward when training) and of
 * the scratch workspaces for forward and backward. */
int crf_block_sizes(const crf_block_desc* d, size_t* saved_bytes, size_t* ws_fwd_bytes, size_t* ws_bwd_bytes);

/* One CRFBlock forward: y = block(x, v).   Replaces CRFBlock.forward (newcrf_layers.py:195-257) including
 * WindowAttention.forward (:110-149), window_partition/window_reverse/torch.roll/F.pad (:212-249), the shift
 * mask (:332-350, evaluated in closed form) and Mlp.forward (:21-27).
 *   y : (B, H*W, C) fp32 contiguous. */
int crf_block_fwd(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, float* y,
                  void* saved, void* ws, size_t ws_bytes, void* stream);

/* Backward of crf_block_fwd.  x and v are the SAME buffers (and descriptor) that were passed to forward: x is
 * re-read when it was fp32 token-major (otherwise forward kept a copy in `saved`), v when v_preconverted.
 *   dy : (B, H*W, C) fp32 contiguous;  dx : (B, H*W, C) fp32 contiguous (overwritten)
 *   dv : (B, H, W, C) fp32 contiguous; dv_accumulate != 0 -> dv += (both blocks of a layer share v) */
int crf_block_bwd(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, const float* dy,
                  const void* saved, float* dx, float* dv, int dv_accumulate, const crf_block_grads* g, void* ws,
                  size_t ws_bytes, void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Layer level: BasicCRFLayer.forward (newcrf_layers.py:323-363) -- `depth` blocks with shift 0, window/2, 0, ...
 * that all read the same v -- optionally followed by the LayerNorm that closes a decoder stage (NewCRF.norm_crf,
 * newcrf_layers.py:430-431), in ONE call each way.  Compared with `depth` crf_block_* calls this converts v once,
 * hands the gradient between blocks in fp32 + bf16 without extra casts and accumulates dv inside the kernels.
 *   d      : descriptor of the layer's input x / v (the shift field is ignored; blocks after the first read the
 *            previous block's contiguous fp32 output).  A v that already is bf16, token-major and contiguous is read
 *            in place by both calls (no copy): it must then still be valid, unchanged, in crf_layer_bwd
 *   y      : (B, H*W, C) contiguous, f32, or bf16 when out_dtype == CRF_DT_BF16 (needs the closing norm)
 *   dy     : gradient of y in y's dtype; dx (B, H*W, C) contiguous in x's dtype (f32 or bf16); dv (B, H, W, C) f32
 *            (both overwritten)
 *   g      : `depth` gradient structs (accumulated, +=); dnorm_w / dnorm_b accumulated, NULL without the norm
 * ------------------------------------------------------------------------------------------------------ */
#define CRF_MAX_DEPTH 8
typedef struct crf_layer_args {
  int32_t depth;
  int32_t out_dtype;               /* CRF_DT_F32 or CRF_DT_BF16 */
  const crf_block_params* params;  /* [depth] */
  const float* norm_w;             /* closing LayerNorm weight (C) or NULL */
  const float* norm_b;
  int32_t out_shuffle;             /* 1: the closing LayerNorm writes y with the decoder's PixelShuffle(2) folded in
                                    * (/root/reference/src/model_mobileV3_large_newCRFs.py:116-120): y and dy are
                                    * (B, 2H, 2W, C/4) NHWC maps, y[b, 2h+i, 2w+j, k] = LN(x)[b, h*W+w, 4k+2i+j].
                                    * Needs the closing norm.  (ABI 3) */
} crf_layer_args;
int crf_layer_sizes(const crf_block_desc* d, int depth, int with_norm, size_t* saved_bytes, size_t* ws_bwd_bytes);
int crf_layer_fwd(const crf_block_desc* d, const crf_layer_args* a, const void* x, const void* v, void* y, void* saved,
                  void* stream);
int crf_layer_bwd(const crf_block_desc* d, const crf_layer_args* a, const void* x, const void* v, const void* dy,
                  const void* saved, void* dx, float* dv, const crf_block_grads* g, float* dnorm_w, float* dnorm_b,
                  void* ws, size_t ws_bytes, void* stream);

/* v (B,H,W,C), any strides, fp32/bf16 -> bf16 token-major (T, C) contiguous; done once per BasicCRFLayer
 * because both blocks read the same v (newcrf_layers.py:352-357). Uses the v_* fields of the descriptor. */
int crf_convert_v(const crf_block_desc* d, const void* v, void* v_bf16, void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Stand-alone index-map entry points (bit-exact tests).
 * crf_window_gather  == F.pad -> torch.roll(-shift) -> window_partition   (newcrf_layers.py:215-233, :30-42)
 * crf_window_scatter == window_reverse -> torch.roll(+shift) -> crop       (newcrf_layers.py:239-249, :45-59)
 * crf_shift_mask     == the attn_mask BasicCRFLayer.forward builds         (newcrf_layers.py:332-350)
 *   x       : (B, H, W, C) fp32 contiguous
 *   windows : (B*nW, window*window, C) fp32 contiguous
 *   mask    : (nW, N, N) fp32, N = window*window, values 0 / -100
 * ------------------------------------------------------------------------------------------------------ */
int crf_window_gather(const float* x, float* windows, int B, int H, int W, int C, int window, int shift,
                      void* stream);
int crf_window_scatter(const float* windows, float* x, int B, int H, int W, int C, int window, int shift,
                       void* stream);
int crf_shift_mask(float* mask, int H, int W, int window, int shift, void* stream);

/* --------------------------------------------------------------------------------------------------------
 * Stage-level entry points (unit tests and profiling of the individual kernels).
 * ------------------------------------------------------------------------------------------------------ */
enum {
  CRF_EPI_STORE_F32 = 0,   /* out0 f32 = acc (+ bias)                                          */
  CRF_EPI_STORE_BF16 = 1,  /* out0 bf16 = (acc + bias) * (n < scale_cols ? scale : 1)           */
  CRF_EPI_BIAS_RES_F32 = 2,/* out0 f32 = acc + bias + res(aux1 f32)                             */
  CRF_EPI_BIAS_GELU = 3,   /* out0 bf16 = pre = acc + bias (optional), out1 bf16 = gelu(pre)    */
  CRF_EPI_MUL_DGELU = 4,   /* out0 bf16 = acc * gelu'(pre), pre = aux1 bf16                     */
  CRF_EPI_SPLITK_F32 = 5   /* out0 f32 += acc; split-K partial tiles in `workspace` + reduce  */
};

/* D[M,N] = sum_k A(m,k) * B(n,k) on tcgen05 (bf16 operands, fp32 accumulate in TMEM), TMA-fed.
 * Each operand is a row-major bf16 matrix in one of two orientations:
 *   major 0 (K-major) : stored (MN, K)   -- e.g. activations (tokens, channels), nn.Linear weight (out,in)
 *   major 1 (MN-major): stored (K, MN)   -- e.g. weight (out,in) contracted over `out`, or (tokens, ch)
 *                                           contracted over tokens (weight gradients) */
typedef struct crf_gemm_args {
  const void* A; const void* B;
  int32_t a_major, b_major;
  int32_t M, N, K;
  int32_t epilogue;
  int32_t split_k;         /* CRF_EPI_SPLITK_F32 only: 0 = automatic, > 0 = upper bound on the K splits */
  void* out0; void* out1;
  const float* bias;       /* (N) or NULL */
  const void* aux1;        /* residual f32 (M,N) or pre bf16 (M,N) */
  int64_t ld_out;          /* row stride (elements) of out0/out1/aux1 */
  float scale; int32_t scale_cols;
  int32_t device;
  void* workspace;         /* CRF_EPI_SPLITK_F32 with CRF_WGRAD_DETERMINISTIC=1: fp32 partial tiles
                            * (crf_gemm_workspace_bytes) or NULL.  Not read by any other GEMM. */
  size_t workspace_bytes;
  float* colsum;           /* MN-major A only: colsum[m] += sum_k A(m,k) (bias gradient fused into wgrad), or NULL */
  int32_t split3;          /* 1: split-operand fp32 emulation.  A and B hold fp32 values as two bf16 terms side by side,
                            * [hi | lo] (twice as many columns as the logical matrix: (M, 2K) / (K, 2M) ...), and the
                            * product accumulates hi*hi + hi*lo + lo*hi in fp32.  fp32 epilogues only. */
} crf_gemm_args;
int crf_gemm(const crf_gemm_args* a, void* stream);
/* workspace a CRF_EPI_SPLITK_F32 GEMM of this shape wants (0 when it runs as a single split) */
size_t crf_gemm_workspace_bytes(int M, int N, int K, int device);

/* The MLP half of a block in ONE kernel (C = 128 or 256):  y = x1 + fc2(GELU(fc1(LayerNorm(x1))))
 * (replaces `x + self.mlp(self.norm2(x))`, /root/reference/src/newcrf_layers.py:255, Mlp.forward :21-27).
 * The 4C-wide hidden activation stays on chip between fc1 and fc2 (TMEM -> registers -> shared memory).
 *   x1, y        f32 (T, C) contiguous (y may not alias x1)
 *   w1_bf16      bf16 (4C, C) = fc1.weight;  w2_bf16 bf16 (C, 4C) = fc2.weight;  b1 (4C), b2 (C), norm_w/norm_b (C) f32
 *   training=1   also writes what the backward kernels read: xn2 bf16 (T, C), stats f32 (T, 2) = (mean, rstd),
 *                pre bf16 (T, 4C) (fc1 output + bias), act bf16 (T, 4C) (GELU of it); training=0: those may be NULL */
typedef struct crf_mlp_args {
  const float* x1; float* y;
  const void* w1_bf16; const void* w2_bf16;
  const float* b1; const float* b2; const float* norm_w; const float* norm_b;
  void* xn2; float* stats; void* pre; void* act;
  float eps;
  int32_t T, C, training, device;
} crf_mlp_args;
int crf_mlp_fwd(const crf_mlp_args* a, void* stream);

/* LayerNorm forward over channels with a layout change: x (B, T_img, C) with arbitrary strides ->
 * xn bf16 (T, C), stats f32 (T, 2) = (mean, rstd), optional contiguous f32 copy of x. */
int crf_ln_fwd(const void* x, int x_dtype, int64_t sb, int64_t st, int64_t sc, int B, int T_img, int C,
               const float* gamma, const float* beta, float eps, void* xn_bf16, float* stats, float* x_copy,
               int device, void* stream);
/* LayerNorm backward: dx = LN'(g) + dres; accumulates dgamma/dbeta (+=). g f32 (T,C), x f32 (T,C). */
int crf_ln_bwd(const float* g, const float* x, const float* stats, const float* gamma, const float* dres, float* dx,
               void* dx_bf16, float* dgamma, float* dbeta, int T, int C, int device, void* stream);
/* Input-gradient GEMM of a projection fused with the LayerNorm backward of its input (C = 128 or 256, K % 64 == 0):
 *   g = dy (T, K) * W (K, C);  dx = LN'(g; x, stats, gamma) + dres;  dgamma / dbeta are ACCUMULATED (+=).
 * The backward of `self.norm2(x)` -> fc1 and of `self.norm1(x)` -> qk (/root/reference/src/newcrf_layers.py:208,255)
 * without the fp32 (T, C) gradient of the normalised rows ever reaching HBM.
 *   dy_bf16 bf16 (T, K); w_bf16 bf16 (K, C) = the Linear's weight (out, in); x f32 (T, C); stats f32 (T, 2);
 *   dres f32 (T, C) or NULL; dx f32 (T, C) and / or dx_bf16 bf16 (T, C) (at least one). */
int crf_dgrad_ln_bwd(const void* dy_bf16, const void* w_bf16, int K, const float* x, const float* stats,
                     const float* gamma, const float* dres, float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T,
                     int C, int device, void* stream);
/* Stand-alone LayerNorm over the channels of contiguous token rows: the `norm_crf` that closes a decoder stage
 * (replaces nn.LayerNorm in NewCRF.forward, /root/reference/src/newcrf_layers.py:430-431).
 *   x f32 (T, C) contiguous; y f32 or bf16 (T, C) (y_dtype = CRF_DT_F32 / CRF_DT_BF16: under bf16 autocast the next
 *   consumer is a convolution that would cast anyway); stats f32 (T, 2) = (mean, rstd) for the backward.
 * Backward: g = dL/dy in f32 or bf16; dx f32 (T, C); dgamma / dbeta are ACCUMULATED (+=). */
int crf_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                      float* stats, int T, int C, int device, void* stream);
int crf_layernorm_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                      float* dgamma, float* dbeta, int T, int C, int device, void* stream);
/* The same LayerNorm with the PixelShuffle(2) that follows a decoder stage folded into its store (forward) / load
 * (backward): x, dx f32 (B*H*W, C) token rows; y, g (B, 2H, 2W, C/4) NHWC, y[b, 2h+i, 2w+j, k] = LN(x)[(b,h,w), 4k+2i+j]
 * -- bit-identical to crf_layernorm_fwd followed by crf_pixel_shuffle_nhwc. */
int crf_layernorm_ps_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                         float* stats, int B, int H, int W, int C, int device, void* stream);
int crf_layernorm_ps_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                         float* dgamma, float* dbeta, int B, int H, int W, int C, int device, void* stream);
/* The training loop's loss, 1.0 * SSIM + 0.1 * L1 (replaces /root/reference/src/train.py:94-100 with the SSIM module of
 * /root/reference/src/loss.py:57-88: reflection pad 1, 3x3 average pools, clamp((1 - n/d) / 2, 0, 1), mean).
 *   pred f32 or bf16 (n_img, H, W) contiguous (n_img = batch x channels), target f32, H, W >= 2.
 *   Forward ADDS to sums[0] the sum of the SSIM values and to sums[1] the sum of |pred - target| (caller zeroes them;
 *   loss = (sums[0] + 0.1 * sums[1]) / (n_img * H * W)); if G != NULL it also writes the three f32 maps
 *   (3, n_img, H, W) the backward needs.  Backward: dpred (dtype of pred) = *grad_loss * dloss/dpred, grad_loss a
 *   device scalar. */
int crf_depth_loss_fwd(const void* pred, int pred_dtype, const float* target, int n_img, int H, int W, float* sums,
                       float* G, int device, void* stream);
int crf_depth_loss_bwd(const void* pred, int pred_dtype, const float* target, const float* G, const float* grad_loss,
                       int n_img, int H, int W, void* dpred, int device, void* stream);
/* PixelShuffle(2) between decoder stages (replaces nn.PixelShuffle(2),
 * /root/reference/src/model_mobileV3_large_newCRFs.py:116-120) on channels-last memory, f32 or bf16:
 *   inverse == 0: src (B, H, W, C) -> dst (B, 2H, 2W, C/4), dst[b, 2h+i, 2w+j, c] = src[b, h, w, 4c + 2i + j]
 *   inverse != 0: src (B, 2H, 2W, C/4) -> dst (B, H, W, C)   (pixel_unshuffle: the backward)
 * B, H, W, C always describe the (B, H, W, C) side; C % 4 == 0. */
int crf_pixel_shuffle_nhwc(const void* src, void* dst, int dtype, int B, int H, int W, int C, int inverse, int device,
                           void* stream);
/* One Adam step over many fp32 tensors (replaces torch.optim.Adam.step of the reference loop,
 * /root/reference/src/train.py:41,108; no amsgrad; weight_decay is torch's L2 form, 0 in the reference).
 *   tensors  HOST array of n_tensors records (device pointers inside); passed to the kernels as launch arguments,
 *            80 tensors per launch, so nothing has to stay alive after the call
 *   chunk_elems  elements one CTA updates (multiple of 4, >= 1024; 16384 is a good value)
 *   step     DEVICE float: number of steps taken so far; the update uses step + 1 and the call then increments it
 *            (so a CUDA graph that captured the call keeps counting on replay)
 * Hyper-parameters are doubles (torch keeps them as Python floats and derives 1 - beta, the bias corrections and
 * lr / bc1 in double before rounding once to fp32; ABI version 2 changed them from float). */
typedef struct crf_adam_tensor {
  float* p;        /* parameter, updated in place */
  const float* g;  /* gradient */
  float* m;        /* exp_avg, updated in place */
  float* v;        /* exp_avg_sq, updated in place */
  int64_t n;       /* elements */
} crf_adam_tensor;
int crf_adam_step(const crf_adam_tensor* tensors, int n_tensors, int chunk_elems, double lr, double beta1, double beta2,
                  double eps, double weight_decay, float* step, int device, void* stream);
/* out[n] += sum_t g[t, n], g bf16 (T, N) contiguous, N % 4 == 0 */
int crf_colsum_bf16(const void* g, float* out, int T, int N, int device, void* stream);
/* f32 -> bf16 contiguous */
int crf_cast_bf16(const float* src, void* dst, int64_t n, int device, void* stream);

/* Training-mode BatchNorm2d + activation over a channels-last bf16 map x, viewed as (T, C) rows (T = B H W >= 2,
 * C % 8 == 0), two kernels each way.  Results follow torch's act(F.batch_norm(x, ..., training=True)) with fp32
 * parameters: the BN output is rounded to bf16 before the activation; only the fp32 summation order differs.
 *   crf_bn_fwd: y = act(bf16(w (x - mean) invstd + b)) (bf16, like x); writes save_mean / save_invstd (fp32, C), updates
 *     running_mean / running_var (unbiased variance) with `momentum` and adds 1 to the int64 num_batches_tracked.
 *   crf_bn_bwd: dx (bf16) from dy (bf16) and the saved statistics, with the BN output recomputed from x; writes
 *     dweight / dbias (fp32, C).
 * workspace: at least crf_bn_workspace_bytes(T, C, device) bytes, 16-byte aligned, contents don't-care.  tickets: at
 * least C / 8 int32 counters, zero before the first call; every call leaves them zero again (CUDA-graph replay safe).
 * One tickets buffer must not serve two calls in flight at once.  x, y, dy, dx: 16-byte aligned, row-contiguous. */
#define CRF_ACT_NONE 0
#define CRF_ACT_RELU 1
#define CRF_ACT_HARDSWISH 2
size_t crf_bn_workspace_bytes(int T, int C, int device);
int crf_bn_fwd(const void* x, void* y, const float* weight, const float* bias, float* running_mean, float* running_var,
               long long* num_batches_tracked, float* save_mean, float* save_invstd, int T, int C, float eps,
               float momentum, int act, void* workspace, size_t workspace_bytes, int* tickets, int device, void* stream);
int crf_bn_bwd(const void* x, const void* dy, const float* weight, const float* bias, const float* save_mean,
               const float* save_invstd, void* dx, float* dweight, float* dbias, int T, int C, int act, void* workspace,
               size_t workspace_bytes, int* tickets, int device, void* stream);

/* Depthwise convolution nn.Conv2d(C, C, k, stride, padding=k // 2, groups=C, bias=False) over a channels-last bf16 map
 * x viewed as (B, H, W, C), k = 3 or 5, stride = 1 or 2, C % 8 == 0; the output is (B, Ho, Wo, C) with
 * Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1.  Results follow torch's conv2d under bf16 autocast: the fp32
 * weight (C, 1, k, k), contiguous, is rounded to bf16 on load; only the fp32 summation order differs.  No atomics: every
 * result is bit-reproducible from run to run.
 *   crf_dwconv_fwd: y (bf16): each output one fp32 sum of bf16 products in a fixed tap order, rounded once.
 *   crf_dwconv_bwd: dx (bf16, like x) and dweight (fp32 (C, 1, k, k), contiguous: summed in fp32 partials and double,
 *     rounded to bf16 and widened, as cuDNN's bf16 weight gradient cast back to fp32) from dy (bf16, like y).  Either
 *     of dx and dweight may be NULL when that gradient is not needed; workspace and tickets serve dweight only.
 * workspace: at least crf_dwconv_workspace_bytes(B, H, W, C, k, stride, device) bytes, 16-byte aligned, contents
 * don't-care.  tickets: at least k * C / 8 int32 counters, zero before the first call; every call leaves them zero
 * again (CUDA-graph replay safe).  One tickets buffer must not serve two calls in flight at once.  x, y, dy, dx: 16-byte
 * aligned, contiguous. */
size_t crf_dwconv_workspace_bytes(int B, int H, int W, int C, int k, int stride, int device);
int crf_dwconv_fwd(const void* x, const float* weight, void* y, int B, int H, int W, int C, int k, int stride, int device,
                   void* stream);
int crf_dwconv_bwd(const void* x, const float* weight, const void* dy, void* dx, float* dweight, int B, int H, int W,
                   int C, int k, int stride, void* workspace, size_t workspace_bytes, int* tickets, int device,
                   void* stream);

/* Window-attention core (everything between the qk projection and the output projection).
 *   qk   bf16 (T, 2C): q already multiplied by scale (cols [0,C)), k (cols [C,2C))
 *   vb   bf16 (T, C)
 *   o    bf16 (T, C)   attention output in token order (window_reverse + un-roll + crop applied)
 *   lse  f32 (B*nW, nH, 64) row log-sum-exp (saved for backward)
 *   qk_bias f32 (2C): q/k of zero-padded tokens are their bias (newcrf_layers.py:215,118) */
/*   mask  optional additive mask f32 (mask_windows, N, N), N = window^2, applied to window (global index % mask_windows), as
 *         WindowAttention.forward's `mask` argument (newcrf_layers.py:129-133); NULL / 0 for none */
int crf_attn_fwd(const crf_block_desc* d, const void* qk, const void* vb, const float* qk_bias, float scale,
                 const float* rpb_table, const float* mask, int mask_windows, void* o, float* lse, void* stream);
/*   dout bf16 (T, C); dqk bf16 (T, 2C) (dq includes the scale factor); dv f32 (T, C) (= or +=);
 *   d_table f32 ((2w-1)^2, nH) +=;  d_qk_bias f32 (2C) += (only the k half receives pad-token gradient) */
int crf_attn_bwd(const crf_block_desc* d, const void* qk, const void* vb, const float* qk_bias, float scale,
                 const float* rpb_table, const float* mask, int mask_windows, const float* lse, const void* dout,
                 void* dqk, float* dv, int dv_accumulate, float* d_table, float* d_qk_bias, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CRF_SM100_H_ */
