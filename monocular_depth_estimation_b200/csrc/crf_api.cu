// extern "C" entry points of libcrf_sm100.so (see include/crf_sm100.h) and the per-block orchestration:
// which kernels run, in what order, on which slices of the caller-provided `saved` / workspace buffers.
#include "crf_host.h"
#include "crf_window.cuh"

namespace crf {
namespace {

inline size_t align_up(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

// Layout of the `saved` buffer (forward products backward needs) -- offsets in bytes.
struct SavedLayout {
  size_t xc, stats1, xn1, qk, vb, lse, attn_o, x1, stats2, xn2, pre, act, wb_qk, wb_proj, wb_fc1, wb_fc2, total;
};
// Layout of the backward workspace.
struct BwdLayout {
  size_t dyb, dhpre, dxn, dx1, dx1b, dob, dqk, partials, partials_bytes, total;
};

// v already is what the attention kernels read: bf16 rows, token-major, contiguous (the channels-last output of the
// proj_v convolution under bf16 autocast) -- the layer then uses it in place instead of making the bf16 copy
bool v_is_token_major_bf16(const crf_block_desc& d) {
  return d.v_dtype == CRF_DT_BF16 && d.v_stride_c == 1 && d.v_stride_w == d.C &&
         d.v_stride_h == static_cast<int64_t>(d.W) * d.C && d.v_stride_b == static_cast<int64_t>(d.H) * d.W * d.C;
}

bool x_is_plain(const crf_block_desc& d) {
  const int64_t T_img = static_cast<int64_t>(d.H) * d.W;
  return d.x_dtype == CRF_DT_F32 && d.x_stride_c == 1 && d.x_stride_t == d.C && d.x_stride_b == T_img * d.C;
}

SavedLayout saved_layout(const crf_block_desc& d) {
  const size_t T = static_cast<size_t>(d.B) * d.H * d.W;
  const size_t C = d.C;
  WindowGeom gm(d.H, d.W, d.window, d.shift);
  SavedLayout L{};
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
  L.xc = take(x_is_plain(d) ? 0 : T * C * 4);
  L.stats1 = take(T * 2 * 4);
  L.xn1 = take(T * C * 2);
  L.qk = take(T * 2 * C * 2);
  L.vb = take(d.v_preconverted ? 0 : T * C * 2);
  L.lse = take(static_cast<size_t>(d.B) * gm.nW * d.num_heads * 64 * 4);
  L.attn_o = take(T * C * 2);
  L.x1 = take(T * C * 4);
  L.stats2 = take(T * 2 * 4);
  L.xn2 = take(T * C * 2);
  L.pre = take(d.training ? T * 4 * C * 2 : 0);
  L.act = take(T * 4 * C * 2);
  L.wb_qk = take(2 * C * C * 2);
  L.wb_proj = take(C * C * 2);
  L.wb_fc1 = take(4 * C * C * 2);
  L.wb_fc2 = take(4 * C * C * 2);
  L.total = o;
  return L;
}

BwdLayout bwd_layout(const crf_block_desc& d) {
  const size_t T = static_cast<size_t>(d.B) * d.H * d.W;
  const size_t C = d.C;
  BwdLayout L{};
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
  L.dyb = take(T * C * 2);
  L.dhpre = take(T * 4 * C * 2);
  L.dxn = take(T * C * 4);
  L.dx1 = take(T * C * 4);
  L.dx1b = take(T * C * 2);
  L.dob = take(T * C * 2);
  L.dqk = take(T * 2 * C * 2);
  // split-K partial tiles of the four weight-gradient GEMMs (used one after the other)
  const int Ti = static_cast<int>(T), Ci = d.C;
  size_t pb = 0;
  const int shapes[4][2] = {{Ci, 4 * Ci}, {4 * Ci, Ci}, {Ci, Ci}, {2 * Ci, Ci}};
  for (auto& s : shapes) {
    const size_t b = gemm_splitk_workspace_bytes(s[0], s[1], Ti, d.device, nullptr);
    if (b > pb) pb = b;
  }
  L.partials_bytes = pb;
  L.partials = take(pb);
  L.total = o;
  return L;
}

int check_desc(const crf_block_desc* d) {
  CRF_CHECK(d != nullptr, "null descriptor");
  CRF_CHECK(d->B > 0 && d->H > 0 && d->W > 0, "empty input (B=%d H=%d W=%d)", d->B, d->H, d->W);
  CRF_CHECK(d->C % 64 == 0 && d->C >= 64 && d->C <= 1024, "C=%d must be a multiple of 64 in [64,1024]", d->C);
  CRF_CHECK(d->num_heads > 0 && d->C % d->num_heads == 0 && head_dim_supported(d->C / d->num_heads),
            "head_dim must be 16, 32, 64 or 128 (C=%d, heads=%d)", d->C, d->num_heads);
  CRF_CHECK(d->window >= kMinWindow && d->window <= kMaxWindow, "window must be in [%d, %d] (got %d)", kMinWindow,
            kMaxWindow, d->window);
  CRF_CHECK(d->shift >= 0 && d->shift < d->window, "shift_size must in 0-window_size");
  CRF_CHECK(static_cast<int64_t>(d->B) * d->H * d->W * 4 * d->C < (int64_t(1) << 31) * 4,
            "problem too large for 32-bit token indexing");
  return 0;
}

int gemm_fprop(const void* A, const void* W, int M, int N, int K, int epi, void* out0, void* out1, const float* bias,
               const void* aux1, float scale, int scale_cols, int device, cudaStream_t st) {
  crf_gemm_args a{};
  a.A = A; a.B = W; a.a_major = 0; a.b_major = 0;
  a.M = M; a.N = N; a.K = K; a.epilogue = epi; a.split_k = 1;
  a.out0 = out0; a.out1 = out1; a.bias = bias; a.aux1 = aux1; a.ld_out = N;
  a.scale = scale; a.scale_cols = scale_cols; a.device = device;
  return launch_gemm(a, st);
}
// dX[M=T, N=Cin] = dY[T, K=Cout] * W[Cout, Cin]
int gemm_dgrad(const void* dY, const void* W, int M, int N, int K, int epi, void* out0, const void* aux1, int device,
               cudaStream_t st) {
  crf_gemm_args a{};
  a.A = dY; a.B = W; a.a_major = 0; a.b_major = 1;
  a.M = M; a.N = N; a.K = K; a.epilogue = epi; a.split_k = 1;
  a.out0 = out0; a.aux1 = aux1; a.ld_out = N; a.scale = 1.f; a.scale_cols = 0; a.device = device;
  return launch_gemm(a, st);
}
// dW[M=Cout, N=Cin] += dY[T, Cout]^T * X[T, Cin]
int gemm_wgrad(const void* dY, const void* X, int M, int N, int K, float* dW, float* db, void* ws, size_t ws_bytes,
               int device, cudaStream_t st) {
  crf_gemm_args a{};
  a.A = dY; a.B = X; a.a_major = 1; a.b_major = 1;
  a.M = M; a.N = N; a.K = K; a.epilogue = CRF_EPI_SPLITK_F32; a.split_k = 0;
  a.out0 = dW; a.ld_out = N; a.scale = 1.f; a.device = device;
  a.workspace = ws; a.workspace_bytes = ws_bytes;
  a.colsum = db;  // bias gradient = column sums of dY, computed by the same kernel
  return launch_gemm(a, st);
}

}  // namespace
}  // namespace crf

using namespace crf;

extern "C" {

const char* crf_last_error(void) { return get_error(); }
int crf_abi_version(void) { return CRF_ABI_VERSION; }
long long crf_kernel_launches(void) { return launch_count(); }
int crf_timing_enable(int on) { timing_enable(on != 0); return 0; }
size_t crf_timing_report(char* buf, size_t cap) { return timing_report(buf, cap); }

int crf_block_sizes(const crf_block_desc* d, size_t* saved_bytes, size_t* ws_fwd_bytes, size_t* ws_bwd_bytes) {
  if (check_desc(d)) return 1;
  const bool fp32 = d->precision == CRF_PREC_FP32;
  if (saved_bytes) *saved_bytes = fp32 ? precise_saved_bytes(*d) : saved_layout(*d).total;
  if (ws_fwd_bytes) *ws_fwd_bytes = 256;  // forward needs no scratch beyond `saved`
  if (ws_bwd_bytes) *ws_bwd_bytes = fp32 ? precise_bwd_bytes(*d) : bwd_layout(*d).total;
  return 0;
}

int crf_convert_v(const crf_block_desc* d, const void* v, void* v_bf16, void* stream) {
  if (check_desc(d)) return 1;
  CRF_CHECK(v != nullptr && v_bf16 != nullptr, "crf_convert_v: null pointer");
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  CRF_CHECK(d->v_stride_h == static_cast<int64_t>(d->W) * d->v_stride_w,
            "crf_convert_v: v must be collapsible over (H, W): stride_h=%lld stride_w=%lld W=%d",
            (long long)d->v_stride_h, (long long)d->v_stride_w, d->W);
  return launch_convert_tokens(v, d->v_dtype, d->v_stride_b, d->v_stride_w, d->v_stride_c, d->B, d->H * d->W, d->C,
                               v_bf16, static_cast<cudaStream_t>(stream));
}

static int block_fwd_impl(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, float* y,
                          void* saved, void* stream) {
  if (check_desc(d)) return 1;
  CRF_CHECK(p && x && v && y && saved, "crf_block_fwd: null pointer");
  CRF_CHECK(p->ext_mask == nullptr || p->ext_mask_windows > 0, "crf_block_fwd: ext_mask needs ext_mask_windows > 0");
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d->precision == CRF_PREC_FP32) return block_fwd_precise(d, p, x, v, y, saved, st);
  const SavedLayout L = saved_layout(*d);
  uint8_t* S = static_cast<uint8_t*>(saved);
  const int T = d->B * d->H * d->W, C = d->C;
  const bool plain = x_is_plain(*d);

  // bf16 operand copies of the four weight matrices (kept in `saved`: backward reuses them)
  {
    const float* const src[4] = {p->qk_w, p->proj_w, p->fc1_w, p->fc2_w};
    void* const dst[4] = {S + L.wb_qk, S + L.wb_proj, S + L.wb_fc1, S + L.wb_fc2};
    const long long n[4] = {2LL * C * C, 1LL * C * C, 4LL * C * C, 4LL * C * C};
    if (launch_cast4_bf16(src, dst, n, st)) return 1;
  }

  // LN1 (+ layout change of the NCHW view into token-major rows)
  float* xc = plain ? nullptr : reinterpret_cast<float*>(S + L.xc);
  if (launch_ln_fwd(x, d->x_dtype, d->x_stride_b, d->x_stride_t, d->x_stride_c, d->B, d->H * d->W, C, p->norm1_w,
                    p->norm1_b, p->ln_eps, S + L.xn1, reinterpret_cast<float*>(S + L.stats1), xc, st))
    return 1;
  const float* x_tok = plain ? static_cast<const float*>(x) : xc;

  const void* vb = v;
  if (!d->v_preconverted) {
    if (crf_convert_v(d, v, S + L.vb, stream)) return 1;
    vb = S + L.vb;
  }
  // q (scaled) and k
  if (gemm_fprop(S + L.xn1, S + L.wb_qk, T, 2 * C, C, CRF_EPI_STORE_BF16, S + L.qk, nullptr, p->qk_b, nullptr,
                 p->qk_scale, C, d->device, st))
    return 1;
  // window attention core
  if (launch_attn_fwd(*d, S + L.qk, vb, p->qk_b, p->qk_scale, p->rpb_table, p->ext_mask, p->ext_mask_windows,
                      S + L.attn_o, d->training ? reinterpret_cast<float*>(S + L.lse) : nullptr, st, /*ext_replaces=*/1))
    return 1;
  // x1 = x + proj(attn)
  if (gemm_fprop(S + L.attn_o, S + L.wb_proj, T, C, C, CRF_EPI_BIAS_RES_F32, S + L.x1, nullptr, p->proj_b, x_tok, 1.f,
                 0, d->device, st))
    return 1;
  // LN2 + MLP + residual in one kernel where the fused kernel exists (C = 128, 256), else the three kernels below
  if (mlp_fused_supported(C)) {
    crf_mlp_args m{};
    m.x1 = reinterpret_cast<const float*>(S + L.x1); m.y = y;
    m.w1_bf16 = S + L.wb_fc1; m.w2_bf16 = S + L.wb_fc2;
    m.b1 = p->fc1_b; m.b2 = p->fc2_b; m.norm_w = p->norm2_w; m.norm_b = p->norm2_b;
    m.xn2 = S + L.xn2; m.stats = reinterpret_cast<float*>(S + L.stats2);
    m.pre = d->training ? S + L.pre : nullptr; m.act = S + L.act;
    m.eps = p->ln_eps; m.T = T; m.C = C; m.training = d->training; m.device = d->device;
    return launch_mlp_fused_fwd(m, st);
  }
  // LN2
  if (launch_ln_fwd(S + L.x1, CRF_DT_F32, static_cast<int64_t>(d->H) * d->W * C, C, 1, d->B, d->H * d->W, C,
                    p->norm2_w, p->norm2_b, p->ln_eps, S + L.xn2, reinterpret_cast<float*>(S + L.stats2), nullptr, st))
    return 1;
  // MLP
  if (gemm_fprop(S + L.xn2, S + L.wb_fc1, T, 4 * C, C, CRF_EPI_BIAS_GELU, d->training ? S + L.pre : nullptr, S + L.act,
                 p->fc1_b, nullptr, 1.f, 0, d->device, st))
    return 1;
  if (gemm_fprop(S + L.act, S + L.wb_fc2, T, C, 4 * C, CRF_EPI_BIAS_RES_F32, y, nullptr, p->fc2_b, S + L.x1, 1.f, 0,
                 d->device, st))
    return 1;
  return 0;
}

// dy_bf16: optional bf16 twin of dy (saves the cast); dx_bf16: optional bf16 twin of dx to write.
static int block_bwd_impl(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v,
                          const float* dy, const void* dy_bf16, const void* saved, float* dx, void* dx_bf16, float* dv,
                          int dv_accumulate, const crf_block_grads* g, void* ws, size_t ws_bytes, void* stream) {
  if (check_desc(d)) return 1;
  CRF_CHECK(p && x && v && dy && saved && (dx || dx_bf16) && dv && g && ws, "crf_block_bwd: null pointer");
  CRF_CHECK(d->training, "crf_block_bwd: forward was not run with training=1");
  if (d->precision == CRF_PREC_FP32) {
    DeviceGuard guard(d->device);
    CRF_CHECK(guard.ok, "cannot select device %d", d->device);
    return block_bwd_precise(d, p, x, v, dy, saved, dx, dx_bf16, dv, dv_accumulate, g, ws, ws_bytes,
                             static_cast<cudaStream_t>(stream));
  }
  const BwdLayout W = bwd_layout(*d);
  CRF_CHECK(ws_bytes >= W.total, "crf_block_bwd: workspace too small (%zu < %zu)", ws_bytes, W.total);
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const SavedLayout L = saved_layout(*d);
  const uint8_t* S = static_cast<const uint8_t*>(saved);
  uint8_t* Wk = static_cast<uint8_t*>(ws);
  const int T = d->B * d->H * d->W, C = d->C, dev = d->device;
  const bool plain = x_is_plain(*d);
  const float* x_tok = plain ? static_cast<const float*>(x) : reinterpret_cast<const float*>(S + L.xc);
  const void* vb = d->v_preconverted ? v : static_cast<const void*>(S + L.vb);
  float* dxn = reinterpret_cast<float*>(Wk + W.dxn);
  float* dx1 = reinterpret_cast<float*>(Wk + W.dx1);

  // ---- MLP ----
  const void* dyb = dy_bf16;
  if (dyb == nullptr) {
    if (launch_cast_bf16(dy, Wk + W.dyb, static_cast<int64_t>(T) * C, st)) return 1;
    dyb = Wk + W.dyb;
  }
  if (gemm_dgrad(dyb, S + L.wb_fc2, T, 4 * C, C, CRF_EPI_MUL_DGELU, Wk + W.dhpre, S + L.pre, dev, st)) return 1;
  if (gemm_wgrad(dyb, S + L.act, C, 4 * C, T, g->fc2_w, g->fc2_b, Wk + W.partials, W.partials_bytes, dev, st)) return 1;
  const bool fuse_ln = dgrad_lnbwd_supported(C, 2 * C);
  if (fuse_ln) {  // dx1 = dy + LN2'(dhpre W1) straight from the GEMM's accumulator rows
    if (launch_dgrad_lnbwd(Wk + W.dhpre, S + L.wb_fc1, 4 * C, reinterpret_cast<const float*>(S + L.x1),
                           reinterpret_cast<const float*>(S + L.stats2), p->norm2_w, dy, dx1, Wk + W.dx1b, g->norm2_w,
                           g->norm2_b, T, C, dev, st))
      return 1;
  } else {
    if (gemm_dgrad(Wk + W.dhpre, S + L.wb_fc1, T, C, 4 * C, CRF_EPI_STORE_F32, dxn, nullptr, dev, st)) return 1;
  }
  if (gemm_wgrad(Wk + W.dhpre, S + L.xn2, 4 * C, C, T, g->fc1_w, g->fc1_b, Wk + W.partials, W.partials_bytes, dev, st)) return 1;
  if (!fuse_ln &&
      launch_ln_bwd(dxn, reinterpret_cast<const float*>(S + L.x1), reinterpret_cast<const float*>(S + L.stats2),
                    p->norm2_w, dy, dx1, Wk + W.dx1b, g->norm2_w, g->norm2_b, T, C, st))
    return 1;
  // ---- attention ----
  if (gemm_dgrad(Wk + W.dx1b, S + L.wb_proj, T, C, C, CRF_EPI_STORE_BF16, Wk + W.dob, nullptr, dev, st)) return 1;
  if (gemm_wgrad(Wk + W.dx1b, S + L.attn_o, C, C, T, g->proj_w, g->proj_b, Wk + W.partials, W.partials_bytes, dev, st)) return 1;
  if (launch_attn_bwd(*d, S + L.qk, vb, p->qk_b, p->qk_scale, p->rpb_table, p->ext_mask, p->ext_mask_windows,
                      reinterpret_cast<const float*>(S + L.lse),
                      Wk + W.dob, Wk + W.dqk, dv, dv_accumulate, g->rpb_table, g->qk_b, st, /*ext_replaces=*/1))
    return 1;
  if (fuse_ln) {  // dx = dx1 + LN1'(dqk Wqk)
    if (launch_dgrad_lnbwd(Wk + W.dqk, S + L.wb_qk, 2 * C, x_tok, reinterpret_cast<const float*>(S + L.stats1), p->norm1_w,
                           dx1, dx, dx_bf16, g->norm1_w, g->norm1_b, T, C, dev, st))
      return 1;
  } else {
    if (gemm_dgrad(Wk + W.dqk, S + L.wb_qk, T, C, 2 * C, CRF_EPI_STORE_F32, dxn, nullptr, dev, st)) return 1;
  }
  if (gemm_wgrad(Wk + W.dqk, S + L.xn1, 2 * C, C, T, g->qk_w, g->qk_b, Wk + W.partials, W.partials_bytes, dev, st)) return 1;
  if (!fuse_ln &&
      launch_ln_bwd(dxn, x_tok, reinterpret_cast<const float*>(S + L.stats1), p->norm1_w, dx1, dx, dx_bf16,
                    g->norm1_w, g->norm1_b, T, C, st))
    return 1;
  return 0;
}

int crf_block_fwd(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, float* y,
                  void* saved, void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;
  return block_fwd_impl(d, p, x, v, y, saved, stream);
}

int crf_block_bwd(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, const float* dy,
                  const void* saved, float* dx, float* dv, int dv_accumulate, const crf_block_grads* g, void* ws,
                  size_t ws_bytes, void* stream) {
  return block_bwd_impl(d, p, x, v, dy, nullptr, saved, dx, nullptr, dv, dv_accumulate, g, ws, ws_bytes, stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// Layer level: BasicCRFLayer.forward (newcrf_layers.py:323-363: `depth` blocks, shift 0 / window/2 alternating, the
// same v for every block) plus, optionally, the LayerNorm that closes the decoder stage (NewCRF.norm_crf, :430-431).
// ---------------------------------------------------------------------------------------------------------------------
namespace {
struct LayerLayout {
  size_t vb, norm_stats, total;
  size_t blk[CRF_MAX_DEPTH], yout[CRF_MAX_DEPTH];  // per block: its `saved` area and its fp32 output (T, C)
};
crf_block_desc block_desc_of(const crf_block_desc& d, int i) {
  crf_block_desc b = d;
  b.shift = (i % 2 == 0) ? 0 : d.window / 2;
  b.v_preconverted = d.precision == CRF_PREC_FP32 ? 0 : 1;  // the fp32 mode reads v as it is, with its own strides
  if (i > 0) {  // blocks after the first read the previous block's contiguous fp32 output
    b.x_dtype = CRF_DT_F32;
    b.x_stride_c = 1;
    b.x_stride_t = d.C;
    b.x_stride_b = static_cast<int64_t>(d.H) * d.W * d.C;
  }
  return b;
}
LayerLayout layer_layout(const crf_block_desc& d, int depth, int with_norm) {
  LayerLayout L{};
  const size_t T = static_cast<size_t>(d.B) * d.H * d.W, C = d.C;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
  const bool fp32 = d.precision == CRF_PREC_FP32;
  L.vb = take(fp32 ? 0 : T * C * 2);
  for (int i = 0; i < depth; ++i) {
    L.blk[i] = take(fp32 ? precise_saved_bytes(block_desc_of(d, i)) : saved_layout(block_desc_of(d, i)).total);
    // the last block's output is the caller's y unless a closing norm follows (then LN backward needs it)
    L.yout[i] = (i + 1 < depth || with_norm) ? take(T * C * 4) : 0;
  }
  L.norm_stats = take(with_norm ? T * 2 * 4 : 0);
  L.total = o;
  return L;
}
struct LayerBwdLayout {
  size_t blk, g_f32, g_bf16, mid_f32[2], mid_bf16[2], total;
};
LayerBwdLayout layer_bwd_layout(const crf_block_desc& d, int depth, int with_norm) {
  LayerBwdLayout L{};
  const size_t T = static_cast<size_t>(d.B) * d.H * d.W, C = d.C;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
  L.blk = take(d.precision == CRF_PREC_FP32 ? precise_bwd_bytes(block_desc_of(d, depth > 1 ? 1 : 0))
                                            : bwd_layout(block_desc_of(d, depth > 1 ? 1 : 0)).total);
  L.g_f32 = take(with_norm ? T * C * 4 : 0);
  L.g_bf16 = take(with_norm ? T * C * 2 : 0);
  for (int k = 0; k < 2; ++k) {  // ping-pong buffers for the gradient between blocks (each slot aligned on its own)
    L.mid_f32[k] = take(depth > 1 ? T * C * 4 : 0);
    L.mid_bf16[k] = take(depth > 1 ? T * C * 2 : 0);
  }
  L.total = o;
  return L;
}
int check_layer(const crf_block_desc* d, const crf_layer_args* a) {
  if (check_desc(d)) return 1;
  CRF_CHECK(a != nullptr && a->params != nullptr, "crf_layer: null arguments");
  CRF_CHECK(a->depth >= 1 && a->depth <= CRF_MAX_DEPTH, "crf_layer: depth %d not in [1, %d]", a->depth, CRF_MAX_DEPTH);
  CRF_CHECK((a->norm_w == nullptr) == (a->norm_b == nullptr), "crf_layer: norm_w and norm_b go together");
  CRF_CHECK(a->out_dtype == CRF_DT_F32 || (a->out_dtype == CRF_DT_BF16 && a->norm_w != nullptr),
            "crf_layer: bf16 output needs the closing LayerNorm");
  CRF_CHECK(a->out_shuffle == 0 || (a->out_shuffle == 1 && a->norm_w != nullptr && d->C % 4 == 0),
            "crf_layer: out_shuffle needs the closing LayerNorm");
  return 0;
}
}  // namespace

int crf_layer_sizes(const crf_block_desc* d, int depth, int with_norm, size_t* saved_bytes, size_t* ws_bwd_bytes) {
  if (check_desc(d)) return 1;
  CRF_CHECK(depth >= 1 && depth <= CRF_MAX_DEPTH, "crf_layer: depth %d not in [1, %d]", depth, CRF_MAX_DEPTH);
  if (saved_bytes) *saved_bytes = layer_layout(*d, depth, with_norm).total;
  if (ws_bwd_bytes) *ws_bwd_bytes = layer_bwd_layout(*d, depth, with_norm).total;
  return 0;
}

int crf_layer_fwd(const crf_block_desc* d, const crf_layer_args* a, const void* x, const void* v, void* y, void* saved,
                  void* stream) {
  if (check_layer(d, a)) return 1;
  CRF_CHECK(x && v && y && saved, "crf_layer_fwd: null pointer");
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  const int with_norm = a->norm_w != nullptr;
  const LayerLayout L = layer_layout(*d, a->depth, with_norm);
  uint8_t* S = static_cast<uint8_t*>(saved);
  const int T = d->B * d->H * d->W;
  const bool fp32 = d->precision == CRF_PREC_FP32;
  const void* vin = v;
  if (!fp32 && !v_is_token_major_bf16(*d)) {
    crf_block_desc d0 = *d;
    d0.v_preconverted = 0;
    if (crf_convert_v(&d0, v, S + L.vb, stream)) return 1;
    vin = S + L.vb;
  }
  const void* xin = x;
  for (int i = 0; i < a->depth; ++i) {
    const crf_block_desc bd = block_desc_of(*d, i);
    float* yo = (i + 1 == a->depth && !with_norm) ? static_cast<float*>(y) : reinterpret_cast<float*>(S + L.yout[i]);
    if (block_fwd_impl(&bd, a->params + i, xin, vin, yo, S + L.blk[i], stream)) return 1;
    xin = yo;
  }
  if (with_norm && launch_layernorm_fwd(static_cast<const float*>(xin), a->norm_w, a->norm_b, a->params[0].ln_eps, y,
                                        a->out_dtype, reinterpret_cast<float*>(S + L.norm_stats), T, d->C,
                                        static_cast<cudaStream_t>(stream), a->out_shuffle ? d->W : 0))
    return 1;
  return 0;
}

int crf_layer_bwd(const crf_block_desc* d, const crf_layer_args* a, const void* x, const void* v, const void* dy,
                  const void* saved, void* dx, float* dv, const crf_block_grads* g, float* dnorm_w, float* dnorm_b,
                  void* ws, size_t ws_bytes, void* stream) {
  if (check_layer(d, a)) return 1;
  CRF_CHECK(x && dy && saved && dx && dv && g && ws, "crf_layer_bwd: null pointer");
  CRF_CHECK((d->precision != CRF_PREC_FP32 && !v_is_token_major_bf16(*d)) || v != nullptr,
            "crf_layer_bwd: the fp32 mode, and a bf16 token-major v (used in place), re-read v");
  CRF_CHECK(d->training, "crf_layer_bwd: forward was not run with training=1");
  const int with_norm = a->norm_w != nullptr;
  CRF_CHECK(!with_norm || (dnorm_w && dnorm_b), "crf_layer_bwd: gradient buffers of the closing norm are missing");
  const LayerLayout L = layer_layout(*d, a->depth, with_norm);
  const LayerBwdLayout W = layer_bwd_layout(*d, a->depth, with_norm);
  CRF_CHECK(ws_bytes >= W.total, "crf_layer_bwd: workspace too small (%zu < %zu)", ws_bytes, W.total);
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint8_t* S = static_cast<const uint8_t*>(saved);
  uint8_t* Wk = static_cast<uint8_t*>(ws);
  const size_t T = static_cast<size_t>(d->B) * d->H * d->W;

  // gradient entering the last block: fp32 + bf16 twin
  const float* g32 = static_cast<const float*>(dy);
  const void* g16 = nullptr;
  if (with_norm) {
    const float* ylast = reinterpret_cast<const float*>(S + L.yout[a->depth - 1]);
    float* gn = reinterpret_cast<float*>(Wk + W.g_f32);
    const float* stats = reinterpret_cast<const float*>(S + L.norm_stats);
    // LayerNorm backward writes dx in fp32 and its bf16 twin in one pass (the MLP GEMMs read the twin)
    if (a->out_dtype == CRF_DT_F32 && !a->out_shuffle) {
      if (launch_ln_bwd(static_cast<const float*>(dy), ylast, stats, a->norm_w, nullptr, gn, Wk + W.g_bf16, dnorm_w,
                        dnorm_b, static_cast<int>(T), d->C, st))
        return 1;
    } else if (launch_layernorm_bwd(dy, a->out_dtype, ylast, stats, a->norm_w, gn, Wk + W.g_bf16, dnorm_w, dnorm_b,
                                    static_cast<int>(T), d->C, st, a->out_shuffle ? d->W : 0)) {
      return 1;
    }
    g32 = gn;
    g16 = Wk + W.g_bf16;
  }
  for (int i = a->depth - 1; i >= 0; --i) {
    const crf_block_desc bd = block_desc_of(*d, i);
    const void* xin = i == 0 ? x : static_cast<const void*>(S + L.yout[i - 1]);
    // the layer's dx leaves in the dtype of x: bf16 inputs get a bf16 gradient straight from the LayerNorm backward
    const bool dx_is_bf16 = d->x_dtype == CRF_DT_BF16;
    float* dxo = i == 0 ? (dx_is_bf16 ? nullptr : static_cast<float*>(dx))
                        : reinterpret_cast<float*>(Wk + W.mid_f32[i & 1]);
    void* dxo16 = i == 0 ? (dx_is_bf16 ? dx : nullptr)
                         : static_cast<void*>(Wk + W.mid_bf16[i & 1]);
    const bool fp32 = d->precision == CRF_PREC_FP32;
    const void* vin = (fp32 || v_is_token_major_bf16(*d)) ? v : static_cast<const void*>(S + L.vb);
    if (block_bwd_impl(&bd, a->params + i, xin, vin, g32, g16, S + L.blk[i], dxo,
                       dxo16, dv, i == a->depth - 1 ? 0 : 1, g + i, Wk + W.blk,
                       fp32 ? precise_bwd_bytes(bd) : bwd_layout(bd).total, stream))
      return 1;
    g32 = dxo;
    g16 = dxo16;
  }
  return 0;
}

int crf_window_gather(const float* x, float* windows, int B, int H, int W, int C, int window, int shift,
                      void* stream) {
  CRF_CHECK(x && windows && B > 0 && H > 0 && W > 0 && C > 0 && window > 0, "crf_window_gather: bad arguments");
  CRF_CHECK(shift >= 0 && shift < window, "shift_size must in 0-window_size");
  return launch_window_gather(x, windows, B, H, W, C, window, shift, static_cast<cudaStream_t>(stream));
}
int crf_window_scatter(const float* windows, float* x, int B, int H, int W, int C, int window, int shift,
                       void* stream) {
  CRF_CHECK(x && windows && B > 0 && H > 0 && W > 0 && C > 0 && window > 0, "crf_window_scatter: bad arguments");
  CRF_CHECK(shift >= 0 && shift < window, "shift_size must in 0-window_size");
  return launch_window_scatter(windows, x, B, H, W, C, window, shift, static_cast<cudaStream_t>(stream));
}
int crf_shift_mask(float* mask, int H, int W, int window, int shift, void* stream) {
  CRF_CHECK(mask && H > 0 && W > 0 && window > 0, "crf_shift_mask: bad arguments");
  CRF_CHECK(shift >= 0 && shift < window, "shift_size must in 0-window_size");
  return launch_shift_mask(mask, H, W, window, shift, static_cast<cudaStream_t>(stream));
}

size_t crf_gemm_workspace_bytes(int M, int N, int K, int device) {
  return gemm_splitk_workspace_bytes(M, N, K, device, nullptr);
}

int crf_layernorm_ps_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                         float* stats, int B, int H, int W, int C, int device, void* stream) {
  CRF_CHECK(x && gamma && beta && y && stats && B > 0 && H > 0 && W > 0, "crf_layernorm_ps_fwd: bad arguments");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_layernorm_fwd(x, gamma, beta, eps, y, y_dtype, stats, B * H * W, C, static_cast<cudaStream_t>(stream),
                              W);
}
int crf_layernorm_ps_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                         float* dgamma, float* dbeta, int B, int H, int W, int C, int device, void* stream) {
  CRF_CHECK(g && x && stats && gamma && dx && dgamma && dbeta && B > 0 && H > 0 && W > 0,
            "crf_layernorm_ps_bwd: bad arguments");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_layernorm_bwd(g, g_dtype, x, stats, gamma, dx, nullptr, dgamma, dbeta, B * H * W, C,
                              static_cast<cudaStream_t>(stream), W);
}

int crf_dgrad_ln_bwd(const void* dy_bf16, const void* w_bf16, int K, const float* x, const float* stats,
                     const float* gamma, const float* dres, float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T,
                     int C, int device, void* stream) {
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_dgrad_lnbwd(dy_bf16, w_bf16, K, x, stats, gamma, dres, dx, dx_bf16, dgamma, dbeta, T, C, device,
                            static_cast<cudaStream_t>(stream));
}

int crf_gemm(const crf_gemm_args* a, void* stream) {
  CRF_CHECK(a && a->A && a->B && (a->out0 || a->out1), "crf_gemm: null pointer");
  DeviceGuard guard(a->device);
  CRF_CHECK(guard.ok, "cannot select device %d", a->device);
  return launch_gemm(*a, static_cast<cudaStream_t>(stream));
}

int crf_mlp_fwd(const crf_mlp_args* a, void* stream) {
  CRF_CHECK(a != nullptr, "crf_mlp_fwd: null arguments");
  DeviceGuard guard(a->device);
  CRF_CHECK(guard.ok, "cannot select device %d", a->device);
  return launch_mlp_fused_fwd(*a, static_cast<cudaStream_t>(stream));
}

/* debug only (not in the public header): timeline of the last crf_mlp_fwd launch made with CRF_MLP_PROF=1 */
int crf_debug_mlp_prof(long long* out, int n) { return mlp_debug_prof(out, n); }

int crf_ln_fwd(const void* x, int x_dtype, int64_t sb, int64_t st, int64_t sc, int B, int T_img, int C,
               const float* gamma, const float* beta, float eps, void* xn_bf16, float* stats, float* x_copy,
               int device, void* stream) {
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_ln_fwd(x, x_dtype, sb, st, sc, B, T_img, C, gamma, beta, eps, xn_bf16, stats, x_copy,
                       static_cast<cudaStream_t>(stream));
}
int crf_ln_bwd(const float* g, const float* x, const float* stats, const float* gamma, const float* dres, float* dx,
               void* dx_bf16, float* dgamma, float* dbeta, int T, int C, int device, void* stream) {
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_ln_bwd(g, x, stats, gamma, dres, dx, dx_bf16, dgamma, dbeta, T, C, static_cast<cudaStream_t>(stream));
}
int crf_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                      float* stats, int T, int C, int device, void* stream) {
  CRF_CHECK(x && gamma && beta && y && stats && T > 0, "crf_layernorm_fwd: bad arguments");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_layernorm_fwd(x, gamma, beta, eps, y, y_dtype, stats, T, C, static_cast<cudaStream_t>(stream));
}
int crf_layernorm_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                      float* dgamma, float* dbeta, int T, int C, int device, void* stream) {
  CRF_CHECK(g && x && stats && gamma && dx && dgamma && dbeta && T > 0, "crf_layernorm_bwd: bad arguments");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_layernorm_bwd(g, g_dtype, x, stats, gamma, dx, nullptr, dgamma, dbeta, T, C,
                              static_cast<cudaStream_t>(stream));
}
int crf_depth_loss_fwd(const void* pred, int pred_dtype, const float* target, int n_img, int H, int W, float* sums,
                       float* G, int device, void* stream) {
  CRF_CHECK(pred && target && sums, "crf_depth_loss_fwd: null pointer");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_depth_loss_fwd(pred, pred_dtype, target, n_img, H, W, sums, G, static_cast<cudaStream_t>(stream));
}
int crf_depth_loss_bwd(const void* pred, int pred_dtype, const float* target, const float* G, const float* grad_loss,
                       int n_img, int H, int W, void* dpred, int device, void* stream) {
  CRF_CHECK(pred && target && G && grad_loss && dpred, "crf_depth_loss_bwd: null pointer");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_depth_loss_bwd(pred, pred_dtype, target, G, grad_loss, n_img, H, W, dpred,
                               static_cast<cudaStream_t>(stream));
}
int crf_pixel_shuffle_nhwc(const void* src, void* dst, int dtype, int B, int H, int W, int C, int inverse, int device,
                           void* stream) {
  CRF_CHECK(src && dst, "crf_pixel_shuffle_nhwc: null pointer");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_pixel_shuffle_nhwc(src, dst, dtype, B, H, W, C, inverse, static_cast<cudaStream_t>(stream));
}
int crf_adam_step(const crf_adam_tensor* tensors, int n_tensors, int chunk_elems, double lr, double beta1, double beta2,
                  double eps, double weight_decay, float* step, int device, void* stream) {
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_adam_step(tensors, n_tensors, chunk_elems, lr, beta1, beta2, eps, weight_decay, step,
                          static_cast<cudaStream_t>(stream));
}
int crf_colsum_bf16(const void* g, float* out, int T, int N, int device, void* stream) {
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_colsum_bf16(g, out, T, N, static_cast<cudaStream_t>(stream));
}
int crf_cast_bf16(const float* src, void* dst, int64_t n, int device, void* stream) {
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  return launch_cast_bf16(src, dst, n, static_cast<cudaStream_t>(stream));
}
size_t crf_bn_workspace_bytes(int T, int C, int device) { return bn_workspace_bytes(T, C, device); }
int crf_bn_fwd(const void* x, void* y, const float* weight, const float* bias, float* running_mean, float* running_var,
               long long* num_batches_tracked, float* save_mean, float* save_invstd, int T, int C, float eps,
               float momentum, int act, void* workspace, size_t workspace_bytes, int* tickets, int device, void* stream) {
  return launch_bn_fwd(x, y, weight, bias, running_mean, running_var, num_batches_tracked, save_mean, save_invstd, T, C,
                       eps, momentum, act, workspace, workspace_bytes, tickets, device, static_cast<cudaStream_t>(stream));
}
int crf_bn_bwd(const void* x, const void* dy, const float* weight, const float* bias, const float* save_mean,
               const float* save_invstd, void* dx, float* dweight, float* dbias, int T, int C, int act, void* workspace,
               size_t workspace_bytes, int* tickets, int device, void* stream) {
  return launch_bn_bwd(x, dy, weight, bias, save_mean, save_invstd, dx, dweight, dbias, T, C, act, workspace,
                       workspace_bytes, tickets, device, static_cast<cudaStream_t>(stream));
}
size_t crf_dwconv_workspace_bytes(int B, int H, int W, int C, int k, int stride, int device) {
  return dwconv_workspace_bytes(B, H, W, C, k, stride, device);
}
int crf_dwconv_fwd(const void* x, const float* weight, void* y, int B, int H, int W, int C, int k, int stride, int device,
                   void* stream) {
  return launch_dwconv_fwd(x, weight, y, B, H, W, C, k, stride, device, static_cast<cudaStream_t>(stream));
}
int crf_dwconv_bwd(const void* x, const float* weight, const void* dy, void* dx, float* dweight, int B, int H, int W,
                   int C, int k, int stride, void* workspace, size_t workspace_bytes, int* tickets, int device,
                   void* stream) {
  return launch_dwconv_bwd(x, weight, dy, dx, dweight, B, H, W, C, k, stride, workspace, workspace_bytes, tickets,
                           device, static_cast<cudaStream_t>(stream));
}

int crf_attn_fwd(const crf_block_desc* d, const void* qk, const void* vb, const float* qk_bias, float scale,
                 const float* rpb_table, const float* mask, int mask_windows, void* o, float* lse, void* stream) {
  if (check_desc(d)) return 1;
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  return launch_attn_fwd(*d, qk, vb, qk_bias, scale, rpb_table, mask, mask_windows, o, lse,
                         static_cast<cudaStream_t>(stream));
}
int crf_attn_bwd(const crf_block_desc* d, const void* qk, const void* vb, const float* qk_bias, float scale,
                 const float* rpb_table, const float* mask, int mask_windows, const float* lse, const void* dout,
                 void* dqk, float* dv, int dv_accumulate, float* d_table, float* d_qk_bias, void* stream) {
  if (check_desc(d)) return 1;
  DeviceGuard guard(d->device);
  CRF_CHECK(guard.ok, "cannot select device %d", d->device);
  return launch_attn_bwd(*d, qk, vb, qk_bias, scale, rpb_table, mask, mask_windows, lse, dout, dqk, dv,
                         dv_accumulate, d_table, d_qk_bias, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
