// The "fp32-accumulate" precision mode of the CRF block (BASELINE.json: rel 1e-3 against the reference's fp32 path;
// crf_block_desc.precision == CRF_PREC_FP32).  Same block, same C ABI, different arithmetic:
//
//   * every dense projection stays on the tcgen05 tensor cores but its fp32 operands are split into two bf16 terms,
//     x = hi + lo (hi = bf16(x), lo = bf16(x - hi): 16 mantissa bits together), stored side by side as (rows, 2 * cols),
//     and the GEMM accumulates the three significant partial products  hi*hi + hi*lo + lo*hi  in fp32 (TMEM) by
//     running its K loop three times over the two halves (crf_gemm_args.split3; the dropped lo*lo term is 2^-18
//     relative).  No new MMA kind, no new tile format: the split is a column offset of the TMA loads;
//   * everything between the GEMMs is fp32: LayerNorm outputs, q / k, the attention output, the MLP hidden activation
//     (exact-erf GELU with erff), all gradients;
//   * the window-attention core (6.5 % of the block's flops) runs in fp32 on the CUDA cores: one CTA per (window, head),
//     q / k / v rows gathered with the same closed-form pad + roll + partition index map (crf_window.cuh), scores,
//     relative-position bias, shift mask, softmax, P V and the whole backward (dq, dk, dv, d table, pad-key bias
//     gradient) held in shared memory.
//
// This mode exists for the tolerance, not for speed (about 3x the tensor work, fp32 traffic): bench.py reports its
// throughput next to the bf16 path.
#include <cuda_bf16.h>
#include <math.h>

#include "crf_host.h"
#include "crf_window.cuh"

namespace crf {

namespace {

inline size_t align_up(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

// ---------------------------------------------------------------------------------------------------------------------
// elementwise kernels
// ---------------------------------------------------------------------------------------------------------------------
// fp32 (rows, cols) -> bf16 (rows, 2 cols): [hi | lo]
__global__ void __launch_bounds__(256)
split_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t rows, int cols) {
  const int64_t n4 = rows * cols / 4;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x; i < n4; i += static_cast<int64_t>(gridDim.x) * 256) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    const int64_t e = i * 4;
    const int64_t r = e / cols;
    const int c = static_cast<int>(e - r * cols);
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y), h2 = __float2bfloat16_rn(v.z),
                        h3 = __float2bfloat16_rn(v.w);
    const __nv_bfloat16 l0 = __float2bfloat16_rn(v.x - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v.y - __bfloat162float(h1)),
                        l2 = __float2bfloat16_rn(v.z - __bfloat162float(h2)), l3 = __float2bfloat16_rn(v.w - __bfloat162float(h3));
    __nv_bfloat16* d = dst + r * 2 * cols + c;
    *reinterpret_cast<__nv_bfloat162*>(d) = __halves2bfloat162(h0, h1);
    *reinterpret_cast<__nv_bfloat162*>(d + 2) = __halves2bfloat162(h2, h3);
    *reinterpret_cast<__nv_bfloat162*>(d + cols) = __halves2bfloat162(l0, l1);
    *reinterpret_cast<__nv_bfloat162*>(d + cols + 2) = __halves2bfloat162(l2, l3);
  }
}

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float dgelu_exact(float x) {
  return 0.5f * (1.0f + erff(x * 0.70710678118654752f)) + x * 0.39894228040143268f * expf(-0.5f * x * x);
}
// mode 0: out = gelu(a);  mode 1: out = a * gelu'(b)   (exact erf form, nn.GELU default, newcrf_layers.py:12,172)
__global__ void __launch_bounds__(256)
gelu_f32_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, int64_t n, int mode) {
  const int64_t n4 = n / 4;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x; i < n4; i += static_cast<int64_t>(gridDim.x) * 256) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(a) + i);
    float4 o;
    if (mode == 0) {
      o = make_float4(gelu_exact(x.x), gelu_exact(x.y), gelu_exact(x.z), gelu_exact(x.w));
    } else {
      const float4 p = __ldg(reinterpret_cast<const float4*>(b) + i);
      o = make_float4(x.x * dgelu_exact(p.x), x.y * dgelu_exact(p.y), x.z * dgelu_exact(p.z), x.w * dgelu_exact(p.w));
    }
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

int launch_split(const float* src, void* dst, int64_t rows, int cols, cudaStream_t st) {
  const int64_t n4 = rows * cols / 4;
  int64_t blocks = (n4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  KernelTimer tm(st, 0.0, 8.0 * rows * cols, "split_bf16x2_%lldx%d", static_cast<long long>(rows), cols);
  split_bf16_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(src, static_cast<__nv_bfloat16*>(dst), rows, cols);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}
int launch_gelu_f32(const float* a, const float* b, float* out, int64_t n, int mode, cudaStream_t st) {
  const int64_t n4 = n / 4;
  int64_t blocks = (n4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  KernelTimer tm(st, 0.0, (mode ? 12.0 : 8.0) * n, "gelu_f32_%s_n%lld", mode ? "bwd" : "fwd", static_cast<long long>(n));
  gelu_f32_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(a, b, out, n, mode);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// fp32 window attention on the CUDA cores: one CTA (64 threads) per (window, head)
// ---------------------------------------------------------------------------------------------------------------------
struct AttnF32 {
  const float* qk;        // (T, 2C) fp32: q (unscaled) | k
  const void* v;          // logical (B, H, W, C), element strides below, fp32 or bf16
  int v_bf16;
  int64_t vsb, vsh, vsw, vsc;
  const float* qk_bias;   // (2C): q / k of a zero-pad token (LayerNorm output is padded with zeros AFTER the norm)
  const float* table;     // ((2ws-1)^2, nH)
  const float* ext_mask;  // (ext_nw, N, N) additive or nullptr (closed-form shift mask), N = ws^2
  int ext_nw;
  float scale;
  int B, H, W, C, nH, hd;
  WindowGeom gm;
  // forward
  float* out;             // (T, C) token order
  // backward
  const float* dout;      // (T, C)
  float* dqk;             // (T, 2C)
  float* dv;              // (B, H, W, C) contiguous
  int dv_acc;
  float* d_table;         // ((2ws-1)^2, nH), +=
  float* d_qk_bias;       // (2C), += (pad keys)
};

__device__ __forceinline__ float load_v(const AttnF32& P, int b, int tok, int c) {
  const int h = tok / P.W, w = tok - h * P.W;
  const int64_t off = b * P.vsb + h * P.vsh + w * P.vsw + c * P.vsc;
  return P.v_bf16 ? __bfloat162float(static_cast<const __nv_bfloat16*>(P.v)[off]) : static_cast<const float*>(P.v)[off];
}
// Per window size WS: kN = WS^2 tokens per window, kPS = kN + 1 the row stride of the kN x kN score tiles in shared
// memory, kTbl floats for a head's relative-position table (49 / 50 / 176 at WS = 7).
template <int WS>
struct Win {
  static constexpr int kN = WS * WS;
  static constexpr int kPS = kN + 1;
  static constexpr int kTbl = rpb_table_padded(WS);
};

// Gathers the window's q (scaled), k, v (and dO) rows of one head into shared memory; tok[n] = token index or -1.
template <int WS, bool BWD>
__device__ void attn_gather(const AttnF32& P, int b, int win, int head, float* q, float* k, float* v, float* dO, int* tok,
                            float* tb) {
  constexpr int kN = Win<WS>::kN;
  const int hd = P.hd, hs = hd + 1, C = P.C;
  for (int n = threadIdx.x; n < kN; n += blockDim.x) tok[n] = P.gm.source(win, n);
  for (int t = threadIdx.x; t < rpb_table_size(WS); t += blockDim.x) tb[t] = P.table[t * P.nH + head];
  __syncthreads();
  for (int idx = threadIdx.x; idx < kN * hd; idx += blockDim.x) {
    const int n = idx / hd, d = idx - n * hd, c = head * hd + d;
    const int tk = tok[n];
    float qv, kv, vv, dov = 0.f;
    if (tk >= 0) {
      const int64_t g = static_cast<int64_t>(b) * P.H * P.W + tk;
      qv = P.qk[g * 2 * C + c];
      kv = P.qk[g * 2 * C + C + c];
      vv = load_v(P, b, tk, c);
      if (BWD) dov = P.dout[g * C + c];
    } else {
      qv = P.qk_bias[c];
      kv = P.qk_bias[C + c];
      vv = 0.f;
    }
    q[n * hs + d] = qv * P.scale;
    k[n * hs + d] = kv;
    v[n * hs + d] = vv;
    if (BWD) dO[n * hs + d] = dov;
  }
  __syncthreads();
}

// scores of query row i -> p[i][.] = softmax_j(q_i . k_j + bias + mask)
template <int WS>
__device__ void attn_softmax_row(const AttnF32& P, int wg, int win, int i, const float* q, const float* k, const float* tb,
                                 float* p) {
  constexpr int kN = Win<WS>::kN, kPS = Win<WS>::kPS;
  const int hd = P.hd, hs = hd + 1;
  const float* xmask = P.ext_mask != nullptr ? P.ext_mask + (static_cast<int64_t>(wg % P.ext_nw) * kN + i) * kN : nullptr;
  const int ri = (P.gm.shift > 0 && xmask == nullptr) ? P.gm.region(win, i) : 0;
  float mx = -INFINITY;
  for (int j = 0; j < kN; ++j) {
    float s = 0.f;
    for (int d = 0; d < hd; ++d) s = fmaf(q[i * hs + d], k[j * hs + d], s);
    s += tb[rel_position_index<WS>(i, j)];
    if (xmask != nullptr) s += xmask[j];
    else if (P.gm.shift > 0 && P.gm.region(win, j) != ri) s += -100.0f;  // newcrf_layers.py:350
    p[i * kPS + j] = s;
    mx = fmaxf(mx, s);
  }
  float sum = 0.f;
  for (int j = 0; j < kN; ++j) {
    const float e = expf(p[i * kPS + j] - mx);
    p[i * kPS + j] = e;
    sum += e;
  }
  const float inv = 1.0f / sum;
  for (int j = 0; j < kN; ++j) p[i * kPS + j] *= inv;
}

template <int WS>
__global__ void __launch_bounds__(64)
attn_fwd_f32_kernel(const AttnF32 P) {
  constexpr int kN = Win<WS>::kN, kPS = Win<WS>::kPS;
  extern __shared__ float sm[];
  const int hd = P.hd, hs = hd + 1;
  float* q = sm;
  float* k = q + kN * hs;
  float* v = k + kN * hs;
  float* p = v + kN * hs;
  float* tb = p + kN * kPS;
  int* tok = reinterpret_cast<int*>(tb + Win<WS>::kTbl);
  const int wg = blockIdx.x, head = blockIdx.y;
  const int b = wg / P.gm.nW, win = wg - b * P.gm.nW;
  attn_gather<WS, false>(P, b, win, head, q, k, v, nullptr, tok, tb);
  const int i = threadIdx.x;
  if (i < kN) {
    attn_softmax_row<WS>(P, wg, win, i, q, k, tb, p);
    if (tok[i] >= 0) {  // pad queries are dropped by the crop (newcrf_layers.py:248-249)
      float* o = P.out + (static_cast<int64_t>(b) * P.H * P.W + tok[i]) * P.C + head * hd;
      for (int d = 0; d < hd; ++d) {
        float acc = 0.f;
        for (int j = 0; j < kN; ++j) acc = fmaf(p[i * kPS + j], v[j * hs + d], acc);
        o[d] = acc;
      }
    }
  }
}

template <int WS>
__global__ void __launch_bounds__(64)
attn_bwd_f32_kernel(const AttnF32 P) {
  constexpr int kN = Win<WS>::kN, kPS = Win<WS>::kPS;
  extern __shared__ float sm[];
  const int hd = P.hd, hs = hd + 1, C = P.C;
  float* q = sm;
  float* k = q + kN * hs;
  float* v = k + kN * hs;
  float* dO = v + kN * hs;
  float* p = dO + kN * hs;
  float* ds = p + kN * kPS;
  float* tb = ds + kN * kPS;
  float* tg = tb + Win<WS>::kTbl;
  int* tok = reinterpret_cast<int*>(tg + Win<WS>::kTbl);
  const int wg = blockIdx.x, head = blockIdx.y;
  const int b = wg / P.gm.nW, win = wg - b * P.gm.nW;
  for (int t = threadIdx.x; t < rpb_table_size(WS); t += blockDim.x) tg[t] = 0.f;
  attn_gather<WS, true>(P, b, win, head, q, k, v, dO, tok, tb);
  const int i = threadIdx.x;
  if (i < kN) {
    attn_softmax_row<WS>(P, wg, win, i, q, k, tb, p);
    // dP = dO V^T ; dS = P o (dP - sum_j P dP)
    float dot = 0.f;
    for (int j = 0; j < kN; ++j) {
      float dp = 0.f;
      for (int d = 0; d < hd; ++d) dp = fmaf(dO[i * hs + d], v[j * hs + d], dp);
      ds[i * kPS + j] = dp;
      dot = fmaf(p[i * kPS + j], dp, dot);
    }
    for (int j = 0; j < kN; ++j) {
      const float g = p[i * kPS + j] * (ds[i * kPS + j] - dot);
      ds[i * kPS + j] = g;
      if (g != 0.f) atomicAdd(&tg[rel_position_index<WS>(i, j)], g);
    }
    if (tok[i] >= 0) {  // dq = scale * dS K   (gradient of the UNSCALED q the qk projection produced)
      float* dq = P.dqk + (static_cast<int64_t>(b) * P.H * P.W + tok[i]) * 2 * C + head * hd;
      for (int d = 0; d < hd; ++d) {
        float acc = 0.f;
        for (int j = 0; j < kN; ++j) acc = fmaf(ds[i * kPS + j], k[j * hs + d], acc);
        dq[d] = acc * P.scale;
      }
    }
  }
  __syncthreads();
  if (i < kN) {  // thread = key j: dk = dS^T (q scaled), dv = P^T dO
    const int j = i;
    const int tk = tok[j];
    for (int d = 0; d < hd; ++d) {
      float dk = 0.f, dvv = 0.f;
      for (int r = 0; r < kN; ++r) {
        dk = fmaf(ds[r * kPS + j], q[r * hs + d], dk);
        dvv = fmaf(p[r * kPS + j], dO[r * hs + d], dvv);
      }
      const int c = head * hd + d;
      if (tk >= 0) {
        const int64_t g = static_cast<int64_t>(b) * P.H * P.W + tk;
        P.dqk[g * 2 * C + C + c] = dk;
        float* dvp = P.dv + g * C + c;
        *dvp = P.dv_acc ? *dvp + dvv : dvv;  // every real token sits in exactly one window slot: no atomics
      } else {
        atomicAdd(P.d_qk_bias + C + c, dk);  // a pad key IS the k bias
      }
    }
  }
  for (int t = threadIdx.x; t < rpb_table_size(WS); t += blockDim.x)
    if (tg[t] != 0.f) atomicAdd(P.d_table + t * P.nH + head, tg[t]);
}

template <int WS>
size_t attn_smem(int hd, bool bwd) {
  constexpr int kN = Win<WS>::kN, kPS = Win<WS>::kPS, kTbl = Win<WS>::kTbl;
  const size_t rows = static_cast<size_t>(kN) * (hd + 1);
  return ((bwd ? 4 : 3) * rows + (bwd ? 2 : 1) * kN * kPS + (bwd ? 2 * kTbl : kTbl) + 64) * sizeof(float);
}

AttnF32 attn_params(const crf_block_desc& d, const crf_block_params& p, const float* qk, const void* v) {
  AttnF32 P{};
  P.qk = qk;
  P.v = v;
  P.v_bf16 = d.v_dtype == CRF_DT_BF16;
  P.vsb = d.v_stride_b; P.vsh = d.v_stride_h; P.vsw = d.v_stride_w; P.vsc = d.v_stride_c;
  P.qk_bias = p.qk_b;
  P.table = p.rpb_table;
  P.ext_mask = p.ext_mask;
  P.ext_nw = p.ext_mask_windows > 0 ? p.ext_mask_windows : 1;
  P.scale = p.qk_scale;
  P.B = d.B; P.H = d.H; P.W = d.W; P.C = d.C; P.nH = d.num_heads; P.hd = d.C / d.num_heads;
  P.gm = WindowGeom(d.H, d.W, d.window, d.shift);
  return P;
}

template <int WS>
int attn_fwd_f32(const crf_block_desc& d, const AttnF32& P, cudaStream_t st) {
  const size_t smem = attn_smem<WS>(P.hd, false);
  CRF_CUDA(cudaFuncSetAttribute(attn_fwd_f32_kernel<WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const double T = static_cast<double>(d.B) * d.H * d.W, N = WS * WS;
  KernelTimer tm(st, 4.0 * N * N * d.C * d.B * P.gm.nW, T * d.C * 16.0, "attn_fwd_f32_B%d_%dx%d_C%d_s%d", d.B, d.H, d.W, d.C,
                 d.shift);
  attn_fwd_f32_kernel<WS><<<dim3(d.B * P.gm.nW, d.num_heads), 64, smem, st>>>(P);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}
template <int WS>
int attn_bwd_f32(const crf_block_desc& d, const AttnF32& P, cudaStream_t st) {
  const size_t smem = attn_smem<WS>(P.hd, true);
  CRF_CUDA(cudaFuncSetAttribute(attn_bwd_f32_kernel<WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const double T = static_cast<double>(d.B) * d.H * d.W, N = WS * WS;
  KernelTimer tm(st, 10.0 * N * N * d.C * d.B * P.gm.nW, T * d.C * 32.0, "attn_bwd_f32_B%d_%dx%d_C%d_s%d", d.B, d.H, d.W, d.C,
                 d.shift);
  attn_bwd_f32_kernel<WS><<<dim3(d.B * P.gm.nW, d.num_heads), 64, smem, st>>>(P);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_attn_fwd_f32(const crf_block_desc& d, const crf_block_params& p, const float* qk, const void* v, float* out,
                        cudaStream_t st) {
  AttnF32 P = attn_params(d, p, qk, v);
  P.out = out;
  const int rc = with_window(d.window, [&](auto w) { return attn_fwd_f32<decltype(w)::value>(d, P, st); });
  return rc >= 0 ? rc : set_error("fp32 attention: no kernel for window %d", d.window);
}
int launch_attn_bwd_f32(const crf_block_desc& d, const crf_block_params& p, const float* qk, const void* v, const float* dout,
                        float* dqk, float* dv, int dv_acc, float* d_table, float* d_qk_bias, cudaStream_t st) {
  AttnF32 P = attn_params(d, p, qk, v);
  P.dout = dout; P.dqk = dqk; P.dv = dv; P.dv_acc = dv_acc; P.d_table = d_table; P.d_qk_bias = d_qk_bias;
  const int rc = with_window(d.window, [&](auto w) { return attn_bwd_f32<decltype(w)::value>(d, P, st); });
  return rc >= 0 ? rc : set_error("fp32 attention: no kernel for window %d", d.window);
}

// ---------------------------------------------------------------------------------------------------------------------
// split-operand GEMM wrapper: operands are (rows, 2 * cols) [hi | lo] bf16 matrices, logical shapes as in crf_gemm
// ---------------------------------------------------------------------------------------------------------------------
int pgemm(const void* A, const void* B, int a_major, int b_major, int M, int N, int K, int epi, void* out0, const float* bias,
          const void* aux1, float* colsum, void* ws, size_t ws_bytes, int device, cudaStream_t st) {
  crf_gemm_args a{};
  a.A = A; a.B = B; a.a_major = a_major; a.b_major = b_major;
  a.M = M; a.N = N; a.K = K; a.epilogue = epi; a.split_k = epi == CRF_EPI_SPLITK_F32 ? 0 : 1;
  a.out0 = out0; a.bias = bias; a.aux1 = aux1; a.ld_out = N; a.scale = 1.f; a.scale_cols = 0; a.device = device;
  a.workspace = ws; a.workspace_bytes = ws_bytes; a.colsum = colsum; a.split3 = 1;
  return launch_gemm(a, st);
}

struct PSaved {  // forward products of the precise mode (offsets in bytes)
  size_t xc, stats1, xnb, xn1f, xn1s, qkf, attn_of, attn_os, x1, stats2, xn2f, xn2s, pre, actf, acts, w_qk, w_proj, w_fc1,
      w_fc2, total;
};
struct PBwd {
  size_t dys, dh, dhs, dxn, dx1, dx1s, dof, dqkf, dqks, partials, partials_bytes, total;
};

bool x_plain(const crf_block_desc& d) {
  const int64_t T_img = static_cast<int64_t>(d.H) * d.W;
  return d.x_dtype == CRF_DT_F32 && d.x_stride_c == 1 && d.x_stride_t == d.C && d.x_stride_b == T_img * d.C;
}

PSaved psaved(const crf_block_desc& d) {
  const size_t T = static_cast<size_t>(d.B) * d.H * d.W, C = d.C;
  PSaved L{};
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
  L.xc = take(x_plain(d) ? 0 : T * C * 4);
  L.stats1 = take(T * 8);
  L.xnb = take(x_plain(d) ? 0 : T * C * 2);  // bf16 by-product of the layout-changing LayerNorm kernel (unused)
  L.xn1f = take(T * C * 4);
  L.xn1s = take(T * C * 4);
  L.qkf = take(T * C * 8);
  L.attn_of = take(T * C * 4);
  L.attn_os = take(T * C * 4);
  L.x1 = take(T * C * 4);
  L.stats2 = take(T * 8);
  L.xn2f = take(T * C * 4);
  L.xn2s = take(T * C * 4);
  L.pre = take(T * C * 16);
  L.actf = take(T * C * 16);
  L.acts = take(T * C * 16);
  L.w_qk = take(2 * C * C * 4);
  L.w_proj = take(C * C * 4);
  L.w_fc1 = take(4 * C * C * 4);
  L.w_fc2 = take(4 * C * C * 4);
  L.total = o;
  return L;
}
PBwd pbwd(const crf_block_desc& d) {
  const size_t T = static_cast<size_t>(d.B) * d.H * d.W, C = d.C;
  PBwd L{};
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
  L.dys = take(T * C * 4);
  L.dh = take(T * C * 16);
  L.dhs = take(T * C * 16);
  L.dxn = take(T * C * 4);
  L.dx1 = take(T * C * 4);
  L.dx1s = take(T * C * 4);
  L.dof = take(T * C * 4);
  L.dqkf = take(T * C * 8);
  L.dqks = take(T * C * 8);
  const int Ti = static_cast<int>(T), Ci = d.C;
  size_t pb = 0;
  const int shapes[4][2] = {{Ci, 4 * Ci}, {4 * Ci, Ci}, {Ci, Ci}, {2 * Ci, Ci}};
  for (auto& s : shapes) {
    const size_t b = gemm_splitk_workspace_bytes(s[0], s[1], 3 * Ti, d.device, nullptr);
    if (b > pb) pb = b;
  }
  L.partials_bytes = pb;
  L.partials = take(pb);
  L.total = o;
  return L;
}

}  // namespace

size_t precise_saved_bytes(const crf_block_desc& d) { return psaved(d).total; }
size_t precise_bwd_bytes(const crf_block_desc& d) { return pbwd(d).total; }

int block_fwd_precise(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, float* y, void* saved,
                      cudaStream_t st) {
  CRF_CHECK(!d->v_preconverted, "precise mode reads v in its own dtype (v_preconverted must be 0)");
  const PSaved L = psaved(*d);
  uint8_t* S = static_cast<uint8_t*>(saved);
  const int T = d->B * d->H * d->W, C = d->C, dev = d->device;
  auto F = [&](size_t off) { return reinterpret_cast<float*>(S + off); };
  // weights -> [hi | lo]
  if (launch_split(p->qk_w, S + L.w_qk, 2 * C, C, st)) return 1;
  if (launch_split(p->proj_w, S + L.w_proj, C, C, st)) return 1;
  if (launch_split(p->fc1_w, S + L.w_fc1, 4 * C, C, st)) return 1;
  if (launch_split(p->fc2_w, S + L.w_fc2, C, 4 * C, st)) return 1;
  // LN1 in fp32 (a strided / bf16 x is first copied to token-major fp32 rows)
  const float* x_tok = static_cast<const float*>(x);
  if (!x_plain(*d)) {
    if (launch_ln_fwd(x, d->x_dtype, d->x_stride_b, d->x_stride_t, d->x_stride_c, d->B, d->H * d->W, C, p->norm1_w, p->norm1_b,
                      p->ln_eps, S + L.xnb, F(L.stats1), F(L.xc), st))
      return 1;
    x_tok = F(L.xc);
  }
  if (launch_layernorm_fwd(x_tok, p->norm1_w, p->norm1_b, p->ln_eps, F(L.xn1f), CRF_DT_F32, F(L.stats1), T, C, st)) return 1;
  if (launch_split(F(L.xn1f), S + L.xn1s, T, C, st)) return 1;
  // q | k (unscaled; the attention kernel applies the scale)
  if (pgemm(S + L.xn1s, S + L.w_qk, 0, 0, T, 2 * C, C, CRF_EPI_STORE_F32, F(L.qkf), p->qk_b, nullptr, nullptr, nullptr, 0, dev, st))
    return 1;
  if (launch_attn_fwd_f32(*d, *p, F(L.qkf), v, F(L.attn_of), st)) return 1;
  if (launch_split(F(L.attn_of), S + L.attn_os, T, C, st)) return 1;
  // x1 = x + proj(attn)
  if (pgemm(S + L.attn_os, S + L.w_proj, 0, 0, T, C, C, CRF_EPI_BIAS_RES_F32, F(L.x1), p->proj_b, x_tok, nullptr, nullptr, 0, dev, st))
    return 1;
  if (launch_layernorm_fwd(F(L.x1), p->norm2_w, p->norm2_b, p->ln_eps, F(L.xn2f), CRF_DT_F32, F(L.stats2), T, C, st)) return 1;
  if (launch_split(F(L.xn2f), S + L.xn2s, T, C, st)) return 1;
  if (pgemm(S + L.xn2s, S + L.w_fc1, 0, 0, T, 4 * C, C, CRF_EPI_STORE_F32, F(L.pre), p->fc1_b, nullptr, nullptr, nullptr, 0, dev, st))
    return 1;
  if (launch_gelu_f32(F(L.pre), nullptr, F(L.actf), static_cast<int64_t>(T) * 4 * C, 0, st)) return 1;
  if (launch_split(F(L.actf), S + L.acts, T, 4 * C, st)) return 1;
  return pgemm(S + L.acts, S + L.w_fc2, 0, 0, T, C, 4 * C, CRF_EPI_BIAS_RES_F32, y, p->fc2_b, F(L.x1), nullptr, nullptr, 0, dev, st);
}

int block_bwd_precise(const crf_block_desc* d, const crf_block_params* p, const void* x, const void* v, const float* dy,
                      const void* saved, float* dx, void* dx_bf16, float* dv, int dv_accumulate, const crf_block_grads* g,
                      void* ws, size_t ws_bytes, cudaStream_t st) {
  const PSaved L = psaved(*d);
  const PBwd W = pbwd(*d);
  CRF_CHECK(ws_bytes >= W.total, "crf_block_bwd (fp32 mode): workspace too small (%zu < %zu)", ws_bytes, W.total);
  uint8_t* S = const_cast<uint8_t*>(static_cast<const uint8_t*>(saved));
  uint8_t* Wk = static_cast<uint8_t*>(ws);
  const int T = d->B * d->H * d->W, C = d->C, dev = d->device;
  auto F = [&](size_t off) { return reinterpret_cast<float*>(S + off); };
  auto G = [&](size_t off) { return reinterpret_cast<float*>(Wk + off); };
  const float* x_tok = x_plain(*d) ? static_cast<const float*>(x) : F(L.xc);
  // ---- MLP ----
  if (launch_split(dy, Wk + W.dys, T, C, st)) return 1;
  if (pgemm(Wk + W.dys, S + L.w_fc2, 0, 1, T, 4 * C, C, CRF_EPI_STORE_F32, G(W.dh), nullptr, nullptr, nullptr, nullptr, 0, dev, st))
    return 1;
  if (launch_gelu_f32(G(W.dh), F(L.pre), G(W.dh), static_cast<int64_t>(T) * 4 * C, 1, st)) return 1;
  if (launch_split(G(W.dh), Wk + W.dhs, T, 4 * C, st)) return 1;
  if (pgemm(Wk + W.dys, S + L.acts, 1, 1, C, 4 * C, T, CRF_EPI_SPLITK_F32, g->fc2_w, nullptr, nullptr, g->fc2_b, Wk + W.partials,
            W.partials_bytes, dev, st))
    return 1;
  if (pgemm(Wk + W.dhs, S + L.w_fc1, 0, 1, T, C, 4 * C, CRF_EPI_STORE_F32, G(W.dxn), nullptr, nullptr, nullptr, nullptr, 0, dev, st))
    return 1;
  if (pgemm(Wk + W.dhs, S + L.xn2s, 1, 1, 4 * C, C, T, CRF_EPI_SPLITK_F32, g->fc1_w, nullptr, nullptr, g->fc1_b, Wk + W.partials,
            W.partials_bytes, dev, st))
    return 1;
  if (launch_ln_bwd(G(W.dxn), F(L.x1), F(L.stats2), p->norm2_w, dy, G(W.dx1), nullptr, g->norm2_w, g->norm2_b, T, C, st)) return 1;
  // ---- attention ----
  if (launch_split(G(W.dx1), Wk + W.dx1s, T, C, st)) return 1;
  if (pgemm(Wk + W.dx1s, S + L.w_proj, 0, 1, T, C, C, CRF_EPI_STORE_F32, G(W.dof), nullptr, nullptr, nullptr, nullptr, 0, dev, st))
    return 1;
  if (pgemm(Wk + W.dx1s, S + L.attn_os, 1, 1, C, C, T, CRF_EPI_SPLITK_F32, g->proj_w, nullptr, nullptr, g->proj_b, Wk + W.partials,
            W.partials_bytes, dev, st))
    return 1;
  if (launch_attn_bwd_f32(*d, *p, F(L.qkf), v, G(W.dof), G(W.dqkf), dv, dv_accumulate, g->rpb_table, g->qk_b, st)) return 1;
  if (launch_split(G(W.dqkf), Wk + W.dqks, T, 2 * C, st)) return 1;
  if (pgemm(Wk + W.dqks, S + L.w_qk, 0, 1, T, C, 2 * C, CRF_EPI_STORE_F32, G(W.dxn), nullptr, nullptr, nullptr, nullptr, 0, dev, st))
    return 1;
  if (pgemm(Wk + W.dqks, S + L.xn1s, 1, 1, 2 * C, C, T, CRF_EPI_SPLITK_F32, g->qk_w, nullptr, nullptr, g->qk_b, Wk + W.partials,
            W.partials_bytes, dev, st))
    return 1;
  return launch_ln_bwd(G(W.dxn), x_tok, F(L.stats1), p->norm1_w, G(W.dx1), dx, dx_bf16, g->norm1_w, g->norm1_b, T, C, st);
}

}  // namespace crf
