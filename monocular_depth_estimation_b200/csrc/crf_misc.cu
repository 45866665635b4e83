// Memory-bound helper kernels of the CRF block: LayerNorm forward (with the NCHW-view -> token-major layout
// change folded in), LayerNorm backward (with the residual add and the gamma/beta reductions folded in), bias
// gradient column sums, dtype casts, and the stand-alone window gather / scatter / mask used by the bit-exact
// index tests.  All of these are HBM-bound: coalesced, vectorised accesses, warp-shuffle reductions.
// The two LayerNorm row kernels (ln_fwd_rows_kernel, ln_bwd_kernel) take the layout of their output / incoming
// gradient as a template type: token-major rows, or the PixelShuffle(2) map that follows a decoder stage's closing
// norm.  The shuffled forms are instances of the same kernels, with the same arithmetic in the same order.
#include <algorithm>

#include "crf_host.h"
#include "crf_colreduce.cuh"
#include "crf_ptx.cuh"
#include "crf_window.cuh"

namespace crf {

namespace {

// ------------------------------------------------------------------------------------------------
// LayerNorm forward / plain conversion with layout change.
// x logical (B, T_img, C), element (b,t,c) at b*sb + t*st + c*sc.  A CTA stages a 32-token x C tile in smem
// (fp32), reading along whichever of (t, c) is contiguous, then one warp per token normalises and writes
// token-major outputs.  DO_LN=false -> plain conversion (used for v).
// ------------------------------------------------------------------------------------------------
constexpr int kLnTok = 32;
constexpr int kLnThreads = 256;

template <typename TIn>
__device__ __forceinline__ float load_as_float(const TIn* p);
template <>
__device__ __forceinline__ float load_as_float<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_as_float<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

template <typename TIn, bool DO_LN>
__global__ void __launch_bounds__(kLnThreads)
ln_fwd_kernel(const TIn* __restrict__ x, int64_t sb, int64_t st, int64_t sc, int T_img, int C,
              const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
              __nv_bfloat16* __restrict__ xn, float* __restrict__ stats, float* __restrict__ x_copy) {
  pdl_prologue();
  extern __shared__ float tile[];  // [kLnTok][C + 1]
  const int ldt = C + 1;
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kLnTok;
  const int nt = min(kLnTok, T_img - t0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TIn* xb = x + static_cast<int64_t>(b) * sb + static_cast<int64_t>(t0) * st;

  if (sc == 1) {  // token rows are contiguous
    for (int t = warp; t < nt; t += kLnThreads / 32)
      for (int c = lane; c < C; c += 32) tile[t * ldt + c] = load_as_float<TIn>(xb + t * st + c);
  } else {  // channel planes (NCHW view): tokens are contiguous (or generic strides)
    for (int c = warp; c < C; c += kLnThreads / 32)
      if (lane < nt) tile[lane * ldt + c] = load_as_float<TIn>(xb + lane * st + c * sc);
  }
  __syncthreads();

  for (int t = warp; t < nt; t += kLnThreads / 32) {
    const float* row = tile + t * ldt;
    const int64_t tg = static_cast<int64_t>(b) * T_img + t0 + t;
    float mean = 0.f, rstd = 1.f;
    if (DO_LN) {
      float s = 0.f;
      for (int c = lane; c < C; c += 32) s += row[c];
      mean = warp_sum(s) / C;
      float q = 0.f;
      for (int c = lane; c < C; c += 32) {
        const float d = row[c] - mean;
        q += d * d;
      }
      rstd = rsqrtf(warp_sum(q) / C + eps);
      if (lane == 0 && stats != nullptr) {
        stats[2 * tg] = mean;
        stats[2 * tg + 1] = rstd;
      }
    }
    for (int c = 2 * lane; c < C; c += 64) {
      float a0 = row[c], a1 = row[c + 1];
      if (x_copy != nullptr) *reinterpret_cast<float2*>(x_copy + tg * C + c) = make_float2(a0, a1);
      if (DO_LN) {
        a0 = (a0 - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
        a1 = (a1 - mean) * rstd * __ldg(gamma + c + 1) + __ldg(beta + c + 1);
      }
      *reinterpret_cast<uint32_t*>(xn + tg * C + c) = pack_bf16(a0, a1);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm forward, row-contiguous fast path (channel stride 1: token-major or channels-last input).
// One warp per token row, the row lives in registers (each lane owns channels {2*lane + 64k, +1}): x is read
// exactly once, two-pass mean / variance like torch's kernel.  Rows is the layout of the output xn (TokenRows /
// ShuffledRows below).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 load2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float2 load2(const __nv_bfloat16* p) {
  const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p));
  return make_float2(bf16_lo(w), bf16_hi(w));
}

__device__ __forceinline__ void store2(__nv_bfloat16* p, float a, float b) {
  *reinterpret_cast<uint32_t*>(p) = pack_bf16(a, b);
}
__device__ __forceinline__ void store2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }

// Row layouts of the two row kernels: where the channel pair (c, c + 1), c even, of token t of a (T, C) tensor p is
// stored (forward output) or loaded from (backward gradient).  Token-major rows: one packed access at p + t * C + c.
struct TokenRows {
  template <int C, typename T>
  __device__ __forceinline__ void store(T* p, int64_t t, int c, float a, float b) const { store2(p + t * C + c, a, b); }
  template <int C, typename T>
  __device__ __forceinline__ float2 load(const T* p, int64_t t, int c) const { return load2(p + t * C + c); }
};

// The same rows through the PixelShuffle(2) that follows a decoder stage (model_mobileV3_large_newCRFs.py:116-120):
// token (b, h, w) of an H x W grid, channel c = 4 k' + 2 i + j  <->  element (b, 2h + i, 2w + j, k') of the
// (B, 2H, 2W, C/4) NHWC map.  A pair (c, c + 1) is j = 0 / 1 of one output row: two scalar accesses C/4 apart.
// Output row 2h + i of image b is row 2 (b H + h) + i of the batch, so only W enters the map.
struct ShuffledRows {
  int W;
  template <int C>
  __device__ __forceinline__ int64_t offset(int64_t t, int c) const {
    const int ti = static_cast<int>(t);  // T = B H W is an int in the launchers
    const int w = ti % W, bh = ti / W;
    // c = 64 k + lo with k the unrolled loop index: written this way the compiler sees that only lo moves the
    // address off a per-lane base, so all of a row's accesses share one base register
    const int lo = c & 63;
    const int64_t pix = (static_cast<int64_t>(bh) * 2 + ((lo >> 1) & 1)) * 2 * W + 2 * w;
    return pix * (C / 4) + (lo >> 2) + 16 * (c >> 6);
  }
  template <int C, typename T>
  __device__ __forceinline__ void store(T* p, int64_t t, int c, float a, float b) const {
    T* o = p + offset<C>(t, c);
    o[0] = T(a);
    o[C / 4] = T(b);
  }
  template <int C, typename T>
  __device__ __forceinline__ float2 load(const T* p, int64_t t, int c) const {
    const T* o = p + offset<C>(t, c);
    return make_float2(static_cast<float>(__ldg(o)), static_cast<float>(__ldg(o + C / 4)));
  }
};

template <typename TIn, int NCH, bool DO_LN, typename TOut, typename Rows>
__global__ void __launch_bounds__(256)
ln_fwd_rows_kernel(const TIn* __restrict__ x, int64_t sb, int64_t st, int T_img, int64_t T,
                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                   TOut* __restrict__ xn, float* __restrict__ stats, float* __restrict__ x_copy, const Rows rows) {
  pdl_prologue();
  constexpr int C = 64 * NCH;
  // Input strided per image (sb, T_img) and the fp32 copy of x are LN1's, which is token-major.  The shuffled
  // (closing-norm) instances read one contiguous (T, C) block (sb = 0, T_img = T) and never copy x: without the 64-bit
  // division and the copy branch they have no stack frame and no spills (launch_ln_fwd_rows checks both conditions).
  constexpr bool kLn1 = std::is_same<Rows, TokenRows>::value;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t warps_total = static_cast<int64_t>(gridDim.x) * 8;
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * 8 + warp; t < T; t += warps_total) {
    const int64_t b = kLn1 ? t / T_img : 0;
    const TIn* row = x + b * sb + (t - b * T_img) * st;
    float2 v[NCH];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      v[k] = load2(row + 64 * k + 2 * lane);
      s += v[k].x + v[k].y;
    }
    float mean = 0.f, rstd = 1.f;
    if (DO_LN) {
      mean = warp_sum(s) * (1.0f / C);
      float q = 0.f;
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        const float d0 = v[k].x - mean, d1 = v[k].y - mean;
        q += d0 * d0 + d1 * d1;
      }
      rstd = rsqrtf(warp_sum(q) * (1.0f / C) + eps);
      if (lane == 0 && stats != nullptr) {
        stats[2 * t] = mean;
        stats[2 * t + 1] = rstd;
      }
    }
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = 64 * k + 2 * lane;
      if (kLn1 && x_copy != nullptr) *reinterpret_cast<float2*>(x_copy + t * C + c) = v[k];
      float a0 = v[k].x, a1 = v[k].y;
      if (DO_LN) {
        const float2 g = __ldg(reinterpret_cast<const float2*>(gamma + c));
        const float2 be = __ldg(reinterpret_cast<const float2*>(beta + c));
        a0 = (a0 - mean) * rstd * g.x + be.x;
        a1 = (a1 - mean) * rstd * g.y + be.y;
      }
      rows.template store<C>(xn, t, c, a0, a1);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward.  One warp per token row (grid-stride); each lane owns channels {2*lane + 64k, +1}.
//   dx = rstd * (g*gamma - mean_c(g*gamma) - xhat * mean_c(g*gamma*xhat)) + dres
//   dgamma += sum_t g * xhat,  dbeta += sum_t g
// Rows is the layout of g (TokenRows / ShuffledRows); x, dres and dx are token-major.
// ------------------------------------------------------------------------------------------------
template <int NCH, typename TG, typename Rows>  // C = 64 * NCH
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const TG* __restrict__ g, const float* __restrict__ x, const float* __restrict__ stats,
              const float* __restrict__ gamma, const float* __restrict__ dres, float* __restrict__ dx,
              __nv_bfloat16* __restrict__ dx_bf16, float* __restrict__ dgamma, float* __restrict__ dbeta, int T,
              const Rows rows) {
  pdl_prologue();
  constexpr int C = 64 * NCH;
  __shared__ __align__(16) float red[8][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float2 gam[NCH], dga[NCH], dbe[NCH];
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    gam[k] = __ldg(reinterpret_cast<const float2*>(gamma + 64 * k + 2 * lane));
    dga[k] = make_float2(0.f, 0.f);
    dbe[k] = make_float2(0.f, 0.f);
  }
  const int warps_total = gridDim.x * 8;
  for (int t = blockIdx.x * 8 + warp; t < T; t += warps_total) {
    const float mean = __ldg(stats + 2 * t), rstd = __ldg(stats + 2 * t + 1);
    float2 gv[NCH], xh[NCH];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      gv[k] = rows.template load<C>(g, t, 64 * k + 2 * lane);
      const float2 xv = __ldg(reinterpret_cast<const float2*>(x + static_cast<int64_t>(t) * C + 64 * k + 2 * lane));
      xh[k] = make_float2((xv.x - mean) * rstd, (xv.y - mean) * rstd);
      dga[k].x += gv[k].x * xh[k].x; dga[k].y += gv[k].y * xh[k].y;
      dbe[k].x += gv[k].x;           dbe[k].y += gv[k].y;
      gv[k].x *= gam[k].x;           gv[k].y *= gam[k].y;
      s1 += gv[k].x + gv[k].y;
      s2 += gv[k].x * xh[k].x + gv[k].y * xh[k].y;
    }
    s1 = warp_sum(s1) * (1.0f / C);
    s2 = warp_sum(s2) * (1.0f / C);
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      float o0 = rstd * (gv[k].x - s1 - xh[k].x * s2);
      float o1 = rstd * (gv[k].y - s1 - xh[k].y * s2);
      const int64_t off = static_cast<int64_t>(t) * C + 64 * k + 2 * lane;
      if (dres != nullptr) {
        const float2 r = __ldg(reinterpret_cast<const float2*>(dres + off));
        o0 += r.x; o1 += r.y;
      }
      if (dx != nullptr) *reinterpret_cast<float2*>(dx + off) = make_float2(o0, o1);
      if (dx_bf16 != nullptr) *reinterpret_cast<uint32_t*>(dx_bf16 + off) = pack_bf16(o0, o1);
    }
  }
  // cross-warp reduction of the per-lane partial column sums, then one atomic per column per CTA
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    for (int pass = 0; pass < 2; ++pass) {
      const float2 v = pass == 0 ? dga[k] : dbe[k];
      red[warp][2 * lane] = v.x;
      red[warp][2 * lane + 1] = v.y;
      __syncthreads();
      if (threadIdx.x < 16) {  // four columns per thread, one vector reduction: 4x fewer atomic operations per CTA
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int w = 0; w < 8; ++w) {
          const float4 v = *reinterpret_cast<const float4*>(&red[w][4 * threadIdx.x]);
          s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        float* dst = (pass == 0 ? dgamma : dbeta) + 64 * k + 4 * threadIdx.x;
        if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
          red_add_f32x4(dst, s);
        } else {  // gradient buffers that are unaligned views (DDP buckets)
          atomicAdd(dst, s.x); atomicAdd(dst + 1, s.y); atomicAdd(dst + 2, s.z); atomicAdd(dst + 3, s.w);
        }
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// out[n] += sum_t g[t,n], g bf16 (T,N), on the shared column reduction (crf_colreduce.cuh): eight rows in flight (128 B
// per thread, 32 KB per CTA); a CTA covers up to 2048 columns x a row chunk, then two vector reductions per thread of
// row lane 0.  Two CTAs per SM: the atomics at the end are per CTA, so more CTAs cost more than they hide (6 CTAs per
// SM: 2.5x slower at N >= 256, measured).
// ------------------------------------------------------------------------------------------------
struct ColSumOp {
  static constexpr int kAcc = 1;
  static constexpr int kRows = 8;
  using Regs = uint4;
  const __nv_bfloat16* __restrict__ g;
  __device__ __forceinline__ uint4 load(int64_t off) const { return __ldg(reinterpret_cast<const uint4*>(g + off)); }
  __device__ __forceinline__ void add(const uint4& w, float (&s)[1][8]) const {
    float v[8];
    unpack_bf16x8(w, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) s[0][k] += v[k];
  }
};

__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const __nv_bfloat16* __restrict__ g, float* __restrict__ out, int T, int N, int rows_per_cta) {
  pdl_prologue();
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const int r0 = blockIdx.y * rows_per_cta;
  float s[1][8];
  colreduce_cta(ColSumOp{g}, c, N, r0, min(T, r0 + rows_per_cta), s);
  if (threadIdx.y == 0 && c < N) {
    const float4 a = make_float4(s[0][0], s[0][1], s[0][2], s[0][3]), b = make_float4(s[0][4], s[0][5], s[0][6], s[0][7]);
    if ((reinterpret_cast<uintptr_t>(out) & 15) == 0) {
      red_add_f32x4(out + c, a);
      red_add_f32x4(out + c + 4, b);
    } else {
      atomicAdd(out + c, a.x); atomicAdd(out + c + 1, a.y); atomicAdd(out + c + 2, a.z); atomicAdd(out + c + 3, a.w);
      atomicAdd(out + c + 4, b.x); atomicAdd(out + c + 5, b.y); atomicAdd(out + c + 6, b.z); atomicAdd(out + c + 7, b.w);
    }
  }
}

__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  pdl_prologue();
  const int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src + i));
    *reinterpret_cast<uint2*>(dst + i) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
  } else {
    for (int64_t j = i; j < n; ++j) dst[j] = __float2bfloat16(src[j]);
  }
}

// four fp32 -> bf16 casts in one launch (the weight matrices of a block); blockIdx.y selects the tensor
struct Cast4 {
  const float* src[4];
  __nv_bfloat16* dst[4];
  long long n[4];
};
__global__ void __launch_bounds__(256) cast4_bf16_kernel(const Cast4 c) {
  pdl_prologue();
  const float* __restrict__ src = c.src[blockIdx.y];
  __nv_bfloat16* __restrict__ dst = c.dst[blockIdx.y];
  const long long n = c.n[blockIdx.y];
  const long long stride = static_cast<long long>(gridDim.x) * 256 * 4;
  long long i = (static_cast<long long>(blockIdx.x) * 256 + threadIdx.x) * 4;
  // four independent 16-byte loads in flight per thread (64 KB per CTA-quad): the one-load loop reached 2.7 TB/s
  for (; i + 3 * stride + 3 < n; i += 4 * stride) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(src + i + u * stride));
#pragma unroll
    for (int u = 0; u < 4; ++u)
      *reinterpret_cast<uint2*>(dst + i + u * stride) = make_uint2(pack_bf16(v[u].x, v[u].y), pack_bf16(v[u].z, v[u].w));
  }
  for (; i < n; i += stride) {
    if (i + 3 < n) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(src + i));
      *reinterpret_cast<uint2*>(dst + i) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
    } else {
      for (long long j = i; j < n; ++j) dst[j] = __float2bfloat16(src[j]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// stand-alone window gather / scatter / mask (bit-exact index tests)
// ------------------------------------------------------------------------------------------------
__global__ void window_gather_kernel(const float* __restrict__ x, float* __restrict__ win, WindowGeom gm, int C) {
  pdl_prologue();
  const int bw = blockIdx.x;  // b * nW + window
  const int b = bw / gm.nW, w = bw - b * gm.nW;
  const int N = gm.ws * gm.ws;
  for (int e = threadIdx.x; e < N * C; e += blockDim.x) {
    const int p = e / C, c = e - p * C;
    const int src = gm.source(w, p);
    win[(static_cast<int64_t>(bw) * N + p) * C + c] =
        src < 0 ? 0.f : x[(static_cast<int64_t>(b) * gm.H * gm.W + src) * C + c];
  }
}
__global__ void window_scatter_kernel(const float* __restrict__ win, float* __restrict__ x, WindowGeom gm, int C) {
  pdl_prologue();
  const int bw = blockIdx.x;
  const int b = bw / gm.nW, w = bw - b * gm.nW;
  const int N = gm.ws * gm.ws;
  for (int e = threadIdx.x; e < N * C; e += blockDim.x) {
    const int p = e / C, c = e - p * C;
    const int dst = gm.source(w, p);
    if (dst >= 0) x[(static_cast<int64_t>(b) * gm.H * gm.W + dst) * C + c] = win[(static_cast<int64_t>(bw) * N + p) * C + c];
  }
}
__global__ void shift_mask_kernel(float* __restrict__ mask, WindowGeom gm) {
  pdl_prologue();
  const int w = blockIdx.x;
  const int N = gm.ws * gm.ws;
  for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
    const int i = e / N, j = e - i * N;
    mask[static_cast<int64_t>(w) * N * N + e] = (gm.shift > 0 && gm.region(w, i) != gm.region(w, j)) ? -100.0f : 0.0f;
  }
}

// ------------------------------------------------------------------------------------------------
// PixelShuffle(2) between decoder stages (model_mobileV3_large_newCRFs.py:116-120) on channels-last memory:
//   dst[b, 2h+i, 2w+j, c'] = src[b, h, w, 4c' + 2i + j]        src (B, H, W, C), dst (B, 2H, 2W, C/4)
// One warp per source pixel: a lane loads the four channels of one output channel c' (one 8- or 16-byte load) and
// writes them to the four output pixels; INVERSE runs the same index map the other way (the backward).
// ------------------------------------------------------------------------------------------------
template <typename T, bool INVERSE>
__global__ void __launch_bounds__(256)
pixel_shuffle_nhwc_kernel(const T* __restrict__ src, T* __restrict__ dst, int B, int H, int W, int C) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int64_t npix = static_cast<int64_t>(B) * H * W;
  const int Cq = C >> 2;
  for (int64_t p = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5); p < npix;
       p += static_cast<int64_t>(gridDim.x) * 8) {
    const int w = static_cast<int>(p % W);
    const int64_t bh = p / W;  // b * H + h
    const T* big = (INVERSE ? dst : src) + p * C;                       // the (B, H, W, C) side
    const T* small00 = (INVERSE ? src : dst) + ((bh * 2) * (2 * W) + 2 * w) * Cq;   // output pixel (2h, 2w)
    const int64_t row = static_cast<int64_t>(2 * W) * Cq;               // one output row down
    for (int cq = lane; cq < Cq; cq += 32) {
      T v[4];
      if (!INVERSE) {
        if (sizeof(T) == 2) *reinterpret_cast<uint2*>(v) = __ldg(reinterpret_cast<const uint2*>(big + 4 * cq));
        else *reinterpret_cast<uint4*>(v) = __ldg(reinterpret_cast<const uint4*>(big + 4 * cq));
        T* o = const_cast<T*>(small00) + cq;
        o[0] = v[0]; o[Cq] = v[1]; o[row] = v[2]; o[row + Cq] = v[3];
      } else {
        const T* o = small00 + cq;
        v[0] = o[0]; v[1] = o[Cq]; v[2] = o[row]; v[3] = o[row + Cq];
        T* d = const_cast<T*>(big) + 4 * cq;
        if (sizeof(T) == 2) *reinterpret_cast<uint2*>(d) = *reinterpret_cast<const uint2*>(v);
        else *reinterpret_cast<uint4*>(d) = *reinterpret_cast<const uint4*>(v);
      }
    }
  }
}

// Calls f(std::integral_constant<int, C / 64>()) for a width the row kernels are instantiated for (C = 64 .. 1024 in
// steps of 64) and returns its result; returns -1 for any other C.
template <typename F>
int with_nch(int C, F&& f) {
  if (C % 64 != 0) return -1;
  switch (C / 64) {
    case 1: return f(std::integral_constant<int, 1>());
    case 2: return f(std::integral_constant<int, 2>());
    case 3: return f(std::integral_constant<int, 3>());
    case 4: return f(std::integral_constant<int, 4>());
    case 5: return f(std::integral_constant<int, 5>());
    case 6: return f(std::integral_constant<int, 6>());
    case 7: return f(std::integral_constant<int, 7>());
    case 8: return f(std::integral_constant<int, 8>());
    case 9: return f(std::integral_constant<int, 9>());
    case 10: return f(std::integral_constant<int, 10>());
    case 11: return f(std::integral_constant<int, 11>());
    case 12: return f(std::integral_constant<int, 12>());
    case 13: return f(std::integral_constant<int, 13>());
    case 14: return f(std::integral_constant<int, 14>());
    case 15: return f(std::integral_constant<int, 15>());
    case 16: return f(std::integral_constant<int, 16>());
    default: return -1;
  }
}

// Calls f with the row layout: the PixelShuffle(2) map of a token grid W wide when W > 0, token-major otherwise
template <typename F>
int with_rows(int W, F&& f) {
  return W > 0 ? f(ShuffledRows{W}) : f(TokenRows{});
}

// Grid of the warp-per-row kernels: one CTA per 8 rows, at most ctas_per_sm CTAs per SM (the kernels grid-stride)
int row_grid(int64_t rows, int ctas_per_sm) {
  int dev = 0;
  cudaGetDevice(&dev);
  return static_cast<int>(std::min<int64_t>((rows + 7) / 8, static_cast<int64_t>(num_sms(dev)) * ctas_per_sm));
}

template <typename TIn, bool DO_LN, typename TOut, typename Rows>
int launch_ln_fwd_rows(const TIn* x, int64_t sb, int64_t st_, int T_img, int64_t T, int C, const float* gamma,
                       const float* beta, float eps, TOut* xn, float* stats, float* x_copy, Rows rows,
                       int ctas_per_sm, cudaStream_t st) {
  // the shuffled instances read one contiguous (T, C) block and write no copy of x (see the kernel)
  CRF_CHECK((std::is_same<Rows, TokenRows>::value || (x_copy == nullptr && sb == 0 && T_img == T)),
            "LayerNorm forward: the PixelShuffle(2) layout takes contiguous rows and no copy of x");
  const int blocks = row_grid(T, ctas_per_sm);
  const int rc = with_nch(C, [&](auto nch) {
    launch_pdl((ln_fwd_rows_kernel<TIn, decltype(nch)::value, DO_LN, TOut, Rows>), blocks, 256, 0, st, x, sb, st_,
               T_img, T, gamma, beta, eps, xn, stats, x_copy, rows);
    return 0;
  });
  if (rc < 0) return set_error("LayerNorm forward: no row kernel for C=%d", C);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

// ctas_per_sm = 0: one resident wave, occupancy x SMs with at most 8 CTAs per SM
template <typename TG, typename Rows>
int launch_ln_bwd_rows(const TG* g, Rows rows, const float* x, const float* stats, const float* gamma,
                       const float* dres, float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T, int C,
                       int ctas_per_sm, cudaStream_t st) {
  __nv_bfloat16* dxb = reinterpret_cast<__nv_bfloat16*>(dx_bf16);
  const int rc = with_nch(C, [&](auto nch) {
    const auto kern = ln_bwd_kernel<decltype(nch)::value, TG, Rows>;
    int cap = ctas_per_sm;
    if (cap == 0) {
      static int occ = 0;
      if (occ == 0) {
        int o = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, 256, 0) != cudaSuccess || o < 1) o = 1;
        occ = o > 8 ? 8 : o;
      }
      cap = occ;
    }
    launch_pdl(kern, row_grid(T, cap), 256, 0, st, g, x, stats, gamma, dres, dx, dxb, dgamma, dbeta, T, rows);
    return 0;
  });
  if (rc < 0) return set_error("LayerNorm backward: no row kernel for C=%d", C);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

template <typename TIn>
int launch_ln_fwd_t(const void* x, int64_t sb, int64_t st_, int64_t sc, int B, int T_img, int C, const float* gamma,
                    const float* beta, float eps, void* xn, float* stats, float* x_copy, cudaStream_t st) {
  const size_t smem = static_cast<size_t>(kLnTok) * (C + 1) * sizeof(float);
  dim3 grid((T_img + kLnTok - 1) / kLnTok, B);
  const double tc = static_cast<double>(B) * T_img * C;
  KernelTimer tm(st, 0.0, tc * (sizeof(TIn) + 2 + (x_copy != nullptr ? 4 : 0)), "%s_T%d_C%d",
                 gamma != nullptr ? "ln_fwd" : "convert_bf16", B * T_img, C);
  const bool aligned = (reinterpret_cast<uintptr_t>(x) % 8 == 0) && (sb % 2 == 0) && (st_ % 2 == 0);
  if (sc == 1 && aligned) {  // rows are contiguous: warp-per-row, row held in registers, x read once
    const TIn* xp = reinterpret_cast<const TIn*>(x);
    const int64_t T = static_cast<int64_t>(B) * T_img;
    __nv_bfloat16* xnp = reinterpret_cast<__nv_bfloat16*>(xn);
    if (gamma != nullptr)
      return launch_ln_fwd_rows<TIn, true>(xp, sb, st_, T_img, T, C, gamma, beta, eps, xnp, stats, x_copy, TokenRows{},
                                           16, st);
    return launch_ln_fwd_rows<TIn, false>(xp, sb, st_, T_img, T, C, nullptr, nullptr, eps, xnp, nullptr, x_copy,
                                          TokenRows{}, 16, st);
  }
  if (gamma != nullptr) {
    auto k = ln_fwd_kernel<TIn, true>;
    CRF_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    launch_pdl(k, grid, kLnThreads, smem, st, reinterpret_cast<const TIn*>(x), sb, st_, sc, T_img, C, gamma, beta, eps,
                                      reinterpret_cast<__nv_bfloat16*>(xn), stats, x_copy);
  } else {
    auto k = ln_fwd_kernel<TIn, false>;
    CRF_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    launch_pdl(k, grid, kLnThreads, smem, st, reinterpret_cast<const TIn*>(x), sb, st_, sc, T_img, C, nullptr, nullptr, eps,
                                      reinterpret_cast<__nv_bfloat16*>(xn), nullptr, x_copy);
  }
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace

int launch_ln_fwd(const void* x, int x_dtype, int64_t sb, int64_t st_, int64_t sc, int B, int T_img, int C,
                  const float* gamma, const float* beta, float eps, void* xn, float* stats, float* x_copy,
                  cudaStream_t st) {
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "ln_fwd: C=%d must be a multiple of 64 in [64,1024]", C);
  CRF_CHECK(gamma != nullptr && beta != nullptr, "ln_fwd: gamma/beta required");
  if (x_dtype == CRF_DT_F32)
    return launch_ln_fwd_t<float>(x, sb, st_, sc, B, T_img, C, gamma, beta, eps, xn, stats, x_copy, st);
  if (x_dtype == CRF_DT_BF16)
    return launch_ln_fwd_t<__nv_bfloat16>(x, sb, st_, sc, B, T_img, C, gamma, beta, eps, xn, stats, x_copy, st);
  return set_error("ln_fwd: unsupported dtype %d", x_dtype);
}

int launch_convert_tokens(const void* src, int dtype, int64_t sb, int64_t st_, int64_t sc, int B, int T_img, int C,
                          void* dst_bf16, cudaStream_t st) {
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "convert: C=%d must be a multiple of 64 in [64,1024]", C);
  if (dtype == CRF_DT_F32)
    return launch_ln_fwd_t<float>(src, sb, st_, sc, B, T_img, C, nullptr, nullptr, 0.f, dst_bf16, nullptr, nullptr, st);
  if (dtype == CRF_DT_BF16)
    return launch_ln_fwd_t<__nv_bfloat16>(src, sb, st_, sc, B, T_img, C, nullptr, nullptr, 0.f, dst_bf16, nullptr,
                                          nullptr, st);
  return set_error("convert: unsupported dtype %d", dtype);
}

int launch_ln_bwd(const float* g, const float* x, const float* stats, const float* gamma, const float* dres,
                  float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T, int C, cudaStream_t st) {
  CRF_CHECK(C % 64 == 0, "ln_bwd: C=%d must be a multiple of 64", C);
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * (12 + (dres != nullptr ? 4 : 0) + (dx_bf16 != nullptr ? 2 : 0)),
                 "ln_bwd_T%d_C%d", T, C);
  // ONE resident wave of CTAs (occupancy x SMs): the wide rows (C >= 512: 100-170 registers per thread, 1-2 CTAs per
  // SM) otherwise ran 300 CTAs as 2.03 waves = 3 rounds of latency-bound work, and every CTA ends with 2 C column
  // reductions into dgamma / dbeta
  return launch_ln_bwd_rows(g, TokenRows{}, x, stats, gamma, dres, dx, dx_bf16, dgamma, dbeta, T, C, 0, st);
}

// Stand-alone LayerNorm over contiguous (T, C) fp32 rows (the final norm_crf of a decoder stage,
// newcrf_layers.py:430-431): y fp32 or bf16, stats (mean, rstd) for the backward.  With shuffle_w > 0 the
// PixelShuffle(2) that follows the stage is folded into the store: y is the (B, 2H, 2W, C/4) NHWC map of the
// (B, H, W) token grid, W = shuffle_w.
int launch_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                         float* stats, int T, int C, cudaStream_t st, int shuffle_w) {
  const bool ps = shuffle_w > 0;
  const char* name = ps ? "layernorm_ps_fwd" : "layernorm_fwd";
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "%s: C=%d must be a multiple of 64 in [64,1024]", name, C);
  CRF_CHECK(y_dtype == CRF_DT_F32 || y_dtype == CRF_DT_BF16, "%s: unsupported output dtype %d", name, y_dtype);
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * (4 + (y_dtype == CRF_DT_F32 ? 4 : 2)), "%s_T%d_C%d", name, T, C);
  const int ctas_per_sm = ps ? 8 : 16;
  return with_rows(shuffle_w, [&](auto rows) {
    if (y_dtype == CRF_DT_F32)
      return launch_ln_fwd_rows<float, true>(x, 0, C, T, T, C, gamma, beta, eps, static_cast<float*>(y), stats, nullptr,
                                             rows, ctas_per_sm, st);
    return launch_ln_fwd_rows<float, true>(x, 0, C, T, T, C, gamma, beta, eps, static_cast<__nv_bfloat16*>(y), stats,
                                           nullptr, rows, ctas_per_sm, st);
  });
}

// Its backward; with shuffle_w > 0, g is the gradient of the shuffled NHWC map.
int launch_layernorm_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                         void* dx_bf16, float* dgamma, float* dbeta, int T, int C, cudaStream_t st, int shuffle_w) {
  const bool ps = shuffle_w > 0;
  const char* name = ps ? "layernorm_ps_bwd" : "layernorm_bwd";
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "%s: C=%d must be a multiple of 64 in [64,1024]", name, C);
  CRF_CHECK(g_dtype == CRF_DT_F32 || g_dtype == CRF_DT_BF16, "%s: unsupported gradient dtype %d", name, g_dtype);
  // the two labels keep the byte formulas they have always reported, so timings stay comparable across versions:
  // only layernorm_ps_bwd counts the bf16 twin of dx
  KernelTimer tm(st, 0.0,
                 static_cast<double>(T) * C * ((g_dtype == CRF_DT_F32 ? 4 : 2) + 8 + (ps && dx_bf16 != nullptr ? 2 : 0)),
                 "%s_T%d_C%d", name, T, C);
  const int ctas_per_sm = ps ? (C >= 512 ? 1 : 4) : 8;
  return with_rows(shuffle_w, [&](auto rows) {
    if (g_dtype == CRF_DT_F32)
      return launch_ln_bwd_rows(static_cast<const float*>(g), rows, x, stats, gamma, nullptr, dx, dx_bf16, dgamma,
                                dbeta, T, C, ctas_per_sm, st);
    return launch_ln_bwd_rows(static_cast<const __nv_bfloat16*>(g), rows, x, stats, gamma, nullptr, dx, dx_bf16, dgamma,
                              dbeta, T, C, ctas_per_sm, st);
  });
}

int launch_pixel_shuffle_nhwc(const void* src, void* dst, int dtype, int B, int H, int W, int C, int inverse,
                              cudaStream_t st) {
  CRF_CHECK(B > 0 && H > 0 && W > 0 && C > 0 && C % 4 == 0, "pixel_shuffle_nhwc: bad shape (B=%d H=%d W=%d C=%d)", B, H, W, C);
  CRF_CHECK(dtype == CRF_DT_F32 || dtype == CRF_DT_BF16, "pixel_shuffle_nhwc: unsupported dtype %d", dtype);
  int dev = 0;
  cudaGetDevice(&dev);
  const int64_t npix = static_cast<int64_t>(B) * H * W;
  int64_t blocks = (npix + 7) / 8;
  const int64_t cap = static_cast<int64_t>(num_sms(dev)) * 16;
  if (blocks > cap) blocks = cap;
  const int esz = dtype == CRF_DT_F32 ? 4 : 2;
  KernelTimer tm(st, 0.0, 2.0 * npix * C * esz, "pixel_%sshuffle_B%d_%dx%d_C%d", inverse ? "un" : "", B, H, W, C);
  const unsigned nb = static_cast<unsigned>(blocks);
  if (dtype == CRF_DT_F32) {
    if (inverse) launch_pdl((pixel_shuffle_nhwc_kernel<float, true>), nb, 256, 0, st, reinterpret_cast<const float*>(src), reinterpret_cast<float*>(dst), B, H, W, C);
    else launch_pdl((pixel_shuffle_nhwc_kernel<float, false>), nb, 256, 0, st, reinterpret_cast<const float*>(src), reinterpret_cast<float*>(dst), B, H, W, C);
  } else {
    if (inverse) launch_pdl((pixel_shuffle_nhwc_kernel<__nv_bfloat16, true>), nb, 256, 0, st, reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), B, H, W, C);
    else launch_pdl((pixel_shuffle_nhwc_kernel<__nv_bfloat16, false>), nb, 256, 0, st, reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), B, H, W, C);
  }
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_colsum_bf16(const void* g, float* out, int T, int N, cudaStream_t st) {
  CRF_CHECK(N % 8 == 0, "colsum: N must be a multiple of 8");
  CRF_CHECK((reinterpret_cast<uintptr_t>(g) & 15) == 0, "colsum: g must be 16-byte aligned");
  int dev = 0;
  cudaGetDevice(&dev);
  int bx = N / 8;                       // column octets
  if (bx > 256) bx = 256;
  int bxp = 1;
  while (bxp < bx) bxp <<= 1;           // power of two so that bx * by == 256
  bx = bxp;
  const int by = 256 / bx;
  const int gx = (N / 8 + bx - 1) / bx;
  // two CTAs per SM (see the kernel)
  int gy = (num_sms(dev) * 2 + gx - 1) / gx;
  int rows = (T + gy - 1) / gy;
  if (rows < 8 * by) rows = 8 * by;
  gy = (T + rows - 1) / rows;
  KernelTimer tm(st, 0.0, 2.0 * T * N, "colsum_T%d_N%d", T, N);
  launch_pdl(colsum_bf16_kernel, dim3(gx, gy), dim3(bx, by), 0, st, reinterpret_cast<const __nv_bfloat16*>(g), out, T, N, rows);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_cast_bf16(const float* src, void* dst, int64_t n, cudaStream_t st) {
  if (n <= 0) return 0;
  const int64_t threads = (n + 3) / 4;
  KernelTimer tm(st, 0.0, 6.0 * n, "cast_bf16_n%lld", static_cast<long long>(n));
  launch_pdl(cast_bf16_kernel, static_cast<unsigned>((threads + 255) / 256), 256, 0, st, 
      src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_cast4_bf16(const float* const src[4], void* const dst[4], const long long n[4], cudaStream_t st) {
  Cast4 c;
  long long nmax = 0, total = 0;
  for (int i = 0; i < 4; ++i) {
    c.src[i] = src[i];
    c.dst[i] = reinterpret_cast<__nv_bfloat16*>(dst[i]);
    c.n[i] = n[i];
    if (n[i] > nmax) nmax = n[i];
    total += n[i];
  }
  int dev = 0;
  cudaGetDevice(&dev);
  long long gx = (nmax / 4 + 255) / 256;
  const long long cap = num_sms(dev) * 2;   // x 4 matrices (grid.y) = 8 CTAs per SM
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  KernelTimer tm(st, 0.0, 6.0 * total, "cast4_bf16_n%lld", total);
  launch_pdl(cast4_bf16_kernel, dim3(static_cast<unsigned>(gx), 4), 256, 0, st, c);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_window_gather(const float* x, float* windows, int B, int H, int W, int C, int window, int shift,
                         cudaStream_t st) {
  WindowGeom gm(H, W, window, shift);
  window_gather_kernel<<<B * gm.nW, 256, 0, st>>>(x, windows, gm, C);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}
int launch_window_scatter(const float* windows, float* x, int B, int H, int W, int C, int window, int shift,
                          cudaStream_t st) {
  WindowGeom gm(H, W, window, shift);
  window_scatter_kernel<<<B * gm.nW, 256, 0, st>>>(windows, x, gm, C);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}
int launch_shift_mask(float* mask, int H, int W, int window, int shift, cudaStream_t st) {
  WindowGeom gm(H, W, window, shift);
  shift_mask_kernel<<<gm.nW, 256, 0, st>>>(mask, gm);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace crf
