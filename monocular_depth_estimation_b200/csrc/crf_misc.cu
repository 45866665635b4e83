// Memory-bound helper kernels of the CRF block: LayerNorm forward (with the NCHW-view -> token-major layout
// change folded in), LayerNorm backward (with the residual add and the gamma/beta reductions folded in), bias
// gradient column sums, dtype casts, and the stand-alone window gather / scatter / mask used by the bit-exact
// index tests.  All of these are HBM-bound: coalesced, vectorised accesses, warp-shuffle reductions.
#include "crf_host.h"
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
// exactly once, two-pass mean / variance like torch's kernel.
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

template <typename TIn, int NCH, bool DO_LN, typename TOut = __nv_bfloat16>
__global__ void __launch_bounds__(256)
ln_fwd_rows_kernel(const TIn* __restrict__ x, int64_t sb, int64_t st, int T_img, int64_t T,
                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                   TOut* __restrict__ xn, float* __restrict__ stats, float* __restrict__ x_copy) {
  pdl_prologue();
  constexpr int C = 64 * NCH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t warps_total = static_cast<int64_t>(gridDim.x) * 8;
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * 8 + warp; t < T; t += warps_total) {
    const int64_t b = t / T_img;
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
      if (x_copy != nullptr) *reinterpret_cast<float2*>(x_copy + t * C + c) = v[k];
      float a0 = v[k].x, a1 = v[k].y;
      if (DO_LN) {
        const float2 g = __ldg(reinterpret_cast<const float2*>(gamma + c));
        const float2 be = __ldg(reinterpret_cast<const float2*>(beta + c));
        a0 = (a0 - mean) * rstd * g.x + be.x;
        a1 = (a1 - mean) * rstd * g.y + be.y;
      }
      store2(xn + t * C + c, a0, a1);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward.  One warp per token row (grid-stride); each lane owns channels {2*lane + 64k, +1}.
//   dx = rstd * (g*gamma - mean_c(g*gamma) - xhat * mean_c(g*gamma*xhat)) + dres
//   dgamma += sum_t g * xhat,  dbeta += sum_t g
// ------------------------------------------------------------------------------------------------
template <int NCH, typename TG = float>  // C = 64 * NCH
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const TG* __restrict__ g, const float* __restrict__ x, const float* __restrict__ stats,
              const float* __restrict__ gamma, const float* __restrict__ dres, float* __restrict__ dx,
              __nv_bfloat16* __restrict__ dx_bf16, float* __restrict__ dgamma, float* __restrict__ dbeta, int T) {
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
    const TG* gr = g + static_cast<int64_t>(t) * C;
    const float* xr = x + static_cast<int64_t>(t) * C;
    float2 gv[NCH], xh[NCH];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      gv[k] = load2(gr + 64 * k + 2 * lane);
      const float2 xv = __ldg(reinterpret_cast<const float2*>(xr + 64 * k + 2 * lane));
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
// out[n] += sum_t g[t,n], g bf16 (T,N).  Thread owns eight adjacent columns (one 16-byte load per row) and keeps eight
// rows in flight (128 B per thread, 32 KB per CTA); a CTA covers up to 2048 columns x a row chunk, the row lanes are
// combined through shared memory, then two vector reductions per thread of row lane 0.  Two CTAs per SM: the atomics at
// the end are per CTA, so more CTAs cost more than they hide (6 CTAs per SM: 2.5x slower at N >= 256, measured).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const __nv_bfloat16* __restrict__ g, float* __restrict__ out, int T, int N, int rows_per_cta) {
  pdl_prologue();
  __shared__ __align__(16) float red[256][8];
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(T, r0 + rows_per_cta);
  float s[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = 0.f;
  if (c < N) {
    const int by = blockDim.y;
    const int64_t step = static_cast<int64_t>(by) * N;
    const __nv_bfloat16* p = g + static_cast<int64_t>(r0 + threadIdx.y) * N + c;
    int r = r0 + threadIdx.y;
    for (; r + 7 * by < r1; r += 8 * by, p += 8 * step) {
      uint4 w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = __ldg(reinterpret_cast<const uint4*>(p + u * step));
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        s[0] += bf16_lo(w[u].x); s[1] += bf16_hi(w[u].x); s[2] += bf16_lo(w[u].y); s[3] += bf16_hi(w[u].y);
        s[4] += bf16_lo(w[u].z); s[5] += bf16_hi(w[u].z); s[6] += bf16_lo(w[u].w); s[7] += bf16_hi(w[u].w);
      }
    }
    for (; r < r1; r += by, p += step) {
      const uint4 w = __ldg(reinterpret_cast<const uint4*>(p));
      s[0] += bf16_lo(w.x); s[1] += bf16_hi(w.x); s[2] += bf16_lo(w.y); s[3] += bf16_hi(w.y);
      s[4] += bf16_lo(w.z); s[5] += bf16_hi(w.z); s[6] += bf16_lo(w.w); s[7] += bf16_hi(w.w);
    }
  }
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  *reinterpret_cast<float4*>(&red[tid][0]) = make_float4(s[0], s[1], s[2], s[3]);
  *reinterpret_cast<float4*>(&red[tid][4]) = make_float4(s[4], s[5], s[6], s[7]);
  __syncthreads();
  if (threadIdx.y == 0 && c < N) {
    float4 a = make_float4(s[0], s[1], s[2], s[3]), b = make_float4(s[4], s[5], s[6], s[7]);
    for (int y = 1; y < blockDim.y; ++y) {
      const float4 p = *reinterpret_cast<const float4*>(&red[y * blockDim.x + threadIdx.x][0]);
      const float4 q = *reinterpret_cast<const float4*>(&red[y * blockDim.x + threadIdx.x][4]);
      a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
      b.x += q.x; b.y += q.y; b.z += q.z; b.w += q.w;
    }
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
    int dev = 0;
    cudaGetDevice(&dev);
    const int64_t T = static_cast<int64_t>(B) * T_img;
    int blocks = static_cast<int>((T + 7) / 8);
    const int cap = num_sms(dev) * 16;
    if (blocks > cap) blocks = cap;
    const TIn* xp = reinterpret_cast<const TIn*>(x);
    __nv_bfloat16* xnp = reinterpret_cast<__nv_bfloat16*>(xn);
#define CRF_LNF(NCH)                                                                                                  \
  case NCH:                                                                                                           \
    if (gamma != nullptr)                                                                                             \
      launch_pdl((ln_fwd_rows_kernel<TIn, NCH, true>), blocks, 256, 0, st, xp, sb, st_, T_img, T, gamma, beta, eps, xnp, stats, x_copy); \
    else                                                                                                              \
      launch_pdl((ln_fwd_rows_kernel<TIn, NCH, false>), blocks, 256, 0, st, xp, sb, st_, T_img, T, nullptr, nullptr, eps, xnp, nullptr, x_copy); \
    break;
    switch (C / 64) {
      CRF_LNF(1) CRF_LNF(2) CRF_LNF(3) CRF_LNF(4) CRF_LNF(5) CRF_LNF(6) CRF_LNF(7) CRF_LNF(8) CRF_LNF(9) CRF_LNF(10)
      CRF_LNF(11) CRF_LNF(12) CRF_LNF(13) CRF_LNF(14) CRF_LNF(15) CRF_LNF(16)
      default: return set_error("ln_fwd: unsupported C=%d for the row kernel", C);
    }
#undef CRF_LNF
    CRF_CUDA(cudaGetLastError());
    note_launch();
    return 0;
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
  int dev = 0;
  cudaGetDevice(&dev);
  // one warp per row, grid-stride; ONE resident wave of CTAs (occupancy x SMs): the wide rows (C >= 512: 100-170
  // registers per thread, 1-2 CTAs per SM) otherwise ran 300 CTAs as 2.03 waves = 3 rounds of latency-bound work, and
  // every CTA ends with 2 C column reductions into dgamma / dbeta
  const int sms = num_sms(dev);
  __nv_bfloat16* dxb = reinterpret_cast<__nv_bfloat16*>(dx_bf16);
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * (12 + (dres != nullptr ? 4 : 0) + (dx_bf16 != nullptr ? 2 : 0)),
                 "ln_bwd_T%d_C%d", T, C);
#define CRF_LNB(NCH)                                                                                         \
  case NCH: {                                                                                                \
    static int occ = 0;                                                                                      \
    if (occ == 0) {                                                                                          \
      int o = 0;                                                                                             \
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, ln_bwd_kernel<NCH, float>, 256, 0) != cudaSuccess || o < 1) o = 1; \
      occ = o > 8 ? 8 : o;                                                                                   \
    }                                                                                                        \
    int blocks = (T + 7) / 8;                                                                                \
    if (blocks > sms * occ) blocks = sms * occ;                                                              \
    launch_pdl((ln_bwd_kernel<NCH>), blocks, 256, 0, st, g, x, stats, gamma, dres, dx, dxb, dgamma, dbeta, T);         \
    break;                                                                                                   \
  }
  switch (C / 64) {
    CRF_LNB(1) CRF_LNB(2) CRF_LNB(3) CRF_LNB(4) CRF_LNB(5) CRF_LNB(6) CRF_LNB(7) CRF_LNB(8) CRF_LNB(9) CRF_LNB(10)
    CRF_LNB(11) CRF_LNB(12) CRF_LNB(13) CRF_LNB(14) CRF_LNB(15) CRF_LNB(16)
    default: return set_error("ln_bwd: unsupported C=%d", C);
  }
#undef CRF_LNB
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// The closing LayerNorm of a decoder stage with the PixelShuffle(2) that follows it folded into its store / load
// (model_mobileV3_large_newCRFs.py:116-120: `PixelShuffle(2)` between the stages, fed by newcrf_layers.py:430-432).
// Token (b, h, w), channel c = 4 k' + 2 i + j  <->  NHWC element (b, 2h + i, 2w + j, k') of the (B, 2H, 2W, C/4) map.
// Same arithmetic, in the same order, as ln_fwd_rows_kernel / ln_bwd_kernel (one warp per row, lane owns channels
// {2 lane + 64 k, +1}): a lane's two channels are the j = 0 / 1 neighbours of one output row i = lane & 1.
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void store1(T* p, float v);
template <>
__device__ __forceinline__ void store1<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void store1<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16(v); }
__device__ __forceinline__ float load1(const float* p) { return __ldg(p); }
__device__ __forceinline__ float load1(const __nv_bfloat16* p) { return __bfloat162float(*p); }

template <int NCH, typename TOut>
__global__ void __launch_bounds__(256)
layernorm_ps_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                        float eps, TOut* __restrict__ y, float* __restrict__ stats, int T, int H, int W) {
  pdl_prologue();
  constexpr int C = 64 * NCH, C4 = C / 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warps_total = gridDim.x * 8;
  for (int t = blockIdx.x * 8 + warp; t < T; t += warps_total) {
    const float* row = x + static_cast<int64_t>(t) * C;
    float2 v[NCH];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      v[k] = load2(row + 64 * k + 2 * lane);
      s += v[k].x + v[k].y;
    }
    const float mean = warp_sum(s) * (1.0f / C);
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const float d0 = v[k].x - mean, d1 = v[k].y - mean;
      q += d0 * d0 + d1 * d1;
    }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / C) + eps);
    if (lane == 0) {
      stats[2 * t] = mean;
      stats[2 * t + 1] = rstd;
    }
    const int w = t % W, bh = t / W, h = bh % H, b = bh / H;
    const int64_t pix = (static_cast<int64_t>(b) * 2 * H + 2 * h + (lane & 1)) * 2 * W + 2 * w;   // (i = lane & 1, j = 0)
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = 64 * k + 2 * lane;
      const float2 g = __ldg(reinterpret_cast<const float2*>(gamma + c));
      const float2 be = __ldg(reinterpret_cast<const float2*>(beta + c));
      const int kp = 16 * k + (lane >> 1);
      store1(y + pix * C4 + kp, (v[k].x - mean) * rstd * g.x + be.x);
      store1(y + (pix + 1) * C4 + kp, (v[k].y - mean) * rstd * g.y + be.y);
    }
  }
}

template <int NCH, typename TG>
__global__ void __launch_bounds__(256)
layernorm_ps_bwd_kernel(const TG* __restrict__ g, const float* __restrict__ x, const float* __restrict__ stats,
                        const float* __restrict__ gamma, float* __restrict__ dx, __nv_bfloat16* __restrict__ dx_bf16,
                        float* __restrict__ dgamma, float* __restrict__ dbeta, int T, int H, int W) {
  pdl_prologue();
  constexpr int C = 64 * NCH, C4 = C / 4;
  __shared__ float red[8][64];
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
    const float* xr = x + static_cast<int64_t>(t) * C;
    const int w = t % W, bh = t / W, h = bh % H, b = bh / H;
    const int64_t pix = (static_cast<int64_t>(b) * 2 * H + 2 * h + (lane & 1)) * 2 * W + 2 * w;
    float2 gv[NCH], xh[NCH];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int kp = 16 * k + (lane >> 1);
      gv[k] = make_float2(load1(g + pix * C4 + kp), load1(g + (pix + 1) * C4 + kp));
      const float2 xv = __ldg(reinterpret_cast<const float2*>(xr + 64 * k + 2 * lane));
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
      const float o0 = rstd * (gv[k].x - s1 - xh[k].x * s2);
      const float o1 = rstd * (gv[k].y - s1 - xh[k].y * s2);
      const int64_t off = static_cast<int64_t>(t) * C + 64 * k + 2 * lane;
      if (dx != nullptr) *reinterpret_cast<float2*>(dx + off) = make_float2(o0, o1);
      if (dx_bf16 != nullptr) *reinterpret_cast<uint32_t*>(dx_bf16 + off) = pack_bf16(o0, o1);
    }
  }
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    for (int pass = 0; pass < 2; ++pass) {
      const float2 v = pass == 0 ? dga[k] : dbe[k];
      red[warp][2 * lane] = v.x;
      red[warp][2 * lane + 1] = v.y;
      __syncthreads();
      if (threadIdx.x < 64) {
        float s = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) s += red[w8][threadIdx.x];
        atomicAdd((pass == 0 ? dgamma : dbeta) + 64 * k + threadIdx.x, s);
      }
      __syncthreads();
    }
  }
}

// Stand-alone LayerNorm over contiguous (T, C) fp32 rows (the final norm_crf of a decoder stage,
// newcrf_layers.py:430-431): y fp32 or bf16, stats (mean, rstd) for the backward.
int launch_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                         float* stats, int T, int C, cudaStream_t st) {
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "layernorm_fwd: C=%d must be a multiple of 64 in [64,1024]", C);
  CRF_CHECK(y_dtype == CRF_DT_F32 || y_dtype == CRF_DT_BF16, "layernorm_fwd: unsupported output dtype %d", y_dtype);
  int dev = 0;
  cudaGetDevice(&dev);
  int blocks = (T + 7) / 8;
  const int cap = num_sms(dev) * 16;
  if (blocks > cap) blocks = cap;
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * (4 + (y_dtype == CRF_DT_F32 ? 4 : 2)), "layernorm_fwd_T%d_C%d", T, C);
#define CRF_LNS(NCH)                                                                                                   \
  case NCH:                                                                                                            \
    if (y_dtype == CRF_DT_F32)                                                                                         \
      launch_pdl((ln_fwd_rows_kernel<float, NCH, true, float>), blocks, 256, 0, st, x, 0, C, T, T, gamma, beta, eps,             \
                                                                            reinterpret_cast<float*>(y), stats, nullptr); \
    else                                                                                                               \
      launch_pdl((ln_fwd_rows_kernel<float, NCH, true, __nv_bfloat16>), blocks, 256, 0, st,                                      \
          x, 0, C, T, T, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(y), stats, nullptr);                       \
    break;
  switch (C / 64) {
    CRF_LNS(1) CRF_LNS(2) CRF_LNS(3) CRF_LNS(4) CRF_LNS(5) CRF_LNS(6) CRF_LNS(7) CRF_LNS(8) CRF_LNS(9) CRF_LNS(10)
    CRF_LNS(11) CRF_LNS(12) CRF_LNS(13) CRF_LNS(14) CRF_LNS(15) CRF_LNS(16)
    default: return set_error("layernorm_fwd: unsupported C=%d", C);
  }
#undef CRF_LNS
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_layernorm_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                         void* dx_bf16, float* dgamma, float* dbeta, int T, int C, cudaStream_t st) {
  __nv_bfloat16* dxb = reinterpret_cast<__nv_bfloat16*>(dx_bf16);
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "layernorm_bwd: C=%d must be a multiple of 64 in [64,1024]", C);
  CRF_CHECK(g_dtype == CRF_DT_F32 || g_dtype == CRF_DT_BF16, "layernorm_bwd: unsupported gradient dtype %d", g_dtype);
  int dev = 0;
  cudaGetDevice(&dev);
  int blocks = (T + 7) / 8;
  const int cap = num_sms(dev) * 8;
  if (blocks > cap) blocks = cap;
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * (8 + (g_dtype == CRF_DT_F32 ? 4 : 2)), "layernorm_bwd_T%d_C%d", T, C);
#define CRF_LNSB(NCH)                                                                                                  \
  case NCH:                                                                                                            \
    if (g_dtype == CRF_DT_F32)                                                                                         \
      launch_pdl((ln_bwd_kernel<NCH, float>), blocks, 256, 0, st, reinterpret_cast<const float*>(g), x, stats, gamma, nullptr,   \
                                                        dx, dxb, dgamma, dbeta, T);                                    \
    else                                                                                                               \
      launch_pdl((ln_bwd_kernel<NCH, __nv_bfloat16>), blocks, 256, 0, st, reinterpret_cast<const __nv_bfloat16*>(g), x, stats,    \
                                                                gamma, nullptr, dx, dxb, dgamma, dbeta, T);            \
    break;
  switch (C / 64) {
    CRF_LNSB(1) CRF_LNSB(2) CRF_LNSB(3) CRF_LNSB(4) CRF_LNSB(5) CRF_LNSB(6) CRF_LNSB(7) CRF_LNSB(8) CRF_LNSB(9)
    CRF_LNSB(10) CRF_LNSB(11) CRF_LNSB(12) CRF_LNSB(13) CRF_LNSB(14) CRF_LNSB(15) CRF_LNSB(16)
    default: return set_error("layernorm_bwd: unsupported C=%d", C);
  }
#undef CRF_LNSB
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

// The closing LayerNorm with the following PixelShuffle(2) folded in: y / g are (B, 2H, 2W, C/4) NHWC maps.
int launch_layernorm_ps_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y, int y_dtype,
                            float* stats, int B, int H, int W, int C, cudaStream_t st) {
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "layernorm_ps_fwd: C=%d must be a multiple of 64 in [64,1024]", C);
  CRF_CHECK(y_dtype == CRF_DT_F32 || y_dtype == CRF_DT_BF16, "layernorm_ps_fwd: unsupported output dtype %d", y_dtype);
  int dev = 0;
  cudaGetDevice(&dev);
  const int T = B * H * W;
  int blocks = (T + 7) / 8;
  const int cap = num_sms(dev) * 8;
  if (blocks > cap) blocks = cap;
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * (4 + (y_dtype == CRF_DT_F32 ? 4 : 2)), "layernorm_ps_fwd_T%d_C%d", T, C);
#define CRF_LPS(NCH)                                                                                                    \
  case NCH:                                                                                                             \
    if (y_dtype == CRF_DT_F32)                                                                                          \
      launch_pdl((layernorm_ps_fwd_kernel<NCH, float>), blocks, 256, 0, st, x, gamma, beta, eps, reinterpret_cast<float*>(y), stats, \
                                                                   T, H, W);                                            \
    else                                                                                                                \
      launch_pdl((layernorm_ps_fwd_kernel<NCH, __nv_bfloat16>), blocks, 256, 0, st, x, gamma, beta, eps,                          \
                                                                           reinterpret_cast<__nv_bfloat16*>(y), stats, T, H, W); \
    break;
  switch (C / 64) {
    CRF_LPS(1) CRF_LPS(2) CRF_LPS(3) CRF_LPS(4) CRF_LPS(5) CRF_LPS(6) CRF_LPS(7) CRF_LPS(8) CRF_LPS(9) CRF_LPS(10)
    CRF_LPS(11) CRF_LPS(12) CRF_LPS(13) CRF_LPS(14) CRF_LPS(15) CRF_LPS(16)
    default: return set_error("layernorm_ps_fwd: unsupported C=%d", C);
  }
#undef CRF_LPS
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_layernorm_ps_bwd(const void* g, int g_dtype, const float* x, const float* stats, const float* gamma, float* dx,
                            void* dx_bf16, float* dgamma, float* dbeta, int B, int H, int W, int C, cudaStream_t st) {
  CRF_CHECK(C % 64 == 0 && C >= 64 && C <= 1024, "layernorm_ps_bwd: C=%d must be a multiple of 64 in [64,1024]", C);
  CRF_CHECK(g_dtype == CRF_DT_F32 || g_dtype == CRF_DT_BF16, "layernorm_ps_bwd: unsupported gradient dtype %d", g_dtype);
  int dev = 0;
  cudaGetDevice(&dev);
  const int T = B * H * W;
  int blocks = (T + 7) / 8;
  const int cap = num_sms(dev) * (C >= 512 ? 1 : 4);
  if (blocks > cap) blocks = cap;
  __nv_bfloat16* dxb = reinterpret_cast<__nv_bfloat16*>(dx_bf16);
  KernelTimer tm(st, 0.0, static_cast<double>(T) * C * ((g_dtype == CRF_DT_F32 ? 4 : 2) + 8 + (dx_bf16 != nullptr ? 2 : 0)),
                 "layernorm_ps_bwd_T%d_C%d", T, C);
#define CRF_LPB(NCH)                                                                                                    \
  case NCH:                                                                                                             \
    if (g_dtype == CRF_DT_F32)                                                                                          \
      launch_pdl((layernorm_ps_bwd_kernel<NCH, float>), blocks, 256, 0, st, reinterpret_cast<const float*>(g), x, stats, gamma, dx, \
                                                                   dxb, dgamma, dbeta, T, H, W);                        \
    else                                                                                                                \
      launch_pdl((layernorm_ps_bwd_kernel<NCH, __nv_bfloat16>), blocks, 256, 0, st, reinterpret_cast<const __nv_bfloat16*>(g), x,  \
                                                                           stats, gamma, dx, dxb, dgamma, dbeta, T, H, W); \
    break;
  switch (C / 64) {
    CRF_LPB(1) CRF_LPB(2) CRF_LPB(3) CRF_LPB(4) CRF_LPB(5) CRF_LPB(6) CRF_LPB(7) CRF_LPB(8) CRF_LPB(9) CRF_LPB(10)
    CRF_LPB(11) CRF_LPB(12) CRF_LPB(13) CRF_LPB(14) CRF_LPB(15) CRF_LPB(16)
    default: return set_error("layernorm_ps_bwd: unsupported C=%d", C);
  }
#undef CRF_LPB
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
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
