// Depthwise k x k convolutions (groups == C, k = 3 or 5, stride 1 or 2, zero padding k / 2, no bias) over channels-last
// bf16 maps viewed as (B, H, W, C): forward, input gradient and weight gradient, one kernel each, no atomics.
//
// The rounding points are those of torch's bf16 autocast conv2d: the fp32 weight is rounded to bf16 on load (what
// autocast's cast produces), each output is one fp32 sum of bf16 products in a fixed tap order rounded once to bf16, and
// the weight gradient, summed in fp32 partials and double, is rounded to bf16 and widened to fp32 (cuDNN's bf16 weight
// gradient, then autocast's cast back).  Every result is bit-reproducible from run to run.
//
// All three kernels share one geometry: a CTA covers a channel group of at most eight octets (64 channels, one 128-byte
// line per pixel), thread (x, y) owns the octet x of the group, and its row lane y takes work items y, y + blockDim.y,
// ... of the CTA's item block.  A work item is a run of kRun consecutive pixels of one row (crf_dwconv.cuh: DwRun); the
// run's input loads hit L1 for the taps its neighbours share, and its k weight octets per tap row come from shared
// memory, where every lane of a warp reads one of at most eight addresses.
//
// The weight gradient runs one grid slice per tap row (blockIdx.z), so that a thread's k x 8 partial sums stay in
// registers; the slices of a work item run side by side and share its loads in L2.  A CTA combines its row lanes in
// order, writes one partial per tap to the workspace and finalises through its column group's ticket
// (crf_colreduce.cuh).
#include <algorithm>

#include "crf_host.h"
#include "crf_colreduce.cuh"
#include "crf_dwconv.cuh"
#include "crf_ptx.cuh"

namespace crf {

namespace {

constexpr int kRun = 4;  // pixels per work item

__device__ __forceinline__ float round_bf16(float v) { return __bfloat162float(__float2bfloat16(v)); }

__device__ __forceinline__ uint4 load_or_zero(const __nv_bfloat16* p, bool ok) {
  return ok ? __ldg(reinterpret_cast<const uint4*>(p)) : make_uint4(0, 0, 0, 0);
}

__device__ __forceinline__ void store_bf16x8(__nv_bfloat16* p, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(p) =
      make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}

// The CTA's weights, rounded to bf16: ws[tap * ncol + col] for channel c0 + col (zero past C).  Ends with a barrier.
template <int K>
__device__ __forceinline__ void stage_weights(const float* __restrict__ weight, float* ws, int c0, int ncol, int C) {
  const int nthr = blockDim.x * blockDim.y;
  for (int e = threadIdx.y * blockDim.x + threadIdx.x; e < K * K * ncol; e += nthr) {
    const int col = e / (K * K), tap = e - col * (K * K);   // consecutive threads: consecutive taps of one channel
    const int c = c0 + col;
    ws[tap * ncol + col] = c < C ? round_bf16(__ldg(weight + static_cast<int64_t>(c) * K * K + tap)) : 0.f;
  }
  __syncthreads();
}

// The thread's octet of the K weights of tap row i
template <int K>
__device__ __forceinline__ void weight_row(const float* ws, int i, int ncol, float (&w)[K][8]) {
  const float* p = ws + i * K * ncol + threadIdx.x * 8;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const float4 a = *reinterpret_cast<const float4*>(p + j * ncol);
    const float4 b = *reinterpret_cast<const float4*>(p + j * ncol + 4);
    w[j][0] = a.x; w[j][1] = a.y; w[j][2] = a.z; w[j][3] = a.w;
    w[j][4] = b.x; w[j][5] = b.y; w[j][6] = b.z; w[j][7] = b.w;
  }
}

// y[b, oh, ow, c] = bf16(sum over i, j (in that order) of x[b, oh S - p + i, ow S - p + j, c] bf16(w[c, i, j]))
template <int K, int S>
__global__ void __launch_bounds__(256, 2)
dw_fwd_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ weight, __nv_bfloat16* __restrict__ y,
              int H, int W, int C, int Ho, int Wo, int rows, int items_per_cta) {
  using R = DwRun<K, S, kRun>;
  __shared__ __align__(16) float ws[K * K * 64];
  pdl_prologue();
  const int ncol = blockDim.x * 8;
  const int c0 = blockIdx.x * ncol;
  stage_weights<K>(weight, ws, c0, ncol, C);
  const int c = c0 + threadIdx.x * 8;
  if (c >= C) return;
  const int runs = (Wo + kRun - 1) / kRun;
  const int e1 = min(rows * runs, static_cast<int>(blockIdx.y + 1) * items_per_cta);
  for (int n = blockIdx.y * items_per_cta + threadIdx.y; n < e1; n += blockDim.y) {
    const int r = n / runs, o0 = (n - r * runs) * kRun;
    const int b = r / Ho, oh = r - b * Ho;
    float acc[kRun][8];
#pragma unroll
    for (int q = 0; q < kRun; ++q)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[q][k] = 0.f;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const int ih = oh * S - R::P + i;
      if (ih < 0 || ih >= H) continue;
      const __nv_bfloat16* xr = x + static_cast<int64_t>(b * H + ih) * W * C + c;
      const int iw0 = o0 * S - R::P;
      uint4 v[R::kIn];
#pragma unroll
      for (int cc = 0; cc < R::kIn; ++cc)
        v[cc] = load_or_zero(xr + static_cast<int64_t>(iw0 + cc) * C, iw0 + cc >= 0 && iw0 + cc < W);
      float w[K][8];
      weight_row<K>(ws, i, ncol, w);
#pragma unroll
      for (int cc = 0; cc < R::kIn; ++cc) {
        float f[8];
        unpack_bf16x8(v[cc], f);
#pragma unroll
        for (int q = 0; q < kRun; ++q) {
          const int j = R::fwd_tap(q, cc);
          if (j < 0) continue;
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[q][k] = fmaf(f[k], w[j][k], acc[q][k]);
        }
      }
    }
    __nv_bfloat16* yr = y + static_cast<int64_t>(b * Ho + oh) * Wo * C + c;
#pragma unroll
    for (int q = 0; q < kRun; ++q)
      if (o0 + q < Wo) store_bf16x8(yr + static_cast<int64_t>(o0 + q) * C, acc[q]);
  }
}

// dx[b, h, w, c] = bf16(sum over the taps (i, j) whose output (oh, ow) reads (h, w) of dy[b, oh, ow, c] bf16(w[c, i, j])),
// i ascending, then j descending.  Gather form: a thread owns a run of inputs.
template <int K, int S>
__global__ void __launch_bounds__(256, 2)
dw_dgrad_kernel(const __nv_bfloat16* __restrict__ dy, const float* __restrict__ weight, __nv_bfloat16* __restrict__ dx,
                int H, int W, int C, int Ho, int Wo, int rows, int items_per_cta) {
  using R = DwRun<K, S, kRun>;
  __shared__ __align__(16) float ws[K * K * 64];
  pdl_prologue();
  const int ncol = blockDim.x * 8;
  const int c0 = blockIdx.x * ncol;
  stage_weights<K>(weight, ws, c0, ncol, C);
  const int c = c0 + threadIdx.x * 8;
  if (c >= C) return;
  const int runs = (W + kRun - 1) / kRun;
  const int e1 = min(rows * runs, static_cast<int>(blockIdx.y + 1) * items_per_cta);
  for (int n = blockIdx.y * items_per_cta + threadIdx.y; n < e1; n += blockDim.y) {
    const int r = n / runs, h0 = (n - r * runs) * kRun;
    const int b = r / H, ih = r - b * H;
    float acc[kRun][8];
#pragma unroll
    for (int q = 0; q < kRun; ++q)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[q][k] = 0.f;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const int t = ih + R::P - i;
      if (t < 0 || t % S != 0 || t / S >= Ho) continue;
      const __nv_bfloat16* gr = dy + static_cast<int64_t>(b * Ho + t / S) * Wo * C + c;
      const int ow0 = h0 / S + R::kLo;
      uint4 v[R::kOut];
#pragma unroll
      for (int d = 0; d < R::kOut; ++d)
        v[d] = load_or_zero(gr + static_cast<int64_t>(ow0 + d) * C, ow0 + d >= 0 && ow0 + d < Wo);
      float w[K][8];
      weight_row<K>(ws, i, ncol, w);
#pragma unroll
      for (int d = 0; d < R::kOut; ++d) {
        float f[8];
        unpack_bf16x8(v[d], f);
#pragma unroll
        for (int q = 0; q < kRun; ++q) {
          const int j = R::dgrad_tap(q, R::kLo + d);
          if (j < 0) continue;
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[q][k] = fmaf(f[k], w[j][k], acc[q][k]);
        }
      }
    }
    __nv_bfloat16* xr = dx + static_cast<int64_t>(b * H + ih) * W * C + c;
#pragma unroll
    for (int q = 0; q < kRun; ++q)
      if (h0 + q < W) store_bf16x8(xr + static_cast<int64_t>(h0 + q) * C, acc[q]);
  }
}

// dW[c, i, j] = bf16(sum over b, oh, ow of dy[b, oh, ow, c] x[b, oh S - p + i, ow S - p + j, c]) as fp32, for the tap row
// i = blockIdx.z.  part: the (K K, gridDim.y, C) fp32 partial table; tickets: gridDim.x counters per tap row.
template <int K, int S>
__global__ void __launch_bounds__(256, 2)
dw_wgrad_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy, int H, int W, int C, int Ho,
                int Wo, int rows, int items_per_cta, float* __restrict__ part, int* tickets,
                float* __restrict__ dweight) {
  using R = DwRun<K, S, kRun>;
  pdl_prologue();
  const int i = blockIdx.z;
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  float s[K][8];
#pragma unroll
  for (int a = 0; a < K; ++a)
#pragma unroll
    for (int k = 0; k < 8; ++k) s[a][k] = 0.f;
  if (c < C) {
    const int runs = (Wo + kRun - 1) / kRun;
    const int e1 = min(rows * runs, static_cast<int>(blockIdx.y + 1) * items_per_cta);
    for (int n = blockIdx.y * items_per_cta + threadIdx.y; n < e1; n += blockDim.y) {
      const int r = n / runs, o0 = (n - r * runs) * kRun;
      const int b = r / Ho, oh = r - b * Ho;
      const __nv_bfloat16* gr = dy + static_cast<int64_t>(b * Ho + oh) * Wo * C + c;
      float g[kRun][8];
#pragma unroll
      for (int q = 0; q < kRun; ++q) unpack_bf16x8(load_or_zero(gr + static_cast<int64_t>(o0 + q) * C, o0 + q < Wo), g[q]);
      const int ih = oh * S - R::P + i;
      if (ih < 0 || ih >= H) continue;
      const __nv_bfloat16* xr = x + static_cast<int64_t>(b * H + ih) * W * C + c;
      const int iw0 = o0 * S - R::P;
      uint4 v[R::kIn];
#pragma unroll
      for (int cc = 0; cc < R::kIn; ++cc)
        v[cc] = load_or_zero(xr + static_cast<int64_t>(iw0 + cc) * C, iw0 + cc >= 0 && iw0 + cc < W);
#pragma unroll
      for (int cc = 0; cc < R::kIn; ++cc) {
        float f[8];
        unpack_bf16x8(v[cc], f);
#pragma unroll
        for (int q = 0; q < kRun; ++q) {
          const int j = R::fwd_tap(q, cc);
          if (j < 0) continue;
#pragma unroll
          for (int k = 0; k < 8; ++k) s[j][k] = fmaf(f[k], g[q][k], s[j][k]);
        }
      }
    }
  }
  combine_row_lanes(s);
  float* zpart = part + static_cast<int64_t>(i) * K * gridDim.y * C;
  store_partials(zpart, s, c, C);
  if (!last_of_column_group(tickets + blockIdx.z * gridDim.x)) return;
  finalize_columns<K>(zpart, C, [&](int ch, const double (&sum)[K]) {
#pragma unroll
    for (int j = 0; j < K; ++j)
      dweight[static_cast<int64_t>(ch) * K * K + i * K + j] = __bfloat162float(__double2bfloat16(sum[j]));
  });
}

// Launch geometry of the three kernels: column groups of at most 8 octets, split evenly; as many row lanes as fit 256
// threads; item blocks of at least one item per row lane, about ctas_per_sm CTAs per SM over the grid's gz slices.
struct DwGrid {
  int bx, by, gx, gy, gz, items_per_cta;
};
DwGrid dw_grid(int items, int C, int gz, int ctas_per_sm, int device) {
  DwGrid g;
  const int oct = C / 8;
  g.gx = (oct + 7) / 8;
  g.bx = (oct + g.gx - 1) / g.gx;
  g.by = 256 / g.bx;
  g.gz = gz;
  const int target = std::max(1, (num_sms(device) * ctas_per_sm + g.gx * gz - 1) / (g.gx * gz));
  g.items_per_cta = std::max((items + target - 1) / target, g.by);
  g.gy = (items + g.items_per_cta - 1) / g.items_per_cta;
  return g;
}

constexpr int kCtasPerSm = 2;   // the kernels' launch bounds; the wgrad partial table grows with the CTA count

DwGrid wgrad_grid(int B, int Ho, int Wo, int C, int k, int device) {
  return dw_grid(B * Ho * ((Wo + kRun - 1) / kRun), C, k, kCtasPerSm, device);
}

size_t dw_ws_bytes(const DwGrid& g, int C, int k) {
  return static_cast<size_t>(k) * k * g.gy * C * sizeof(float);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Argument checks that need no device
int dw_check(const char* name, int B, int H, int W, int C, int k, int stride) {
  CRF_CHECK(B >= 1 && H >= 1 && W >= 1, "%s: B=%d H=%d W=%d must be positive", name, B, H, W);
  CRF_CHECK(C > 0 && C % 8 == 0, "%s: C=%d must be a positive multiple of 8", name, C);
  CRF_CHECK(k == 3 || k == 5, "%s: kernel size %d is not supported (3 or 5)", name, k);
  CRF_CHECK(stride == 1 || stride == 2, "%s: stride %d is not supported (1 or 2)", name, stride);
  CRF_CHECK(static_cast<int64_t>(B) * H * W * C < (int64_t(1) << 31), "%s: the map has 2^31 elements or more", name);
  return 0;
}

template <typename F>
int with_geometry(int k, int stride, F&& f) {
  if (k == 3 && stride == 1) return f(std::integral_constant<int, 3>(), std::integral_constant<int, 1>());
  if (k == 3) return f(std::integral_constant<int, 3>(), std::integral_constant<int, 2>());
  if (stride == 1) return f(std::integral_constant<int, 5>(), std::integral_constant<int, 1>());
  return f(std::integral_constant<int, 5>(), std::integral_constant<int, 2>());
}

}  // namespace

size_t dwconv_workspace_bytes(int B, int H, int W, int C, int k, int stride, int device) {
  if (B < 1 || H < 1 || W < 1 || C < 8 || C % 8 != 0 || (k != 3 && k != 5) || (stride != 1 && stride != 2)) return 0;
  return dw_ws_bytes(wgrad_grid(B, dw_out_size(H, k, stride), dw_out_size(W, k, stride), C, k, device), C, k);
}

int launch_dwconv_fwd(const void* x, const float* weight, void* y, int B, int H, int W, int C, int k, int stride,
                      int device, cudaStream_t st) {
  CRF_CHECK(x && weight && y, "crf_dwconv_fwd: null pointer");
  if (dw_check("crf_dwconv_fwd", B, H, W, C, k, stride)) return 1;
  CRF_CHECK(aligned16(x) && aligned16(y), "crf_dwconv_fwd: the bf16 maps must be 16-byte aligned");
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  const int Ho = dw_out_size(H, k, stride), Wo = dw_out_size(W, k, stride);
  const DwGrid g = dw_grid(B * Ho * ((Wo + kRun - 1) / kRun), C, 1, kCtasPerSm, device);
  const double out = static_cast<double>(B) * Ho * Wo * C;
  KernelTimer tm(st, 2.0 * k * k * out, 2.0 * (static_cast<double>(B) * H * W * C + out) + 4.0 * C * k * k,
                 "dw_fwd_C%d_%dx%d_k%d_s%d", C, H, W, k, stride);
  return with_geometry(k, stride, [&](auto kk, auto ss) {
    CRF_CUDA(launch_pdl(dw_fwd_kernel<decltype(kk)::value, decltype(ss)::value>, dim3(g.gx, g.gy), dim3(g.bx, g.by), 0,
                        st, static_cast<const __nv_bfloat16*>(x), weight, static_cast<__nv_bfloat16*>(y), H, W, C, Ho,
                        Wo, B * Ho, g.items_per_cta));
    note_launch();
    return 0;
  });
}

int launch_dwconv_bwd(const void* x, const float* weight, const void* dy, void* dx, float* dweight, int B, int H, int W,
                      int C, int k, int stride, void* ws, size_t ws_bytes, int* tickets, int device, cudaStream_t st) {
  CRF_CHECK(x && weight && dy, "crf_dwconv_bwd: null pointer");
  CRF_CHECK(dx || dweight, "crf_dwconv_bwd: neither dx nor dweight requested");
  if (dw_check("crf_dwconv_bwd", B, H, W, C, k, stride)) return 1;
  CRF_CHECK(aligned16(x) && aligned16(dy) && aligned16(dx), "crf_dwconv_bwd: the bf16 maps must be 16-byte aligned");
  CRF_CHECK(!dweight || (tickets != nullptr && ws != nullptr),
            "crf_dwconv_bwd: workspace and tickets are required for dweight");
  CRF_CHECK(aligned16(ws), "crf_dwconv_bwd: the workspace must be 16-byte aligned");
  const int Ho = dw_out_size(H, k, stride), Wo = dw_out_size(W, k, stride);
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  const DwGrid gw = wgrad_grid(B, Ho, Wo, C, k, device);
  CRF_CHECK(!dweight || ws_bytes >= dw_ws_bytes(gw, C, k),
            "crf_dwconv_bwd: workspace of %zu bytes is too small (%zu needed)", ws_bytes, dw_ws_bytes(gw, C, k));
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* dyb = static_cast<const __nv_bfloat16*>(dy);
  const double in = static_cast<double>(B) * H * W * C, out = static_cast<double>(B) * Ho * Wo * C;
  return with_geometry(k, stride, [&](auto kk, auto ss) {
    constexpr int K = decltype(kk)::value, S = decltype(ss)::value;
    if (dx) {
      const DwGrid g = dw_grid(B * H * ((W + kRun - 1) / kRun), C, 1, kCtasPerSm, device);
      KernelTimer tm(st, 2.0 * K * K * out, 2.0 * (in + out) + 4.0 * C * K * K, "dw_dgrad_C%d_%dx%d_k%d_s%d", C, H, W, K,
                     S);
      CRF_CUDA(launch_pdl(dw_dgrad_kernel<K, S>, dim3(g.gx, g.gy), dim3(g.bx, g.by), 0, st, dyb, weight,
                          static_cast<__nv_bfloat16*>(dx), H, W, C, Ho, Wo, B * H, g.items_per_cta));
      note_launch();
    }
    if (dweight) {
      KernelTimer tm(st, 2.0 * K * K * out, 2.0 * (in + out) + 4.0 * C * K * K, "dw_wgrad_C%d_%dx%d_k%d_s%d", C, H, W,
                     K, S);
      CRF_CUDA(launch_pdl(dw_wgrad_kernel<K, S>, dim3(gw.gx, gw.gy, gw.gz), dim3(gw.bx, gw.by), 0, st, xb, dyb, H, W, C,
                          Ho, Wo, B * Ho, gw.items_per_cta, static_cast<float*>(ws), tickets, dweight));
      note_launch();
    }
    return 0;
  });
}

}  // namespace crf
