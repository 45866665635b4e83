// Training-mode BatchNorm2d followed by an activation (none, ReLU, Hardswish) over channels-last bf16 maps, viewed as
// T = B H W rows of C channels: two kernels forward (statistics, apply) and two backward (reduce, elementwise).
//
// The rounding points are those of torch's act(F.batch_norm(x)) on bf16 input with fp32 parameters: the BN output z is
// rounded to bf16 before the activation, the activation's output and its gradient are rounded to bf16, and the
// expressions follow ATen's channels-last kernels (Normalization.cuh) and its ReLU / Hardswish backward.  What remains
// different from torch is the fp32 summation order of the reductions.
//
// The two reductions run on the shared column reduction and its ticketed finalisation (crf_colreduce.cuh).
#include <algorithm>

#include "crf_host.h"
#include "crf_colreduce.cuh"
#include "crf_ptx.cuh"

namespace crf {

namespace {

__device__ __forceinline__ float round_bf16(float v) { return __bfloat162float(__float2bfloat16(v)); }

// ATen batch_norm_transform_input_channels_last_kernel, rounded to the bf16 output
__device__ __forceinline__ float bn_out(float x, float m, float inv, float w, float b) {
  return round_bf16(w * (x - m) * inv + b);
}

template <int ACT>
__device__ __forceinline__ float act_fwd(float z) {
  if (ACT == CRF_ACT_RELU) return z > 0.f ? z : 0.f;
  if (ACT == CRF_ACT_HARDSWISH) return z * fminf(fmaxf(z + 3.f, 0.f), 6.f) * (1.0f / 6.0f);
  return z;
}

// torch's threshold_backward (ReLU) and hardswish_backward, rounded to bf16 like their bf16 outputs
template <int ACT>
__device__ __forceinline__ float act_bwd(float g, float z) {
  if (ACT == CRF_ACT_RELU) return z <= 0.f ? 0.f : g;
  if (ACT == CRF_ACT_HARDSWISH) return z <= -3.f ? 0.f : (z < 3.f ? round_bf16(g * ((z / 3.f) + 0.5f)) : g);
  return g;
}

// The per-channel constants of a thread's column octet (scalar loads: parameters may be views of a flat buffer)
struct Octet {
  float v[8];
  __device__ __forceinline__ void load(const float* __restrict__ p, int c) {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = __ldg(p + c + k);
  }
};

__device__ __forceinline__ uint4 pack_bf16x8(const float (&v)[8]) {
  return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}

// Forward statistics: sums of d = x - p and d^2, shifted by a per-channel pivot p (the channel's value in row 0), so that
// a channel whose mean is large against its spread loses no precision to cancellation.
struct StatsOp {
  static constexpr int kAcc = 2;
  static constexpr int kRows = 8;
  using Regs = uint4;
  const __nv_bfloat16* __restrict__ x;
  float p[8];
  __device__ __forceinline__ uint4 load(int64_t off) const { return __ldg(reinterpret_cast<const uint4*>(x + off)); }
  __device__ __forceinline__ void add(const uint4& w, float (&s)[2][8]) const {
    float v[8];
    unpack_bf16x8(w, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float d = v[k] - p[k];
      s[0][k] += d;
      s[1][k] = fmaf(d, d, s[1][k]);
    }
  }
};

// Backward reduction: dz = act'(z) dy with z recomputed from x; sums of dz and dz (x - mean)
template <int ACT>
struct BwdOp {
  static constexpr int kAcc = 2;
  static constexpr int kRows = 4;  // two operands: 128 bytes in flight per thread, as the other reductions
  struct Regs { uint4 x, g; };
  const __nv_bfloat16* __restrict__ x;
  const __nv_bfloat16* __restrict__ dy;
  Octet m, inv, w, b;
  __device__ __forceinline__ Regs load(int64_t off) const {
    return {__ldg(reinterpret_cast<const uint4*>(x + off)), __ldg(reinterpret_cast<const uint4*>(dy + off))};
  }
  __device__ __forceinline__ void add(const Regs& r, float (&s)[2][8]) const {
    float xv[8], gv[8];
    unpack_bf16x8(r.x, xv);
    unpack_bf16x8(r.g, gv);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float dz = ACT == CRF_ACT_NONE ? gv[k] : act_bwd<ACT>(gv[k], bn_out(xv[k], m.v[k], inv.v[k], w.v[k], b.v[k]));
      s[0][k] += dz;
      s[1][k] += dz * (xv[k] - m.v[k]);
    }
  }
};

__global__ void __launch_bounds__(256)
bn_stats_kernel(const __nv_bfloat16* __restrict__ x, int T, int C, int rows_per_cta, float* __restrict__ part,
                int* tickets, float eps, float momentum, float* __restrict__ save_mean, float* __restrict__ save_invstd,
                float* __restrict__ running_mean, float* __restrict__ running_var, long long* num_batches_tracked) {
  pdl_prologue();
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const int r0 = blockIdx.y * rows_per_cta;
  StatsOp op{x, {}};
  if (c < C) {
    float v[8];
    unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(x + c)), v);
#pragma unroll
    for (int k = 0; k < 8; ++k) op.p[k] = v[k];
  }
  float s[2][8];
  colreduce_cta(op, c, C, r0, min(T, r0 + rows_per_cta), s);
  store_partials(part, s, c, C);
  if (!last_of_column_group(tickets)) return;
  finalize_columns<2>(part, C, [&](int ch, const double (&sum)[2]) {
    // mean and biased variance from the shifted sums; running statistics as ATen's batch_norm_reduce_statistics_kernel
    const double n = T;
    const double pivot = __bfloat162float(x[ch]);
    const double dm = sum[0] / n;
    const double var = fmax(sum[1] / n - dm * dm, 0.0);
    const double mean = pivot + dm;
    save_mean[ch] = static_cast<float>(mean);
    save_invstd[ch] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const double mom = momentum;
    running_mean[ch] = static_cast<float>((1.0 - mom) * running_mean[ch] + mom * mean);
    running_var[ch] = static_cast<float>((1.0 - mom) * running_var[ch] + mom * (var * n / (n - 1.0)));
  });
  if (blockIdx.x == 0 && threadIdx.x == 0 && threadIdx.y == 0) *num_batches_tracked += 1;
}

template <int ACT>
__device__ __forceinline__ uint4 bn_apply_octet(const uint4& w, const Octet& m, const Octet& inv, const Octet& g,
                                                const Octet& b) {
  float v[8];
  unpack_bf16x8(w, v);
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = act_fwd<ACT>(bn_out(v[k], m.v[k], inv.v[k], g.v[k], b.v[k]));
  return pack_bf16x8(v);
}

// y = act(bf16(w (x - mean) invstd + b)); thread (x, y) owns a column octet and every blockDim.y-th row of its CTA's
// row block, four rows in flight
template <int ACT>
__global__ void __launch_bounds__(256)
bn_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, const float* __restrict__ mean,
                const float* __restrict__ invstd, const float* __restrict__ weight, const float* __restrict__ bias, int T,
                int C, int rows_per_cta) {
  pdl_prologue();
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (c >= C) return;
  Octet m, inv, g, b;
  m.load(mean, c); inv.load(invstd, c); g.load(weight, c); b.load(bias, c);
  const int by = blockDim.y;
  const int r1 = min(T, static_cast<int>(blockIdx.y + 1) * rows_per_cta);
  int r = blockIdx.y * rows_per_cta + threadIdx.y;
  for (; r + 3 * by < r1; r += 4 * by) {
    uint4 w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) w[u] = __ldg(reinterpret_cast<const uint4*>(x + static_cast<int64_t>(r + u * by) * C + c));
#pragma unroll
    for (int u = 0; u < 4; ++u)
      *reinterpret_cast<uint4*>(y + static_cast<int64_t>(r + u * by) * C + c) = bn_apply_octet<ACT>(w[u], m, inv, g, b);
  }
  for (; r < r1; r += by) {
    const int64_t off = static_cast<int64_t>(r) * C + c;
    *reinterpret_cast<uint4*>(y + off) = bn_apply_octet<ACT>(__ldg(reinterpret_cast<const uint4*>(x + off)), m, inv, g, b);
  }
}

template <int ACT>
__global__ void __launch_bounds__(256, 2)
bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                     const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ weight,
                     const float* __restrict__ bias, int T, int C, int rows_per_cta, float* __restrict__ part,
                     int* tickets, float* __restrict__ sums, float* __restrict__ dweight, float* __restrict__ dbias) {
  pdl_prologue();
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const int r0 = blockIdx.y * rows_per_cta;
  BwdOp<ACT> op{x, dy, {}, {}, {}, {}};
  if (c < C) {
    op.m.load(mean, c); op.inv.load(invstd, c); op.w.load(weight, c); op.b.load(bias, c);
  }
  float s[2][8];
  colreduce_cta(op, c, C, r0, min(T, r0 + rows_per_cta), s);
  store_partials(part, s, c, C);
  if (!last_of_column_group(tickets)) return;
  finalize_columns<2>(part, C, [&](int ch, const double (&sum)[2]) {
    // sums = (sum_dy, sum_dy_xmu) as ATen keeps them; dweight = sum_dy_xmu * invstd, dbias = sum_dy
    const float sum_dy = static_cast<float>(sum[0]), sum_dy_xmu = static_cast<float>(sum[1]);
    sums[ch] = sum_dy;
    sums[C + ch] = sum_dy_xmu;
    dbias[ch] = sum_dy;
    dweight[ch] = sum_dy_xmu * invstd[ch];
  });
}

// ATen batch_norm_backward_elemt_channels_last_kernel on dz = bf16(act'(z) dy)
template <int ACT>
__device__ __forceinline__ uint4 bn_bwd_octet(const uint4& xw, const uint4& gw, const Octet& m, const Octet& inv,
                                              const Octet& w, const Octet& b, const Octet& m_dy, const Octet& f1,
                                              const Octet& f2) {
  float xv[8], gv[8];
  unpack_bf16x8(xw, xv);
  unpack_bf16x8(gw, gv);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float dz = ACT == CRF_ACT_NONE ? gv[k] : act_bwd<ACT>(gv[k], bn_out(xv[k], m.v[k], inv.v[k], w.v[k], b.v[k]));
    gv[k] = (dz - m_dy.v[k] - (xv[k] - m.v[k]) * f1.v[k]) * f2.v[k];
  }
  return pack_bf16x8(gv);
}

template <int ACT>
__global__ void __launch_bounds__(256)
bn_bwd_elemt_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                    const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ weight,
                    const float* __restrict__ bias, const float* __restrict__ sums, float norm_fct, int T, int C,
                    int rows_per_cta, __nv_bfloat16* __restrict__ dx) {
  pdl_prologue();
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (c >= C) return;
  Octet m, inv, w, b, m_dy, f1, f2;
  m.load(mean, c); inv.load(invstd, c); w.load(weight, c); b.load(bias, c);
  m_dy.load(sums, c); f1.load(sums + C, c);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    m_dy.v[k] = m_dy.v[k] * norm_fct;
    f2.v[k] = w.v[k] * inv.v[k];
    f1.v[k] = inv.v[k] * inv.v[k] * f1.v[k] * norm_fct;
  }
  const int by = blockDim.y;
  const int r1 = min(T, static_cast<int>(blockIdx.y + 1) * rows_per_cta);
  int r = blockIdx.y * rows_per_cta + threadIdx.y;
  for (; r + 3 * by < r1; r += 4 * by) {
    uint4 xw[4], gw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t off = static_cast<int64_t>(r + u * by) * C + c;
      xw[u] = __ldg(reinterpret_cast<const uint4*>(x + off));
      gw[u] = __ldg(reinterpret_cast<const uint4*>(dy + off));
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      *reinterpret_cast<uint4*>(dx + static_cast<int64_t>(r + u * by) * C + c) =
          bn_bwd_octet<ACT>(xw[u], gw[u], m, inv, w, b, m_dy, f1, f2);
  }
  for (; r < r1; r += by) {
    const int64_t off = static_cast<int64_t>(r) * C + c;
    *reinterpret_cast<uint4*>(dx + off) = bn_bwd_octet<ACT>(__ldg(reinterpret_cast<const uint4*>(x + off)),
                                                            __ldg(reinterpret_cast<const uint4*>(dy + off)), m, inv, w,
                                                            b, m_dy, f1, f2);
  }
}

// Launch geometry of all four kernels: column groups of at most 8 octets (64 channels, one 128-byte line per row), split
// evenly; as many row lanes as fit 256 threads; row blocks of at least eight row lanes' worth, about ctas_per_sm CTAs
// per SM: two for the reductions (their partial table grows with the CTA count), four for the elementwise kernels.
// Narrow groups keep the partial table a group's last CTA sums short, and the groups finalise in parallel.
struct BnGrid {
  int bx, by, gx, gy, rows;
};
BnGrid bn_grid(int T, int C, int device, int ctas_per_sm = 2) {
  BnGrid g;
  const int oct = C / 8;
  g.gx = (oct + 7) / 8;
  g.bx = (oct + g.gx - 1) / g.gx;
  g.by = 256 / g.bx;
  const int target = (num_sms(device) * ctas_per_sm + g.gx - 1) / g.gx;
  g.rows = std::max((T + target - 1) / target, 8 * g.by);
  g.gy = (T + g.rows - 1) / g.rows;
  return g;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

size_t bn_ws_bytes(const BnGrid& g, int C) { return (2 * static_cast<size_t>(g.gy) + 2) * C * sizeof(float); }

// Argument checks that need no device, then the workspace size for the current device
int bn_check(const char* name, const void* x, const void* xo, const void* xo2, int T, int C, int act, void* ws,
             size_t ws_bytes, const int* tickets, int device) {
  CRF_CHECK(C > 0 && C % 8 == 0, "%s: C=%d must be a positive multiple of 8", name, C);
  CRF_CHECK(T >= 2, "%s: T=%d: training-mode BatchNorm needs more than one value per channel", name, T);
  CRF_CHECK(act == CRF_ACT_NONE || act == CRF_ACT_RELU || act == CRF_ACT_HARDSWISH, "%s: unknown activation %d", name, act);
  CRF_CHECK(tickets != nullptr && ws != nullptr, "%s: workspace and tickets are required", name);
  CRF_CHECK(aligned16(x) && aligned16(xo) && aligned16(xo2) && aligned16(ws),
            "%s: the bf16 maps and the workspace must be 16-byte aligned", name);
  CRF_CHECK(ws_bytes >= bn_ws_bytes(bn_grid(T, C, device), C), "%s: workspace of %zu bytes is too small (%zu needed)",
            name, ws_bytes, bn_ws_bytes(bn_grid(T, C, device), C));
  return 0;
}

template <typename F>
int with_act(int act, F&& f) {
  if (act == CRF_ACT_RELU) return f(std::integral_constant<int, CRF_ACT_RELU>());
  if (act == CRF_ACT_HARDSWISH) return f(std::integral_constant<int, CRF_ACT_HARDSWISH>());
  return f(std::integral_constant<int, CRF_ACT_NONE>());
}

}  // namespace

size_t bn_workspace_bytes(int T, int C, int device) {
  if (T < 1 || C < 8) return 0;
  return bn_ws_bytes(bn_grid(T, C, device), C);
}

int launch_bn_fwd(const void* x, void* y, const float* weight, const float* bias, float* running_mean,
                  float* running_var, long long* num_batches_tracked, float* save_mean, float* save_invstd, int T, int C,
                  float eps, float momentum, int act, void* ws, size_t ws_bytes, int* tickets, int device,
                  cudaStream_t st) {
  CRF_CHECK(x && y && weight && bias && running_mean && running_var && num_batches_tracked && save_mean && save_invstd,
            "crf_bn_fwd: null pointer");
  if (bn_check("crf_bn_fwd", x, y, y, T, C, act, ws, ws_bytes, tickets, device)) return 1;
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  const BnGrid g = bn_grid(T, C, device);
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  {
    KernelTimer tm(st, 0.0, 2.0 * T * C, "bn_stats_C%d_T%d", C, T);
    CRF_CUDA(launch_pdl(bn_stats_kernel, dim3(g.gx, g.gy), dim3(g.bx, g.by), 0, st, xb, T, C, g.rows,
                        static_cast<float*>(ws), tickets, eps, momentum, save_mean, save_invstd, running_mean,
                        running_var, num_batches_tracked));
    note_launch();
  }
  const BnGrid ge = bn_grid(T, C, device, 4);
  KernelTimer tm(st, 0.0, 4.0 * T * C, "bn_apply_C%d_T%d", C, T);
  return with_act(act, [&](auto a) {
    CRF_CUDA(launch_pdl(bn_apply_kernel<decltype(a)::value>, dim3(ge.gx, ge.gy), dim3(ge.bx, ge.by), 0, st, xb,
                        static_cast<__nv_bfloat16*>(y), save_mean, save_invstd, weight, bias, T, C, ge.rows));
    note_launch();
    return 0;
  });
}

int launch_bn_bwd(const void* x, const void* dy, const float* weight, const float* bias, const float* save_mean,
                  const float* save_invstd, void* dx, float* dweight, float* dbias, int T, int C, int act, void* ws,
                  size_t ws_bytes, int* tickets, int device, cudaStream_t st) {
  CRF_CHECK(x && dy && weight && bias && save_mean && save_invstd && dx && dweight && dbias, "crf_bn_bwd: null pointer");
  if (bn_check("crf_bn_bwd", x, dy, dx, T, C, act, ws, ws_bytes, tickets, device)) return 1;
  DeviceGuard guard(device);
  CRF_CHECK(guard.ok, "cannot select device %d", device);
  const BnGrid g = bn_grid(T, C, device);
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* dyb = static_cast<const __nv_bfloat16*>(dy);
  float* part = static_cast<float*>(ws);
  float* sums = part + 2 * static_cast<size_t>(g.gy) * C;
  return with_act(act, [&](auto a) {
    constexpr int A = decltype(a)::value;
    {
      KernelTimer tm(st, 0.0, 4.0 * T * C, "bn_bwd_reduce_C%d_T%d", C, T);
      CRF_CUDA(launch_pdl(bn_bwd_reduce_kernel<A>, dim3(g.gx, g.gy), dim3(g.bx, g.by), 0, st, xb, dyb, save_mean,
                          save_invstd, weight, bias, T, C, g.rows, part, tickets, sums, dweight, dbias));
      note_launch();
    }
    KernelTimer tm(st, 0.0, 6.0 * T * C, "bn_bwd_elemt_C%d_T%d", C, T);
    const float norm_fct = static_cast<float>(1.0 / T);
    const BnGrid ge = bn_grid(T, C, device, 4);
    CRF_CUDA(launch_pdl(bn_bwd_elemt_kernel<A>, dim3(ge.gx, ge.gy), dim3(ge.bx, ge.by), 0, st, xb, dyb, save_mean,
                        save_invstd, weight, bias, sums, norm_fct, T, C, ge.rows, static_cast<__nv_bfloat16*>(dx)));
    note_launch();
    return 0;
  });
}

}  // namespace crf
