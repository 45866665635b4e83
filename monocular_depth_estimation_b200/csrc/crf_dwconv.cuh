// Tap map of the depthwise convolutions (crf_dwconv.cu): a k-tap axis with stride s and zero padding p = k / 2, as
// nn.Conv2d(C, C, k, s, k // 2, groups=C) has along H and along W.  Output o, tap i reads input o s - p + i; the
// border taps fall into the padding.  Host and device code: the kernels and a host-compiled test use the same maps.
#pragma once

namespace crf {

// Outputs of an axis of n inputs
__host__ __device__ constexpr int dw_out_size(int n, int k, int s) { return (n + 2 * (k / 2) - k) / s + 1; }

// The input that tap i of output o reads, or -1 where that is padding
__host__ __device__ inline int dw_src(int o, int i, int k, int s, int n) {
  const int h = o * s - k / 2 + i;
  return h >= 0 && h < n ? h : -1;
}

// The output whose tap i reads input h, or -1 if there is none (the parity differs at stride 2, or the border)
__host__ __device__ inline int dw_dst(int h, int i, int k, int s, int n_out) {
  const int t = h + k / 2 - i;
  if (t < 0 || t % s != 0) return -1;
  return t / s < n_out ? t / s : -1;
}

// A thread's run of Q consecutive pixels along W, as compile-time tables.
//   Forward and weight gradient: outputs o0 .. o0 + Q - 1 read the kIn inputs o0 s - p + c, c = 0 .. kIn - 1; output q
//   takes input c through tap fwd_tap(q, c) (-1: none).
//   Input gradient: inputs h0 .. h0 + Q - 1 with h0 % s == 0 gather the outputs h0 / s + d, d = kLo .. kHi; input q
//   takes output d through tap dgrad_tap(q, d) (-1: none).
// Inputs and outputs past the axis' ends are zero: the kernels load zeros there and store nothing.
template <int K, int S, int Q>
struct DwRun {
  static_assert(Q % S == 0, "a run starts at a multiple of the stride");
  static constexpr int P = K / 2;
  static constexpr int kIn = (Q - 1) * S + K;
  static constexpr int kLo = -((P + S - 1) / S);   // floor(-P / S)
  static constexpr int kHi = (Q - 1 + P) / S;
  static constexpr int kOut = kHi - kLo + 1;
  __host__ __device__ static constexpr int fwd_tap(int q, int c) { return c - q * S >= 0 && c - q * S < K ? c - q * S : -1; }
  __host__ __device__ static constexpr int dgrad_tap(int q, int d) {
    return q + P - d * S >= 0 && q + P - d * S < K ? q + P - d * S : -1;
  }
};

}  // namespace crf
