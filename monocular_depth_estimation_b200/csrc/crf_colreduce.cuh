// Column reduction over a row-major bf16 (T, N) matrix: a channels-last activation map viewed as T = B H W rows of N
// channels.  Shared by the bias-gradient column sums (colsum_bf16_kernel, crf_misc.cu) and the BatchNorm statistics and
// backward reduction (crf_bn.cu).
#pragma once
#include "crf_ptx.cuh"

namespace crf {

// Thread (x, y) of a CTA of at most 256 threads owns the column octet c = (blockIdx.x * blockDim.x + x) * 8 (one 16-byte
// load per row and operand) and the rows r0 + y, r0 + y + blockDim.y, ... below r1, with Op::kRows rows in flight.
// The CTA then combines its row lanes through shared memory; on return the threads of row lane 0 (threadIdx.y == 0)
// hold the CTA's sums, added in the order y = 0, 1, 2, ...  Every thread of the CTA must call it.
//
// Op supplies the per-row work:
//   static constexpr int kAcc;                                 accumulators per column
//   static constexpr int kRows;                                rows in flight per thread
//   using Regs = ...;                                          what the loads of one row return
//   Regs load(int64_t off) const;                              off = r * N + c
//   void add(const Regs& w, float (&s)[kAcc][8]) const;        accumulate one row
template <typename Op>
__device__ __forceinline__ void colreduce_cta(const Op& op, int c, int N, int r0, int r1, float (&s)[Op::kAcc][8]) {
#pragma unroll
  for (int a = 0; a < Op::kAcc; ++a)
#pragma unroll
    for (int k = 0; k < 8; ++k) s[a][k] = 0.f;
  if (c < N) {
    const int by = blockDim.y;
    int r = r0 + threadIdx.y;
    constexpr int U = Op::kRows;
    for (; r + (U - 1) * by < r1; r += U * by) {
      typename Op::Regs w[U];
#pragma unroll
      for (int u = 0; u < U; ++u) w[u] = op.load(static_cast<int64_t>(r + u * by) * N + c);
#pragma unroll
      for (int u = 0; u < U; ++u) op.add(w[u], s);
    }
    for (; r < r1; r += by) op.add(op.load(static_cast<int64_t>(r) * N + c), s);
  }
  __shared__ __align__(16) float red[256][8];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
#pragma unroll
  for (int a = 0; a < Op::kAcc; ++a) {
    if (a > 0) __syncthreads();
    *reinterpret_cast<float4*>(&red[tid][0]) = make_float4(s[a][0], s[a][1], s[a][2], s[a][3]);
    *reinterpret_cast<float4*>(&red[tid][4]) = make_float4(s[a][4], s[a][5], s[a][6], s[a][7]);
    __syncthreads();
    if (threadIdx.y == 0) {
      for (int y = 1; y < blockDim.y; ++y) {
        const float4 p = *reinterpret_cast<const float4*>(&red[y * blockDim.x + threadIdx.x][0]);
        const float4 q = *reinterpret_cast<const float4*>(&red[y * blockDim.x + threadIdx.x][4]);
        s[a][0] += p.x; s[a][1] += p.y; s[a][2] += p.z; s[a][3] += p.w;
        s[a][4] += q.x; s[a][5] += q.y; s[a][6] += q.z; s[a][7] += q.w;
      }
    }
  }
}

// The eight bf16 of a 16-byte load as floats
__device__ __forceinline__ void unpack_bf16x8(const uint4& w, float (&v)[8]) {
  v[0] = bf16_lo(w.x); v[1] = bf16_hi(w.x); v[2] = bf16_lo(w.y); v[3] = bf16_hi(w.y);
  v[4] = bf16_lo(w.z); v[5] = bf16_hi(w.z); v[6] = bf16_lo(w.w); v[7] = bf16_hi(w.w);
}

}  // namespace crf
