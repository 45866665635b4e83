// Column reduction over a row-major bf16 (T, N) matrix: a channels-last activation map viewed as T = B H W rows of N
// channels.  Shared by the bias-gradient column sums (colsum_bf16_kernel, crf_misc.cu) and the BatchNorm statistics and
// backward reduction (crf_bn.cu); the depthwise weight gradient (crf_dwconv.cu) uses the row-lane combine, the partial
// table and the ticketed finalisation.
//
// Grid-wide reductions: every CTA writes its per-column partial sums to a workspace table and takes a ticket from its
// column group's counter; the last CTA of a group sums the partials in double, in a fixed order, and finalises the
// group's columns.  It resets the counter, so the next launch (or CUDA-graph replay) starts from zero; no CTA waits for
// another.
#pragma once
#include "crf_ptx.cuh"

namespace crf {

// Adds the per-thread sums s of every row lane (threadIdx.y) into row lane 0, in the order y = 0, 1, 2, ...  Every
// thread of the CTA (at most 256) must call it; on return the threads of row lane 0 hold the CTA's sums.
template <int NACC>
__device__ __forceinline__ void combine_row_lanes(float (&s)[NACC][8]) {
  __shared__ __align__(16) float red[256][8];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
#pragma unroll
  for (int a = 0; a < NACC; ++a) {
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
  combine_row_lanes(s);
}

// part[(a * gridDim.y + blockIdx.y) * C + c]: accumulator a of the CTA's row block
template <int NACC>
__device__ __forceinline__ void store_partials(float* __restrict__ part, const float (&s)[NACC][8], int c, int C) {
  if (threadIdx.y != 0 || c >= C) return;
#pragma unroll
  for (int a = 0; a < NACC; ++a) {
    float* dst = part + (static_cast<int64_t>(a) * gridDim.y + blockIdx.y) * C + c;
    *reinterpret_cast<float4*>(dst) = make_float4(s[a][0], s[a][1], s[a][2], s[a][3]);
    *reinterpret_cast<float4*>(dst + 4) = make_float4(s[a][4], s[a][5], s[a][6], s[a][7]);
  }
}

// True in the CTA that arrives last of its column group (blockIdx.x); that CTA resets the group's counter.
__device__ __forceinline__ bool last_of_column_group(int* tickets) {
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0 && threadIdx.y == 0) {
    last = atomicAdd(tickets + blockIdx.x, 1) == static_cast<int>(gridDim.y) - 1;
    if (last) tickets[blockIdx.x] = 0;
  }
  __syncthreads();
  if (last) __threadfence();
  return last;
}

// In the last CTA of a column group: sums each column's NACC partials over the grid's row blocks in double -- thread
// slices take every slices-th row block, then slice 0 adds the slices in order -- and calls f(c, sums) once per column.
template <int NACC, typename F>
__device__ __forceinline__ void finalize_columns(const float* part, int C, F&& f) {
  __shared__ double red[256][NACC];
  const int c0 = blockIdx.x * blockDim.x * 8;
  const int ncol = min(static_cast<int>(blockDim.x) * 8, C - c0);
  const int nthr = blockDim.x * blockDim.y;
  const int slices = nthr / ncol;  // >= 4: at most 64 columns per group
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int col = tid % ncol, sl = tid / ncol;
  double acc[NACC];
#pragma unroll
  for (int a = 0; a < NACC; ++a) acc[a] = 0.0;
  if (sl < slices) {
    const int gy = gridDim.y;
    const float* p = part + c0 + col;
    auto at = [&](int a, int y) { return __ldcg(p + (static_cast<int64_t>(a) * gy + y) * C); };
    int y = sl;
    for (; y + 7 * slices < gy; y += 8 * slices) {  // eight row blocks' loads in flight, added in row-block order
      float v[8][NACC];
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int a = 0; a < NACC; ++a) v[u][a] = at(a, y + u * slices);
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int a = 0; a < NACC; ++a) acc[a] += v[u][a];
    }
    for (; y < gy; y += slices) {
#pragma unroll
      for (int a = 0; a < NACC; ++a) acc[a] += at(a, y);
    }
  }
#pragma unroll
  for (int a = 0; a < NACC; ++a) red[tid][a] = acc[a];
  __syncthreads();
  if (tid < ncol) {
    for (int s = 1; s < slices; ++s) {
#pragma unroll
      for (int a = 0; a < NACC; ++a) acc[a] += red[s * ncol + tid][a];
    }
    f(c0 + tid, acc);
  }
}

// The eight bf16 of a 16-byte load as floats
__device__ __forceinline__ void unpack_bf16x8(const uint4& w, float (&v)[8]) {
  v[0] = bf16_lo(w.x); v[1] = bf16_hi(w.x); v[2] = bf16_lo(w.y); v[3] = bf16_hi(w.y);
  v[4] = bf16_lo(w.z); v[5] = bf16_hi(w.z); v[6] = bf16_lo(w.w); v[7] = bf16_hi(w.w);
}

}  // namespace crf
