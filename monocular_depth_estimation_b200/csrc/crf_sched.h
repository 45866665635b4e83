// Work-decomposition arithmetic shared by host launchers and kernels (and compiled on the host by
// tests/test_sched_host.py and tests/test_gemm_plan_host.py): rows per tile of the persistent row-tiled kernels, and
// which GEMM kernel runs for a problem.
#pragma once

#ifndef __CUDACC__
#ifndef __host__
#define __host__
#endif
#ifndef __device__
#define __device__
#endif
#endif

#include "../../include/crf_sm100.h"

namespace crf {

// Rows per tile for a persistent kernel whose MMA tile is 128 rows: only `tm` (a multiple of 8, <= 128) rows are loaded
// and stored per tile, chosen so that the tiles fill whole rounds of `sms` CTAs (T = 38400 on 148 SMs: 300 tiles of 128
// rows are 2.03 rounds, i.e. 3; 437 tiles of 88 rows are 2.95 rounds of a 31 % shorter tile).
__host__ __device__ inline int balanced_tile_rows(int T, int sms) {
  const int full = (T + 127) / 128;
  const int g0 = full < sms ? full : sms;
  const int rows_per_cta = (T + g0 - 1) / g0;
  const int n = (rows_per_cta + 127) / 128;
  int tm = (((rows_per_cta + n - 1) / n) + 7) & ~7;
  return tm > 128 ? 128 : tm;
}

// The widest tile of the tiled GEMM (gemm_kernel<BN>, crf_gemm.cu) that divides N, a multiple of 64.
inline int gemm_tile_n(int N) { return N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 64); }

enum GemmKernel { kGemmPair, kGemmPersistent, kGemmTiled };
struct GemmPlan {
  GemmKernel kernel;
  int bn;  // kGemmTiled: the tile width BN; 0 otherwise
};

// The kernel launch_gemm runs for an M x N x K problem (a_major and split3 as in crf_gemm_args):
//  - the CTA-pair kernel (crf_gemm_pair.cu, 256 x 256 tiles): A K-major, N % 256 == 0, N >= 512, K >= 512, no split3,
//    not split-K.  Measured 15-30 % faster than the single-CTA kernels on every C >= 512 projection
//    (profiles/r02_gemm_pair.md);
//  - else the persistent kernel (crf_gemm_persist.cu, 128 x 128 tiles): A K-major, N % 128 == 0, no split3, not split-K;
//  - else the tiled kernel gemm_kernel<BN>: BN = gemm_tile_n(N), at most 128 with K-major A (the fprop / dgrad GEMMs are
//    epilogue-bound and run faster with more, narrower CTAs per SM).
inline GemmPlan plan_gemm(int /*M*/, int N, int K, int a_major, int epilogue, int split3) {
  const bool token_major = a_major == 0 && epilogue != CRF_EPI_SPLITK_F32 && !split3;
  if (token_major && N % 256 == 0 && N >= 512 && K >= 512) return {kGemmPair, 0};
  if (token_major && N % 128 == 0) return {kGemmPersistent, 0};
  const int bn = gemm_tile_n(N);
  return {kGemmTiled, a_major == 0 && bn > 128 ? 128 : bn};
}

}  // namespace crf
