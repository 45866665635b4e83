// Work-decomposition arithmetic shared by host launchers and kernels (and compiled on the host by
// tests/test_sched_host.py): rows per tile of the persistent row-tiled kernels.
#pragma once

#ifndef __CUDACC__
#ifndef __host__
#define __host__
#endif
#ifndef __device__
#define __device__
#endif
#endif

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

}  // namespace crf
