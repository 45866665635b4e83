// Fused MLP half of a CRF block, forward:  y = x1 + fc2(GELU(fc1(LayerNorm2(x1))))
// (CRFBlock.forward, /root/reference/src/newcrf_layers.py:255 with Mlp.forward :21-27), ONE kernel for C = 128 / 256.
//
// A persistent CTA per SM loops over 128-token tiles.  The 4C-wide hidden activation never goes to HBM on the way
// from fc1 to fc2: it lives in TMEM (fc1 accumulator chunks), registers (bias + GELU) and shared memory (the bf16
// A-operand chunk of fc2), 64 hidden columns at a time, while the fc2 accumulator of the tile stays in TMEM.
//
//   warps 0-7    LayerNorm-2 prologue: eight lanes per row, fp32 rows straight from HBM (32 KB in flight per SM), row
//                statistics by three shuffles, the normalised row written as bf16 into the swizzled UMMA A-operand
//                tile (double-buffered across tiles at C = 128); training: the same smem tile is TMA-stored as `xn2`,
//                (mean, rstd) go to `stats` (both are what the backward kernels read today)
//   warps 8-15   two GELU groups (thread = accumulator row): fc1 chunk j from TMEM, + bias, exact-erf GELU in packed
//                fp32x2 arithmetic, bf16 into the A-operand chunk of fc2; training: pre-activation and activation
//                chunks leave by TMA store
//   warps 16-19  final epilogue: fc2 accumulator + bias + residual x1 (row segments prefetched into registers) -> y,
//                32-column fp32 slabs leaving by TMA store
//   warps 20/21  TMA producers: W1 / W2 chunks stream through two rings of 16 KB stages; the weights stay L2-resident
//   warps 22/23  MMA issuers: one thread issues every fc1 chunk, another every fc2 chunk, so fc1 runs ahead of fc2 as
//                far as the four TMEM chunk buffers allow (also across tile boundaries) and the GELU warps never wait
//                for a main loop
//
// TMEM: four fc1 chunk accumulators (4 x 64 columns) + the fc2 accumulator(s) (2 x 128 at C = 128, 1 x 256 at C = 256).
// Algorithmic work per token: 16 C^2 flops; HBM bytes: 8 C (x1 in, y out) + training saves 2 C + 16 C (xn2, pre, act).
#include <stdlib.h>

#include "crf_gemm_epi.cuh"
#include "crf_sched.h"

namespace crf {

namespace {

constexpr int TM = 128;  // tokens per tile (UMMA M)
constexpr int HC = 64;   // hidden columns per chunk (one 128-byte swizzle atom of bf16)
constexpr int kThreads = 768;  // 8 LayerNorm + 8 GELU + 4 final-epilogue warps, 2 TMA producers, 2 MMA issuers
constexpr int kPreBufs = 4;
constexpr int kSlab = TM * 128;  // 16 KB: 128 rows x 128 bytes

template <int C>
struct MlpPlan {
  static constexpr int NCH = C / 64;                 // 64-column atoms per normalised row
  static constexpr int NJ = 4 * C / HC;              // hidden chunks per tile
  static constexpr int kXnTile = NCH * kSlab;        // A operand of fc1: NCH atoms of 128 rows x 128 B
  static constexpr int kXnBufs = C <= 128 ? 2 : 1;
  static constexpr int NSUB = C / 128;               // ring stages per weight chunk
  static constexpr int kStage = HC * 128 * 2;        // 16 KB: W1[chunk rows, 128 k-columns] or W2[128 rows, chunk columns]
  static constexpr int kS1 = 2, kS2 = 2;             // stages of the W1 / W2 rings
  static constexpr int kYBufs = C <= 128 ? 2 : 1;
  static constexpr int kXnOff = 0;
  static constexpr int kW1Off = kXnOff + kXnBufs * kXnTile;
  static constexpr int kW2Off = kW1Off + kS1 * kStage;
  static constexpr int kActOff = kW2Off + kS2 * kStage;         // 2 x 16 KB: A operand chunks of fc2
  static constexpr int kPreOff = kActOff + 2 * kSlab;           // 2 x 16 KB: staging of the pre-activation store
  static constexpr int kOutOff = kPreOff + 2 * kSlab;           // out slab of the final epilogue
  static constexpr int kBiasOff = kOutOff + kSlab;              // b1 (4C floats), b2, gamma, beta (C floats each)
  static constexpr int kBarOff = kBiasOff + 7 * C * 4;
  // barriers: xn_full/empty[2], w1_full/empty[kS1], w2_full/empty[kS2], pre_full/empty[4], act_full/empty[2], y_full/empty[2]
  static constexpr int kNumBars = 4 + 2 * kS1 + 2 * kS2 + 2 * kPreBufs + 4 + 4;
  static constexpr int kSmemBytes = kBarOff + 8 * kNumBars + 16 + 1024;
  static_assert(kSmemBytes <= 232448, "shared-memory plan exceeds 227 KB");
  static_assert(kPreBufs * HC + kYBufs * C <= 512, "TMEM plan exceeds 512 columns");
};

// Debug timeline (CRF_MLP_PROF=1): clock64 stamps of CTA 0's pipeline events for the first kProfChunks chunks, read back
// with crf_debug_mlp_prof().  Events: 0/1 fc1 issue begin/end, 2 GELU sees pre_full, 3 GELU math done, 4 GELU passed the
// tile waits, 5 GELU arrived act_full, 6 fc2 sees act_full, 7 fc2 sees W2, 8 fc2 issued, 9 W1 load issued, 10 W2 load
// issued, 11/12 LayerNorm tile begin/end (index = tile), 13/14 final epilogue begin/end (index = tile).
constexpr int kProfEvents = 16, kProfChunks = 96;
__device__ long long g_mlp_prof[kProfEvents * kProfChunks];
#define MLP_PROF(ev, idx)                                                                          \
  do {                                                                                             \
    if (a.prof && blockIdx.x == 0 && (idx) < kProfChunks) g_mlp_prof[(ev) * kProfChunks + (idx)] = clock64(); \
  } while (0)

struct MlpArgs {
  const float* x1;     // (T, C) fp32 residual stream
  const float* gamma;  // LayerNorm-2 weight / bias
  const float* beta;
  const float* b1;     // (4C)
  const float* b2;     // (C)
  float* stats;        // (T, 2) (mean, rstd) or nullptr
  float eps;
  int T;
  int training;        // 1: xn2 / pre / act are stored for the backward pass
  int prof;            // debug timeline on
  int tm;              // token rows per tile actually loaded / stored (<= 128, multiple of 8): see launch_mlp_c
};

template <int C>
__global__ void __launch_bounds__(kThreads, 1)
mlp_fused_fwd_kernel(const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                     const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmXn,
                     const __grid_constant__ CUtensorMap tmPre, const __grid_constant__ CUtensorMap tmAct,
                     const MlpArgs a) {
  pdl_launch_dependents();
  using PL = MlpPlan<C>;
  constexpr int NCH = PL::NCH, NJ = PL::NJ, NSUB = PL::NSUB, kS1 = PL::kS1, kS2 = PL::kS2, kXnBufs = PL::kXnBufs,
                kYBufs = PL::kYBufs;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar0 = base + PL::kBarOff;
  int bi = 0;
  const uint32_t xn_full = bar0 + 8u * bi; bi += 2;
  const uint32_t xn_empty = bar0 + 8u * bi; bi += 2;
  const uint32_t w1_full = bar0 + 8u * bi; bi += kS1;
  const uint32_t w1_empty = bar0 + 8u * bi; bi += kS1;
  const uint32_t w2_full = bar0 + 8u * bi; bi += kS2;
  const uint32_t w2_empty = bar0 + 8u * bi; bi += kS2;
  const uint32_t pre_full = bar0 + 8u * bi; bi += kPreBufs;
  const uint32_t pre_empty = bar0 + 8u * bi; bi += kPreBufs;
  const uint32_t act_full = bar0 + 8u * bi; bi += 2;
  const uint32_t act_empty = bar0 + 8u * bi; bi += 2;
  const uint32_t y_full = bar0 + 8u * bi; bi += 2;
  const uint32_t y_empty = bar0 + 8u * bi; bi += 2;
  const uint32_t tmem_ptr_addr = bar0 + 8u * PL::kNumBars;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen + PL::kBarOff + 8 * PL::kNumBars);
  float* bias_s = reinterpret_cast<float*>(gen + PL::kBiasOff);  // b1[0 .. 4C), b2, gamma, beta [0 .. C) each

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tm = a.tm;
  const int total_tiles = (a.T + tm - 1) / tm;
  const int my_tiles =
      (total_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const uint32_t n_chunks = static_cast<uint32_t>(my_tiles) * NJ;  // global chunk index g = tile * NJ + j

  for (int c = threadIdx.x; c < 7 * C; c += kThreads)
    bias_s[c] = c < 4 * C ? a.b1[c] : c < 5 * C ? a.b2[c - 4 * C] : c < 6 * C ? a.gamma[c - 5 * C] : a.beta[c - 6 * C];
  if (warp == 20 && lane == 0) {
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
    tma_prefetch_desc(&tmY);
    for (int i = 0; i < 2; ++i) {
      mbar_init(xn_full + 8u * i, 1);
      mbar_init(xn_empty + 8u * i, 1);
      mbar_init(act_full + 8u * i, 1);
      mbar_init(act_empty + 8u * i, 1);
      mbar_init(y_full + 8u * i, 1);
      mbar_init(y_empty + 8u * i, 128);
    }
    for (int i = 0; i < kS1; ++i) {
      mbar_init(w1_full + 8u * i, 1);
      mbar_init(w1_empty + 8u * i, 1);
    }
    for (int i = 0; i < kS2; ++i) {
      mbar_init(w2_full + 8u * i, 1);
      mbar_init(w2_empty + 8u * i, 1);
    }
    for (int i = 0; i < kPreBufs; ++i) {
      mbar_init(pre_full + 8u * i, 1);
      mbar_init(pre_empty + 8u * i, 128);
    }
    fence_mbar_init();
  }
  if (warp == 22) {
    tmem_alloc(tmem_ptr_addr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_ptr_gen;
  const uint32_t tmem_pre = tmem_base, tmem_y = tmem_base + kPreBufs * HC;

  if (warp == 20) {
    // ===== W1 producer: chunk g needs W1[(g % NJ) * HC .. +HC, :] as NSUB stages of two 64-column atoms =====
    if (lane == 0) {
      uint32_t it = 0;
      for (uint32_t g = 0; g < n_chunks; ++g) {
        const int s = static_cast<int>(g % NJ);
        for (int h = 0; h < NSUB; ++h, ++it) {
          const uint32_t st = it % kS1;
          if (it >= static_cast<uint32_t>(kS1)) mbar_wait(w1_empty + 8u * st, ((it / kS1) - 1) & 1);
          const uint32_t dst = base + PL::kW1Off + st * PL::kStage;
          mbar_expect_tx(w1_full + 8u * st, PL::kStage);
          tma_load_2d(dst, &tmW1, w1_full + 8u * st, 128 * h, s * HC);
          tma_load_2d(dst + HC * 128, &tmW1, w1_full + 8u * st, 128 * h + 64, s * HC);
          MLP_PROF(9, g);
        }
      }
    }
  } else if (warp == 21) {
    // ===== W2 producer: chunk g needs W2[:, (g % NJ) * HC .. +HC) as NSUB stages of 128 output rows =====
    if (lane == 0) {
      uint32_t it = 0;
      for (uint32_t g = 0; g < n_chunks; ++g) {
        const int j = static_cast<int>(g % NJ);
        for (int h = 0; h < NSUB; ++h, ++it) {
          const uint32_t st = it % kS2;
          if (it >= static_cast<uint32_t>(kS2)) mbar_wait(w2_empty + 8u * st, ((it / kS2) - 1) & 1);
          const uint32_t dst = base + PL::kW2Off + st * PL::kStage;
          mbar_expect_tx(w2_full + 8u * st, PL::kStage);
          tma_load_2d(dst, &tmW2, w2_full + 8u * st, j * HC, 128 * h);
          MLP_PROF(10, g);
        }
      }
    }
  } else if (warp == 22) {
    // ===== fc1 issuer: pre[g % 4][128 x HC] = xn[128 x C] * W1 chunk^T; runs ahead of fc2 as far as the four TMEM
    //       chunk buffers allow (also across the tile boundary) =====
    if (lane == 0) {
      const uint32_t idesc1 = make_idesc(1u, 0u, 0u, TM, HC);
      uint32_t it = 0;
      for (uint32_t g = 0; g < n_chunks; ++g) {
        const int i = static_cast<int>(g / NJ), s = static_cast<int>(g % NJ);
        const int xb = i % kXnBufs;
        const uint32_t pb = g % kPreBufs;
        if (s == 0) {
          mbar_wait(xn_full + 8u * xb, (i / kXnBufs) & 1);
          tc_fence_after();
        }
        if (g >= static_cast<uint32_t>(kPreBufs)) {
          mbar_wait(pre_empty + 8u * pb, ((g / kPreBufs) - 1) & 1);
          tc_fence_after();
        }
        const SmemDescBase ad = make_smem_desc_base(base + PL::kXnOff + xb * PL::kXnTile, 16, 1024, kSwizzle128);
        for (int h = 0; h < NSUB; ++h, ++it) {
          const uint32_t st = it % kS1;
          mbar_wait(w1_full + 8u * st, (it / kS1) & 1);
          tc_fence_after();
          MLP_PROF(0, g);
          const SmemDescBase bd = make_smem_desc_base(base + PL::kW1Off + st * PL::kStage, 16, 1024, kSwizzle128);
#pragma unroll
          for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_bf16(tmem_pre + pb * HC, smem_desc_at(ad, (2 * h + k) * kSlab + ks * 32),
                        smem_desc_at(bd, k * (HC * 128) + ks * 32), idesc1, (h > 0 || k > 0 || ks > 0) ? 1u : 0u);
          umma_commit(w1_empty + 8u * st);
        }
        umma_commit(pre_full + 8u * pb);
        MLP_PROF(1, g);
        if (s == NJ - 1) umma_commit(xn_empty + 8u * xb);
      }
    }
  } else if (warp == 23) {
    // ===== fc2 issuer: y[128 x C] += act chunk[128 x HC] * W2[:, chunk]^T =====
    if (lane == 0) {
      const uint32_t idesc2 = make_idesc(1u, 0u, 0u, TM, 128);
      uint32_t it = 0;
      for (uint32_t g = 0; g < n_chunks; ++g) {
        const int i = static_cast<int>(g / NJ), j = static_cast<int>(g % NJ);
        const int yb = i % kYBufs;
        const uint32_t ab = g & 1u;
        if (j == 0 && i >= kYBufs) {
          mbar_wait(y_empty + 8u * yb, ((i / kYBufs) - 1) & 1);
          tc_fence_after();
        }
        mbar_wait(act_full + 8u * ab, (g >> 1) & 1);
        tc_fence_after();
        MLP_PROF(6, g);
        const SmemDescBase ad = make_smem_desc_base(base + PL::kActOff + ab * kSlab, 16, 1024, kSwizzle128);
        for (int h = 0; h < NSUB; ++h, ++it) {  // output columns [128h, 128h + 128)
          const uint32_t st = it % kS2;
          mbar_wait(w2_full + 8u * st, (it / kS2) & 1);
          tc_fence_after();
          MLP_PROF(7, g);
          const SmemDescBase bd = make_smem_desc_base(base + PL::kW2Off + st * PL::kStage, 16, 1024, kSwizzle128);
#pragma unroll
          for (int ks = 0; ks < HC / 16; ++ks)
            umma_bf16(tmem_y + yb * C + h * 128, smem_desc_at(ad, ks * 32), smem_desc_at(bd, ks * 32), idesc2,
                      (j > 0 || ks > 0) ? 1u : 0u);
          umma_commit(w2_empty + 8u * st);
        }
        umma_commit(act_empty + 8u * ab);
        MLP_PROF(8, g);
        if (j == NJ - 1) umma_commit(y_full + 8u * yb);
      }
    }
  } else if (warp < 8) {
    // ===== LayerNorm-2 prologue, eight warps: warp w normalises rows 16w .. 16w+15 of every tile.  Eight lanes share a
    //       row (lane = 8 * row-in-step + sub; sub owns columns 32k + 4 sub .. +3), so one warp-wide 16-byte load
    //       covers 128 contiguous bytes of four rows and the row statistics cost three shuffles each; 8 (C = 128) or
    //       4 (C = 256) rows are in flight per warp, 32 KB per SM =====
    constexpr int NV = C / 32;              // float4 per lane and row
    constexpr int SB = C <= 128 ? 2 : 1;    // 4-row steps in flight
    const int tid = threadIdx.x;            // 0..255
    const int sub = lane & 7, rq = lane >> 3;
    const float* gamma_s = bias_s + 5 * C;
    const float* beta_s = bias_s + 6 * C;
    for (int i = 0; i < my_tiles; ++i) {
      const int t0 = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) * tm;
      const int xb = i % kXnBufs;
      if (tid == 0) {
        if (i >= kXnBufs) mbar_wait_sleep(xn_empty + 8u * xb, ((i / kXnBufs) - 1) & 1);  // fc1 of tile i-kXnBufs has read it
        if (a.training) bulk_wait_read<0>();                                              // and so has its xn2 store
      }
      named_bar_sync(1, 256);
      if (tid == 0) MLP_PROF(11, i);
      uint8_t* xn_g = gen + PL::kXnOff + xb * PL::kXnTile;
#pragma unroll 1
      for (int st0 = 0; st0 < 4; st0 += SB) {
        float4 v[SB][NV];
#pragma unroll
        for (int q = 0; q < SB; ++q) {
          const int rr = 16 * warp + 4 * (st0 + q) + rq, t = t0 + rr;
          const int tc = (rr < tm && t < a.T) ? t : t0;  // rows past the tile / the input re-read row t0 (zeroed below, never stored)
          const float4* row = reinterpret_cast<const float4*>(a.x1 + static_cast<size_t>(tc) * C) + sub;
#pragma unroll
          for (int k = 0; k < NV; ++k) v[q][k] = __ldg(row + 8 * k);
        }
#pragma unroll
        for (int q = 0; q < SB; ++q) {
          const int r = 16 * warp + 4 * (st0 + q) + rq, t = t0 + r;
          float sum = 0.f;
#pragma unroll
          for (int k = 0; k < NV; ++k) sum += (v[q][k].x + v[q][k].y) + (v[q][k].z + v[q][k].w);
          sum += __shfl_xor_sync(0xffffffffu, sum, 1);
          sum += __shfl_xor_sync(0xffffffffu, sum, 2);
          sum += __shfl_xor_sync(0xffffffffu, sum, 4);
          const float mean = sum * (1.0f / C);
          float d2 = 0.f;
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const float d0 = v[q][k].x - mean, d1 = v[q][k].y - mean, e0 = v[q][k].z - mean, e1 = v[q][k].w - mean;
            d2 += (d0 * d0 + d1 * d1) + (e0 * e0 + e1 * e1);
          }
          d2 += __shfl_xor_sync(0xffffffffu, d2, 1);
          d2 += __shfl_xor_sync(0xffffffffu, d2, 2);
          d2 += __shfl_xor_sync(0xffffffffu, d2, 4);
          const float rstd = rsqrtf(d2 * (1.0f / C) + a.eps);
          const bool live = r < tm && t < a.T;   // rows >= tm of the 128-row MMA tile belong to the next tile: zero, never stored
          if (live && sub == 0 && a.stats != nullptr)
            *reinterpret_cast<float2*>(a.stats + 2 * static_cast<size_t>(t)) = make_float2(mean, rstd);
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const int c = 32 * k + 4 * sub;  // first of this lane's four columns
            const float4 gm = *reinterpret_cast<const float4*>(gamma_s + c);
            const float4 bt = *reinterpret_cast<const float4*>(beta_s + c);
            const float o0 = (v[q][k].x - mean) * rstd * gm.x + bt.x, o1 = (v[q][k].y - mean) * rstd * gm.y + bt.y;
            const float o2 = (v[q][k].z - mean) * rstd * gm.z + bt.z, o3 = (v[q][k].w - mean) * rstd * gm.w + bt.w;
            // atom c / 64, row r, 16-byte chunk (c % 64) / 8, 8-byte half (c % 8) / 4
            *reinterpret_cast<uint2*>(xn_g + (c >> 6) * kSlab + sw128_offset(r, (c & 63) >> 3) + ((c & 4) << 1)) =
                live ? make_uint2(pack_bf16(o0, o1), pack_bf16(o2, o3)) : make_uint2(0u, 0u);
          }
        }
      }
      fence_proxy_async_smem();
      named_bar_sync(1, 256);
      if (tid == 0) {
        MLP_PROF(12, i);
        mbar_arrive(xn_full + 8u * xb);
        if (a.training) {
#pragma unroll
          for (int k = 0; k < NCH; ++k) tma_store_2d(&tmXn, base + PL::kXnOff + xb * PL::kXnTile + k * kSlab, 64 * k, t0);
          bulk_commit();
        }
      }
    }
    if (tid == 0) bulk_wait_read<0>();
  } else if (warp < 16) {
    // ===== GELU groups: two groups of four warps (thread = accumulator row); group gi takes the chunks with (global)
    //       parity gi.  The first 32 columns are computed BEFORE the waits for the shared-memory tiles (fc2 of chunk g-2
    //       has read the act tile; the TMA stores of chunk g-2 have read both tiles), so those latencies hide behind it =====
    const int gi = (warp - 8) >> 2;
    const int r = threadIdx.x & 127;
    const bool leader = r == 0;
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    uint8_t* act_g = gen + PL::kActOff + gi * kSlab;
    uint8_t* pre_g = gen + PL::kPreOff + gi * kSlab;
    const uint32_t act_s = base + PL::kActOff + gi * kSlab, pre_s = base + PL::kPreOff + gi * kSlab;
#pragma unroll 1
    for (uint32_t g = gi; g < n_chunks; g += 2) {
      const int i = static_cast<int>(g / NJ), j = static_cast<int>(g % NJ);
      const int t0 = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) * tm;
      const uint32_t pb = g % kPreBufs;
      mbar_wait(pre_full + 8u * pb, (g / kPreBufs) & 1);
      tc_fence_after();
      if (leader) MLP_PROF(2, g);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t acc[32];
        tmem_ld32(tmem_pre + pb * HC + half * 32 + lane_base, acc);
        tmem_ld_wait();
        if (half == 1) {  // accumulator chunk fully read: hand the TMEM buffer back to the fc1 issuer
          tc_fence_before();
          mbar_arrive(pre_empty + 8u * pb);
        }
        uint32_t pp[16], pa[16];  // bf16 pairs of the pre-activation and the activation
        const float4* b4 = reinterpret_cast<const float4*>(bias_s + j * HC + half * 32);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 b = b4[q];
          float v0 = __uint_as_float(acc[4 * q + 0]) + b.x, v1 = __uint_as_float(acc[4 * q + 1]) + b.y;
          float v2 = __uint_as_float(acc[4 * q + 2]) + b.z, v3 = __uint_as_float(acc[4 * q + 3]) + b.w;
          pp[2 * q] = pack_bf16(v0, v1);
          pp[2 * q + 1] = pack_bf16(v2, v3);
          gelu_erf2(v0, v1);
          gelu_erf2(v2, v3);
          pa[2 * q] = pack_bf16(v0, v1);
          pa[2 * q + 1] = pack_bf16(v2, v3);
        }
        if (half == 0) {
          if (leader) MLP_PROF(3, g);
          if (leader && a.training) bulk_wait_read<0>();  // this group's previous pre / act stores have read their tiles
          if (g >= 2) mbar_wait(act_empty + 8u * gi, ((g >> 1) - 1) & 1);  // fc2 of chunk g-2 has read the act tile
          named_bar_sync(2 + gi, 128);
          if (leader) MLP_PROF(4, g);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (a.training)
            *reinterpret_cast<uint4*>(pre_g + sw128_offset(r, half * 4 + q)) =
                make_uint4(pp[4 * q], pp[4 * q + 1], pp[4 * q + 2], pp[4 * q + 3]);
          *reinterpret_cast<uint4*>(act_g + sw128_offset(r, half * 4 + q)) =
              make_uint4(pa[4 * q], pa[4 * q + 1], pa[4 * q + 2], pa[4 * q + 3]);
        }
      }
      fence_proxy_async_smem();
      named_bar_sync(2 + gi, 128);
      if (leader) {
        MLP_PROF(5, g);
        mbar_arrive(act_full + 8u * gi);
        if (a.training) {
          tma_store_2d(&tmPre, pre_s, j * HC, t0);
          tma_store_2d(&tmAct, act_s, j * HC, t0);
          bulk_commit();
        }
      }
    }
    if (leader) bulk_wait_read<0>();
  } else {
    // ===== final epilogue: y = fc2 accumulator + b2 + x1, 32-column fp32 slabs.  Thread = accumulator row; the
    //       residual row segment (128 contiguous bytes) is fetched straight into registers before the accumulator is
    //       awaited, so its latency hides behind the wait =====
    const int r = threadIdx.x & 127;
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t out_s = base + PL::kOutOff;
    uint8_t* outb = gen + PL::kOutOff;
    const float* b2_s = bias_s + 4 * C;
    for (int i = 0; i < my_tiles; ++i) {
      const int t0 = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) * tm;
      const int yb = i % kYBufs;
      const int t = (r < tm && t0 + r < a.T) ? t0 + r : t0;  // rows past the tile / the input: not stored (TMA box = tm rows)
      const float4* xrow = reinterpret_cast<const float4*>(a.x1 + static_cast<size_t>(t) * C);
      float4 xr[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) xr[q] = __ldg(xrow + q);
      mbar_wait_sleep(y_full + 8u * yb, (i / kYBufs) & 1);
      tc_fence_after();
      if (r == 0) MLP_PROF(13, i);
#pragma unroll 1
      for (int s = 0; s < C / 32; ++s) {
        if (r == 0) bulk_wait_read<0>();  // the previous store has read the out slab
        named_bar_sync(4, 128);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t acc[16];
          tmem_ld16(tmem_y + yb * C + s * 32 + hh * 16 + lane_base, acc);
          tmem_ld_wait();
          if (s == C / 32 - 1 && hh == 1) {
            tc_fence_before();
            mbar_arrive(y_empty + 8u * yb);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 b = *reinterpret_cast<const float4*>(b2_s + s * 32 + hh * 16 + 4 * q);
            const float4 x = xr[hh * 4 + q];
            *reinterpret_cast<float4*>(outb + sw128_offset(r, hh * 4 + q)) =
                make_float4(__uint_as_float(acc[4 * q + 0]) + b.x + x.x, __uint_as_float(acc[4 * q + 1]) + b.y + x.y,
                            __uint_as_float(acc[4 * q + 2]) + b.z + x.z, __uint_as_float(acc[4 * q + 3]) + b.w + x.w);
          }
        }
        if (s + 1 < C / 32) {
#pragma unroll
          for (int q = 0; q < 8; ++q) xr[q] = __ldg(xrow + (s + 1) * 8 + q);  // next slab of the residual, in flight below
        }
        fence_proxy_async_smem();
        named_bar_sync(4, 128);
        if (r == 0) {
          tma_store_2d(&tmY, out_s, s * 32, t0);
          bulk_commit();
        }
      }
      if (r == 0) MLP_PROF(14, i);
    }
    if (r == 0) bulk_wait_read<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 22) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int C>
int launch_mlp_c(const crf_mlp_args& m, cudaStream_t st) {
  using PL = MlpPlan<C>;
  CUtensorMap tmW1, tmW2, tmY, tmXn, tmPre, tmAct;
  if (make_tmap_bf16(&tmW1, m.w1_bf16, 4 * C, C, HC)) return 1;
  if (make_tmap_bf16(&tmW2, m.w2_bf16, C, 4 * C, 128)) return 1;
  // Rows per tile: the MMA tile is always 128 rows; only `tm` of them are normalised, multiplied for real and stored, with
  // tm chosen so that the tiles fill whole rounds of the persistent grid (T = 38400: 300 tiles of 128 rows = 2.03 rounds
  // on 148 SMs, i.e. 3 rounds; 437 tiles of 88 rows = 2.95 rounds of a shorter tile).
  const int sms = num_sms(m.device);
  const int tm = balanced_tile_rows(m.T, sms);
  if (make_tmap_f32(&tmY, m.y, m.T, C, tm)) return 1;
  if (m.training) {
    if (make_tmap_bf16(&tmXn, m.xn2, m.T, C, tm)) return 1;
    if (make_tmap_bf16(&tmPre, m.pre, m.T, 4 * C, tm)) return 1;
    if (make_tmap_bf16(&tmAct, m.act, m.T, 4 * C, tm)) return 1;
  } else {
    tmXn = tmW1; tmPre = tmW1; tmAct = tmW1;
  }
  auto kern = mlp_fused_fwd_kernel<C>;
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, PL::kSmemBytes));
  const int tiles = (m.T + tm - 1) / tm;
  int grid = sms;
  if (grid > tiles) grid = tiles;
  static const int prof = [] { const char* e = getenv("CRF_MLP_PROF"); return e != nullptr && e[0] == '1' ? 1 : 0; }();
  MlpArgs a{m.x1, m.norm_w, m.norm_b, m.b1, m.b2, m.training ? m.stats : nullptr, m.eps, m.T, m.training ? 1 : 0, prof, tm};
  const double tc = static_cast<double>(m.T) * C;
  KernelTimer timer(st, 16.0 * tc * C, tc * (8.0 + (m.training ? 18.0 : 0.0)) + 16.0 * C * C, "mlp_fused_fwd_T%d_C%d%s",
                 m.T, C, m.training ? "" : "_infer");
  launch_pdl(kern, grid, kThreads, PL::kSmemBytes, st, tmW1, tmW2, tmY, tmXn, tmPre, tmAct, a);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace

bool mlp_fused_supported(int C) { return C == 128 || C == 256; }

// debug: copy the timeline of the last profiled launch (kProfEvents x kProfChunks clock64 stamps) to the host
int mlp_debug_prof(long long* out, int n) {
  if (n > kProfEvents * kProfChunks) n = kProfEvents * kProfChunks;
  CRF_CUDA(cudaDeviceSynchronize());
  CRF_CUDA(cudaMemcpyFromSymbol(out, g_mlp_prof, sizeof(long long) * n));
  return 0;
}

int launch_mlp_fused_fwd(const crf_mlp_args& m, cudaStream_t st) {
  CRF_CHECK(m.x1 && m.y && m.w1_bf16 && m.w2_bf16 && m.b1 && m.b2 && m.norm_w && m.norm_b, "crf_mlp_fwd: null pointer");
  CRF_CHECK(m.T > 0, "crf_mlp_fwd: empty input");
  CRF_CHECK(!m.training || (m.xn2 && m.stats && m.pre && m.act), "crf_mlp_fwd: training needs xn2, stats, pre, act");
  switch (m.C) {
    case 128: return launch_mlp_c<128>(m, st);
    case 256: return launch_mlp_c<256>(m, st);
    default: return set_error("crf_mlp_fwd: C=%d is not supported by the fused kernel (128, 256)", m.C);
  }
}

}  // namespace crf
