// Input-gradient GEMM of a projection with the LayerNorm backward of its input fused into the epilogue (C = 128 / 256):
//
//   g  = dY (T, K) * W (K, C)                                  -- d fc1 (K = 4C) or d qk (K = 2C): gradient w.r.t. xn = LN(x)
//   dx = rstd * (g*gamma - mean_c(g*gamma) - xhat * mean_c(g*gamma*xhat)) + dres,   dgamma += sum_t g*xhat,  dbeta += sum_t g
//
// i.e. the backward of `self.norm2(x)` / `self.norm1(x)` in CRFBlock.forward (/root/reference/src/newcrf_layers.py:208,255)
// applied to the gradient coming out of fc1 / qk, plus the residual branch (`dres`).  Unfused, g is an fp32 (T, C)
// tensor that one kernel writes and the next reads (158 MB per LayerNorm at the 1/4 scale); here a persistent CTA's output
// tile spans whole rows (tm <= 128 tokens x C columns; tm balanced against the grid, crf_sched.h), so the row reductions
// happen on the accumulator in TMEM:
//
//   warp 8        TMA producer of the A / B ring (A: 128 x 64 K-major tile of dY; B: 64 x C MN-major tile of W, from L2)
//   warp 9        MMA issuer: tile i accumulates into TMEM buffer i % (512 / C)
//   warp 10       slab producer: streams 128 x 32 fp32 slabs of x (pass 1) and of x, dres (pass 2) through a 4-stage ring
//   warps 0-7     epilogue, thread = token row = TMEM lane, two halves of four warps that split the 32-column slabs.
//                 Pass 1: s1 = sum g*gamma, s2 = sum g*gamma*xhat and the column partial sums of g*xhat, g (warp
//                 transpose-reduce: 31 shuffles per 32 columns, kept in registers across all tiles of the CTA).
//                 Pass 2: dx, written as fp32 slabs and as a bf16 twin by TMA stores.
//
// Slab release (found the hard way, profiles/r02_dgrad_lnbwd.md): an mbarrier.arrive issued right after the LDS of a
// TMA-written slab can overtake those loads -- the producer's next TMA load then lands in the slab while a few lanes are
// still reading it (4-column glitches in ~1 of 3 launches).  A slab is therefore released only after an instruction that
// consumed every value loaded from it in every lane (the transpose-reduce shuffles in pass 1, the named barrier that
// follows the output stores in pass 2).
//
// Algorithmic bytes per token: 2K (dY) + 4C (x) + 4C (dres) + 4C (dx) + 2C (bf16 twin); flops 2 K C.
#include "crf_host.h"
#include "crf_ptx.cuh"
#include "crf_sched.h"

namespace crf {

namespace {

constexpr int TM = 128, BK = 64;
constexpr int kThreads = 352;   // 8 epilogue warps, A/B producer, MMA issuer, slab producer
constexpr int kSlab = TM * 128;     // 16 KB: 128 rows x 32 fp32 (or x 64 bf16)

// Shared-memory plan (runtime stage counts: n_ring A/B stages, n_slab slab stages)
constexpr int kMaxStages = 6;
template <int C>
struct LnPlan {
  static constexpr int kAcc = 512 / C;
  static constexpr int kATile = TM * 128, kBTile = C * 128, kStage = kATile + kBTile;
  static constexpr int kNumBars = 2 * kMaxStages + 2 * kAcc + 2 * kMaxStages;
  // ring | slabs | out32 x 2 | out16 | gamma | row-sum exchange | barriers
  static constexpr int bytes(int n_ring, int n_slab) {
    return n_ring * kStage + n_slab * kSlab + 3 * kSlab + C * 4 + 2 * 128 * 8 + 8 * kNumBars + 16 + 1024;
  }
};

struct LnArgs {
  const float* stats;   // (T, 2) = (mean, rstd)
  const float* gamma;
  float* dgamma;
  float* dbeta;
  int T, K;
  int has_dres, has_dx, has_dxb;
  int n_ring, n_slab;   // stages of the A/B ring and of the slab ring
  int tm;               // token rows per tile (<= 128, multiple of 8): see launch_c
};

// v[0] of lane L <- sum over the warp's 32 lanes of v[L]  (transpose-reduce, 31 shuffles)
__device__ __forceinline__ float warp_transpose_sum(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = up ? v[i] : v[i + off];
      const float keep = up ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

template <int C>
__global__ void __launch_bounds__(kThreads, 1)
dgrad_lnbwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmRes,
                   const __grid_constant__ CUtensorMap tmDx, const __grid_constant__ CUtensorMap tmDxb, const LnArgs a) {
  pdl_launch_dependents();
  using PL = LnPlan<C>;
  constexpr int kAcc = PL::kAcc, NS = C / 32;
  const int kStages = a.n_ring, kSlabStages = a.n_slab;
  const int kSlabOff = kStages * PL::kStage, kOut32Off = kSlabOff + kSlabStages * kSlab, kOut16Off = kOut32Off + 2 * kSlab,
            kGammaOff = kOut16Off + kSlab, kExchOff = kGammaOff + C * 4, kBarOff = kExchOff + 2 * 128 * 8;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar0 = base + kBarOff;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kMaxStages + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * kMaxStages + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * kMaxStages + kAcc + b); };
  auto sfull_bar = [&](int s) { return bar0 + 8u * (2 * kMaxStages + 2 * kAcc + s); };
  auto sempty_bar = [&](int s) { return bar0 + 8u * (2 * kMaxStages + 2 * kAcc + kMaxStages + s); };
  const uint32_t tmem_ptr_addr = bar0 + 8u * PL::kNumBars;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen + kBarOff + 8 * PL::kNumBars);
  float* gam_s = reinterpret_cast<float*>(gen + kGammaOff);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tm = a.tm;
  const int total_tiles = (a.T + tm - 1) / tm;
  const int my_tiles =
      (total_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int nk = a.K / BK;

  for (int c = threadIdx.x; c < C; c += kThreads) gam_s[c] = a.gamma[c];
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmX);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < kAcc; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), 256);
    }
    for (int s = 0; s < kSlabStages; ++s) {
      mbar_init(sfull_bar(s), 1);
      mbar_init(sempty_bar(s), 4);
    }
    fence_mbar_init();
  }
  if (warp == 9) {
    tmem_alloc(tmem_ptr_addr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 8) {
    // ===== A / B ring =====
    if (lane == 0) {
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int m0 = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) * tm;
        for (int kc = 0; kc < nk; ++kc, ++it) {
          const int s = it % kStages;
          if (it >= kStages) mbar_wait(empty_bar(s), ((it / kStages) - 1) & 1);
          const uint32_t a_dst = base + s * PL::kStage, b_dst = a_dst + PL::kATile;
          mbar_expect_tx(full_bar(s), tm * 128 + PL::kBTile);
          tma_load_2d(a_dst, &tmA, full_bar(s), kc * BK, m0);
#pragma unroll
          for (int j = 0; j < C / 64; ++j) tma_load_2d(b_dst + 8192 * j, &tmB, full_bar(s), 64 * j, kc * BK);
        }
      }
    }
  } else if (warp == 9) {
    // ===== MMA issuer =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc(1u, 0u, 1u, TM, C);
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int b = i % kAcc;
        if (i >= kAcc) {
          mbar_wait(tempty_bar(b), ((i / kAcc) - 1) & 1);
          tc_fence_after();
        }
        const uint32_t d_tmem = tmem_base + b * C;
        for (int kc = 0; kc < nk; ++kc, ++it) {
          const int s = it % kStages;
          mbar_wait(full_bar(s), (it / kStages) & 1);
          tc_fence_after();
          const uint32_t a_src = base + s * PL::kStage, b_src = a_src + PL::kATile;
#pragma unroll
          for (int ks = 0; ks < BK / 16; ++ks)
            umma_bf16(d_tmem, make_smem_desc(a_src + ks * 32, 16, 1024, kSwizzle128),
                      make_smem_desc(b_src + ks * 2048, 8192, 1024, kSwizzle128), idesc, (kc > 0 || ks > 0) ? 1u : 0u);
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(b));
      }
    }
  } else if (warp == 10) {
    // ===== slab producer: per tile x[0..NS) (pass 1), then (x[s], dres[s]) for s in [0, NS) (pass 2) =====
    if (lane == 0) {
      int it = 0;
      auto push = [&](const CUtensorMap* map, int col, int m0) {
        const int s = it % kSlabStages;
        if (it >= kSlabStages) mbar_wait(sempty_bar(s), ((it / kSlabStages) - 1) & 1);
        mbar_expect_tx(sfull_bar(s), tm * 128);
        tma_load_2d(base + kSlabOff + s * kSlab, map, sfull_bar(s), col, m0);
        ++it;
      };
      for (int i = 0; i < my_tiles; ++i) {
        const int m0 = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) * tm;
        for (int s = 0; s < NS; ++s) push(&tmX, 32 * s, m0);
        for (int s = 0; s < NS; ++s) {
          push(&tmX, 32 * s, m0);
          if (a.has_dres) push(&tmRes, 32 * s, m0);
        }
      }
    }
  } else {
    // ===== epilogue, warps 0-7: two halves of four warps.  Thread = token row = TMEM lane; half h takes the 32-column
    //       slabs s with s % 2 == h (two warps per scheduler hide each other's TMEM / shared-memory / barrier latencies).
    //       The halves exchange their partial row sums between the passes and share the bf16 output slab (64 columns). =====
    const int half = warp >> 2;
    const int r = threadIdx.x & 127;
    const bool leader = r == 0;
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    uint8_t* out32 = gen + kOut32Off + half * kSlab;
    uint8_t* out16 = gen + kOut16Off;
    float2* exch = reinterpret_cast<float2*>(gen + kExchOff);   // [2 halves][128 rows] (s1, s2)
    const uint32_t out32_s = base + kOut32Off + half * kSlab, out16_s = base + kOut16Off;
    constexpr int NH = NS / 2;
    const int per_tile = NS + NS * (1 + a.has_dres);   // slabs the producer pushes per tile
    float dga[NH], dbe[NH];
#pragma unroll
    for (int k = 0; k < NH; ++k) dga[k] = dbe[k] = 0.f;
    for (int i = 0; i < my_tiles; ++i) {
      const int m0 = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) * tm;
      const int b = i % kAcc;
      const int t = m0 + r;
      const int ring0 = i * per_tile;
      const bool live = r < tm && t < a.T;   // rows >= tm of the 128-row MMA tile hold stale data: computed, never used
      float mean = 0.f, rstd = 0.f;
      if (live) {
        const float2 st = __ldg(reinterpret_cast<const float2*>(a.stats) + t);
        mean = st.x;
        rstd = st.y;
      }
      const uint32_t taddr = tmem_base + b * C + lane_base;
      mbar_wait(tfull_bar(b), (i / kAcc) & 1);
      tc_fence_after();
      // ---- pass 1: row sums and column partial sums over this half's slabs ----
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int k = 0; k < NH; ++k) {
        const int s = 2 * k + half;
        const int idx = ring0 + s, st = idx % kSlabStages;
        mbar_wait(sfull_bar(st), (idx / kSlabStages) & 1);
        const uint8_t* xs = gen + kSlabOff + st * kSlab;
        // (tcgen05.ld and its wait stay adjacent, with the warp converged: they are warp-collective)
        __syncwarp();
        uint32_t acc[32];
        tmem_ld32(taddr + s * 32, acc);
        tmem_ld_wait();
        float pa[32], pb[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 xv = *reinterpret_cast<const float4*>(xs + sw128_offset(r, q));
          const float4 gm = *reinterpret_cast<const float4*>(gam_s + 32 * s + 4 * q);
          const float xe[4] = {xv.x, xv.y, xv.z, xv.w};
          const float ge[4] = {gm.x, gm.y, gm.z, gm.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float g = __uint_as_float(acc[4 * q + e]);
            const float xh = (xe[e] - mean) * rstd;
            const float gg = g * ge[e];
            s1 += gg;
            s2 += gg * xh;
            pa[4 * q + e] = live ? g * xh : 0.f;
            pb[4 * q + e] = live ? g : 0.f;
          }
        }
        dga[k] += warp_transpose_sum(pa, lane);
        dbe[k] += warp_transpose_sum(pb, lane);
        // release the slab only now: the shuffles above consumed every value loaded from it, in every lane
        __syncwarp();
        if (lane == 0) mbar_arrive(sempty_bar(st));
      }
      exch[half * 128 + r] = make_float2(s1, s2);
      named_bar_sync(1, 256);
      {
        const float2 o = exch[(half ^ 1) * 128 + r];
        s1 = (s1 + o.x) * (1.0f / C);
        s2 = (s2 + o.y) * (1.0f / C);
      }
      // ---- pass 2: dx, one pair of slabs (2k, 2k + 1) at a time, the halves in step ----
#pragma unroll 1
      for (int k = 0; k < NH; ++k) {
        const int s = 2 * k + half;
        const int idx_x = ring0 + NS + s * (1 + a.has_dres), stx = idx_x % kSlabStages;
        mbar_wait(sfull_bar(stx), (idx_x / kSlabStages) & 1);
        int std_ = stx;
        if (a.has_dres) {
          const int idx_d = idx_x + 1;
          std_ = idx_d % kSlabStages;
          mbar_wait(sfull_bar(std_), (idx_d / kSlabStages) & 1);
        }
        const uint8_t* xs = gen + kSlabOff + stx * kSlab;
        const uint8_t* ds = gen + kSlabOff + std_ * kSlab;
        __syncwarp();
        uint32_t acc[32];
        tmem_ld32(taddr + s * 32, acc);
        tmem_ld_wait();
        if (k == NH - 1) {  // accumulator fully read by this thread: hand the TMEM buffer back to the MMA warp
          tc_fence_before();
          mbar_arrive(tempty_bar(b));
        }
        float o[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 xv = *reinterpret_cast<const float4*>(xs + sw128_offset(r, q));
          const float4 gm = *reinterpret_cast<const float4*>(gam_s + 32 * s + 4 * q);
          float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (a.has_dres) dv = *reinterpret_cast<const float4*>(ds + sw128_offset(r, q));
          float xe[4] = {xv.x, xv.y, xv.z, xv.w};
          const float ge[4] = {gm.x, gm.y, gm.z, gm.w};
          float de[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float g = __uint_as_float(acc[4 * q + e]);
            const float xh = (xe[e] - mean) * rstd;
            o[4 * q + e] = rstd * (g * ge[e] - s1 - xh * s2) + de[e];
          }
        }
        // the leaders' previous TMA stores have read the out slabs (half 1's leader also stores the shared bf16 slab)
        if (leader) bulk_wait_read<0>();
        named_bar_sync(1, 256);
        if (a.has_dx) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(out32 + sw128_offset(r, q)) = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
        }
        if (a.has_dxb) {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(out16 + sw128_offset(r, half * 4 + q)) =
                make_uint4(pack_bf16(o[8 * q], o[8 * q + 1]), pack_bf16(o[8 * q + 2], o[8 * q + 3]),
                           pack_bf16(o[8 * q + 4], o[8 * q + 5]), pack_bf16(o[8 * q + 6], o[8 * q + 7]));
        }
        fence_proxy_async_smem();
        named_bar_sync(1, 256);
        // every thread has stored values that depend on everything it read from the x / dres slabs: release them
        if (lane == 0) {
          mbar_arrive(sempty_bar(stx));
          if (a.has_dres) mbar_arrive(sempty_bar(std_));
        }
        if (leader) {
          if (a.has_dx) tma_store_2d(&tmDx, out32_s, 32 * s, m0);
          if (a.has_dxb && half == 1) tma_store_2d(&tmDxb, out16_s, 64 * k, m0);
          bulk_commit();
        }
      }
    }
    if (leader) bulk_wait_read<0>();
    // ---- column sums: 4 warps per column -> shared memory -> one atomic per column and CTA ----
    named_bar_sync(1, 256);
    float* red = reinterpret_cast<float*>(gen + kOut32Off);   // [4 sub-partitions][2][C] floats (<= 8 KB)
#pragma unroll
    for (int k = 0; k < NH; ++k) {
      const int s = 2 * k + half;
      red[((warp & 3) * 2 + 0) * C + 32 * s + lane] = dga[k];
      red[((warp & 3) * 2 + 1) * C + 32 * s + lane] = dbe[k];
    }
    named_bar_sync(1, 256);
    for (int c = threadIdx.x; c < 2 * C; c += 256) {
      const float v = red[c] + red[2 * C + c] + red[4 * C + c] + red[6 * C + c];
      atomicAdd((c < C ? a.dgamma : a.dbeta) + (c < C ? c : c - C), v);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int C>
int launch_c(const void* dY, const void* W, int K, const float* x, const float* stats, const float* gamma,
             const float* dres, float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T, int device, cudaStream_t st) {
  using PL = LnPlan<C>;
  CUtensorMap tmA, tmB, tmX, tmRes, tmDx, tmDxb;
  // Rows per tile: the MMA tile is always 128 rows, but only `tm` of them are loaded, reduced and stored, with tm chosen
  // so that the tiles fill whole rounds of the persistent grid (T = 38400: 300 tiles of 128 rows are 2.03 rounds on 148
  // SMs, i.e. 3; 437 tiles of 88 rows are 2.95 rounds of a shorter tile: -31 % row-time).
  const int sms = num_sms(device);
  const int tm = balanced_tile_rows(T, sms);
  if (make_tmap_bf16(&tmA, dY, T, K, tm)) return 1;
  if (make_tmap_bf16(&tmB, W, K, C, 64)) return 1;
  if (make_tmap_f32(&tmX, x, T, C, tm)) return 1;
  tmRes = tmX; tmDx = tmX; tmDxb = tmA;
  if (dres != nullptr && make_tmap_f32(&tmRes, dres, T, C, tm)) return 1;
  if (dx != nullptr && make_tmap_f32(&tmDx, dx, T, C, tm)) return 1;
  if (dx_bf16 != nullptr && make_tmap_bf16(&tmDxb, dx_bf16, T, C, tm)) return 1;
  auto kern = dgrad_lnbwd_kernel<C>;
  // stages (measured: the counts hardly matter once >= 2): 96 KB of A/B ring + 4 slab stages
  const int n_ring = C <= 128 ? 3 : 2, n_slab = 4;
  const int smem_bytes = PL::bytes(n_ring, n_slab);
  CRF_CHECK(smem_bytes <= 232448, "dgrad_lnbwd: shared-memory plan exceeds 227 KB");
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  const int tiles = (T + tm - 1) / tm;
  int grid = sms;
  if (grid > tiles) grid = tiles;
  LnArgs a{stats, gamma, dgamma, dbeta, T, K, dres != nullptr ? 1 : 0, dx != nullptr ? 1 : 0, dx_bf16 != nullptr ? 1 : 0,
           n_ring, n_slab, tm};
  const double tc = static_cast<double>(T) * C;
  KernelTimer timer(st, 2.0 * tc * K,
                 2.0 * T * K + 2.0 * K * C + tc * (4.0 + (dres ? 4.0 : 0.0) + (dx ? 4.0 : 0.0) + (dx_bf16 ? 2.0 : 0.0)),
                 "dgrad_lnbwd_T%d_C%d_K%d", T, C, K);
  launch_pdl(kern, grid, kThreads, smem_bytes, st, tmA, tmB, tmX, tmRes, tmDx, tmDxb, a);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace

bool dgrad_lnbwd_supported(int C, int K) { return (C == 128 || C == 256) && K % BK == 0 && K >= BK; }

// dx (fp32 and / or bf16) = LayerNorm'(dY W) + dres;  dgamma / dbeta accumulate (+=).  dY bf16 (T, K), W bf16 (K, C).
int launch_dgrad_lnbwd(const void* dY, const void* W, int K, const float* x, const float* stats, const float* gamma,
                       const float* dres, float* dx, void* dx_bf16, float* dgamma, float* dbeta, int T, int C, int device,
                       cudaStream_t st) {
  CRF_CHECK(dY && W && x && stats && gamma && dgamma && dbeta && (dx || dx_bf16), "dgrad_lnbwd: null pointer");
  CRF_CHECK(T > 0 && dgrad_lnbwd_supported(C, K), "dgrad_lnbwd: unsupported shape (T=%d C=%d K=%d)", T, C, K);
  switch (C) {
    case 128: return launch_c<128>(dY, W, K, x, stats, gamma, dres, dx, dx_bf16, dgamma, dbeta, T, device, st);
    default: return launch_c<256>(dY, W, K, x, stats, gamma, dres, dx, dx_bf16, dgamma, dbeta, T, device, st);
  }
}

}  // namespace crf
