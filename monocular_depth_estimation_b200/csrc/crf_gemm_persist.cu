// Persistent variant of the TMA-fed tcgen05 GEMM for the token-major projections (fprop / dgrad, A K-major).
//
// Same tiles, descriptors and epilogue math as gemm_kernel (crf_gemm.cu), but one CTA per SM loops over output
// tiles and the three stages of a tile run CONCURRENTLY on different tiles:
//
//   warp 16        TMA producer : keeps the 3- or 5-stage A/B ring (see Plan) full across tile boundaries
//   warp 17        MMA issuer   : accumulates tile i into TMEM buffer i % 4 (4 x 128 columns = all 512 columns)
//   warps 0-15     epilogue     : four groups of four warps; group g drains the tiles with i % 4 == g
//                                 (thread = accumulator row), each group with its own output / aux slab buffers
//
// so the epilogue warps -- which bound these GEMMs (GELU, conversions, HBM stores) -- never wait for a main loop,
// and barrier init / TMEM allocation / descriptor prefetch are paid once per SM instead of once per tile.
// Barriers: full/empty[stages] (TMA <-> MMA), tmem_full[4] (MMA -> epilogue, tcgen05.commit), tmem_empty[4]
// (epilogue -> MMA, 128 arrivals), aux[4] (TMA aux-slab loads of each group).
#include "crf_gemm_epi.cuh"

namespace crf {

namespace {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int kAcc = 4;
constexpr int kThreads = 576;  // 16 epilogue warps + TMA warp + MMA warp
constexpr int kATile = BM * 128, kBTile = BN * 128, kStage = kATile + kBTile;  // 16 KB + 16 KB
constexpr int kSlab = BM * 128;                                                // 16 KB
// Shared-memory plan per epilogue: each of the four epilogue groups owns an output slab and, if the epilogue reads an
// aux tile or writes a second output, a second slab; whatever is left of the 227 KB goes to the A/B ring:
// 3 stages (96 KB) with two slabs per group, 5 stages (160 KB) with one (plain stores: qk, the dX GEMMs).
template <int EPI>
struct Plan {
  static constexpr int kSlabsPerGroup = (EpiTraits<EPI>::kHasAux || EpiTraits<EPI>::kHasOut1) ? 2 : 1;
  static constexpr int kSlabBytes = kAcc * kSlabsPerGroup * kSlab;
  static constexpr int kStages = kSlabsPerGroup == 2 ? 3 : 5;
  static constexpr int kRing = kStages * kStage;
  static constexpr int kBarOff = kRing + kSlabBytes;
  static constexpr int kNumBars = 2 * kStages + 3 * kAcc;
  static constexpr int kSmemBytes = kBarOff + 8 * kNumBars + 16 + 1024;
  static_assert(kSmemBytes <= 232448, "shared-memory plan exceeds 227 KB");
};

template <int EPI>
__global__ void __launch_bounds__(kThreads, 1)
gemm_persistent_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       const __grid_constant__ CUtensorMap tmO0, const __grid_constant__ CUtensorMap tmO1,
                       const __grid_constant__ CUtensorMap tmAux, int M, int N, int K, int b_major, EpiParams ep,
                       int splits) {
  pdl_launch_dependents();
  // splits > 1 (fp32-output epilogues only): every output tile is computed by `splits` work units, each over a
  // contiguous range of K chunks, and every unit ADDS its fp32 tile into the (zero-filled) output with a TMA reduction;
  // unit 0 of a tile also adds the bias / residual.  Used where the tile count quantises badly on the SM count
  // (M = 2400 at the 1/32 scale: 152 tiles on 148 SMs = a whole second round for 4 tiles).
  using TR = EpiTraits<EPI>;
  using PL = Plan<EPI>;
  constexpr int kStages = PL::kStages, kRing = PL::kRing, kBarOff = PL::kBarOff, kNumBars = PL::kNumBars;
  constexpr int kGroupSlabs = PL::kSlabsPerGroup * kSlab;
  constexpr int kSlabCols = TR::kSlabCols;
  constexpr int kNumSlabs = BN / kSlabCols;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar0 = base + kBarOff;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * kStages + kAcc + a); };
  auto aux_bar = [&](int a) { return bar0 + 8u * (2 * kStages + 2 * kAcc + a); };
  const uint32_t tmem_ptr_addr = bar0 + 8u * kNumBars;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen + kBarOff + 8 * kNumBars);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = N / BN;
  const int total_tiles = ((M + BM - 1) / BM) * n_tiles;
  const int nk_all = (K + BK - 1) / BK;
  const int nk_split = (nk_all + splits - 1) / splits;          // K chunks per work unit (the last one may be shorter)
  const int total_units = total_tiles * splits;                 // unit u: tile u % total_tiles, split u / total_tiles
  const int my_tiles = (total_units - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 16 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmO0);
    if (TR::kHasOut1) tma_prefetch_desc(&tmO1);
    if (TR::kHasAux) tma_prefetch_desc(&tmAux);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < kAcc; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 128);
      mbar_init(aux_bar(a), 1);
    }
    fence_mbar_init();
  }
  if (warp == 17) {
    tmem_alloc(tmem_ptr_addr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 16) {
    // ===== TMA producer =====
    if (lane == 0) {
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int u = blockIdx.x + i * gridDim.x;
        const int t = u % total_tiles, sp = u / total_tiles;
        const int m0 = (t / n_tiles) * BM, n0 = (t % n_tiles) * BN;
        const int kc0 = sp * nk_split, kc1 = min(nk_all, kc0 + nk_split);
        for (int kc = kc0; kc < kc1; ++kc, ++it) {
          const int s = it % kStages;
          if (it >= kStages) mbar_wait(empty_bar(s), ((it / kStages) - 1) & 1);
          const uint32_t a_dst = base + s * kStage, b_dst = a_dst + kATile;
          mbar_expect_tx(full_bar(s), kStage);
          tma_load_2d(a_dst, &tmA, full_bar(s), kc * BK, m0);
          if (b_major == 0) {
            tma_load_2d(b_dst, &tmB, full_bar(s), kc * BK, n0);
          } else {
            tma_load_2d(b_dst, &tmB, full_bar(s), n0, kc * BK);
            tma_load_2d(b_dst + 8192, &tmB, full_bar(s), n0 + 64, kc * BK);
          }
        }
      }
    }
  } else if (warp == 17) {
    // ===== MMA issuer =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc(1u, 0u, static_cast<uint32_t>(b_major), BM, BN);
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int a = i % kAcc;
        if (i >= kAcc) {
          mbar_wait(tempty_bar(a), ((i / kAcc) - 1) & 1);  // the epilogue has drained this accumulator buffer
          tc_fence_after();
        }
        const uint32_t d_tmem = tmem_base + a * BN;
        const int sp = (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) / total_tiles;
        const int kc0 = sp * nk_split, kc1 = min(nk_all, kc0 + nk_split);
        for (int kc = kc0; kc < kc1; ++kc, ++it) {
          const int s = it % kStages;
          mbar_wait(full_bar(s), (it / kStages) & 1);
          tc_fence_after();
          const uint32_t a_src = base + s * kStage, b_src = a_src + kATile;
#pragma unroll
          for (int ks = 0; ks < BK / 16; ++ks) {
            const uint64_t ad = make_smem_desc(a_src + ks * 32, 16, 1024, kSwizzle128);
            const uint64_t bd = (b_major == 0) ? make_smem_desc(b_src + ks * 32, 16, 1024, kSwizzle128)
                                               : make_smem_desc(b_src + ks * 2048, 8192, 1024, kSwizzle128);
            umma_bf16(d_tmem, ad, bd, idesc, (kc > kc0 || ks > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(a));
      }
    }
  } else {
    // ===== epilogue groups =====
    const int g = warp >> 2;
    const int r = threadIdx.x & 127;
    const uint32_t out0_s = base + kRing + g * kGroupSlabs, x_s = out0_s + kSlab;  // x_s only with two slabs / group
    uint8_t* o0 = gen + kRing + g * kGroupSlabs;
    uint8_t* xb = o0 + kSlab;
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    int aux_cnt = 0;
    for (int i = g, n_i = 0; i < my_tiles; i += kAcc, ++n_i) {
      const int u = blockIdx.x + i * gridDim.x;
      const int t = u % total_tiles;
      const bool first_split = u < total_tiles;   // the unit that also adds bias / residual
      const int m0 = (t / n_tiles) * BM, n0 = (t % n_tiles) * BN;
      const uint32_t taddr = tmem_base + g * BN + lane_base;
      if (TR::kHasAux && first_split && r == 0) {  // first aux slab of the tile; the buffer was consumed before the last barrier
        mbar_expect_tx(aux_bar(g), kSlab);
        tma_load_2d(x_s, &tmAux, aux_bar(g), n0, m0);
      }
      mbar_wait(tfull_bar(g), n_i & 1);
      tc_fence_after();
#pragma unroll 1
      for (int s = 0; s < kNumSlabs; ++s) {
        const int nc = n0 + s * kSlabCols;
        if (r == 0) bulk_wait_read<0>();  // previous TMA store of this group has drained its slab buffers
        named_bar_sync(1 + g, 128);
        if (TR::kHasAux && first_split) {
          mbar_wait(aux_bar(g), aux_cnt & 1);
          ++aux_cnt;
        }
#pragma unroll
        for (int half = 0; half < kSlabCols / 32; ++half) {
          uint32_t acc[32];
          tmem_ld32(taddr + s * kSlabCols + half * 32, acc);
          tmem_ld_wait();
          if (TR::kOutF32 && !first_split) {   // later K splits contribute the bare partial product
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<float4*>(o0 + sw128_offset(r, j)) =
                  make_float4(__uint_as_float(acc[4 * j]), __uint_as_float(acc[4 * j + 1]), __uint_as_float(acc[4 * j + 2]),
                              __uint_as_float(acc[4 * j + 3]));
          } else {
            epi_group32<EPI>(acc, ep, nc + half * 32, r, half, o0, xb);
          }
        }
        if (s == kNumSlabs - 1) {  // accumulator fully read: hand the TMEM buffer back to the MMA warp
          tc_fence_before();
          mbar_arrive(tempty_bar(g));
        }
        fence_proxy_async_smem();
        named_bar_sync(1 + g, 128);
        if (r == 0) {
          if (TR::kOutF32 && splits > 1) tma_reduce_add_2d(&tmO0, out0_s, nc, m0);
          else if (EPI != CRF_EPI_BIAS_GELU || ep.store_out0) tma_store_2d(&tmO0, out0_s, nc, m0);
          if (TR::kHasOut1) tma_store_2d(&tmO1, x_s, nc, m0);
          bulk_commit();
          if (TR::kHasAux && first_split && s + 1 < kNumSlabs) {
            mbar_expect_tx(aux_bar(g), kSlab);
            tma_load_2d(x_s, &tmAux, aux_bar(g), nc + kSlabCols, m0);
          }
        }
      }
    }
    if (r == 0) bulk_wait_read<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 17) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int EPI>
int launch_p(const GemmMaps& m, const crf_gemm_args& a, cudaStream_t st) {
  auto kern = gemm_persistent_kernel<EPI>;
  constexpr int kSmemBytes = Plan<EPI>::kSmemBytes;
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int tiles = ((a.M + BM - 1) / BM) * (a.N / BN);
  const int sms = num_sms(a.device);
  // K splits for the fp32-output epilogues when the tile count quantises badly on the SM count: pick the split count
  // (<= 4, >= 512 K elements per unit) that minimises rounds / splits.
  int splits = 1;
  if (EpiTraits<EPI>::kOutF32 && tiles >= sms / 2) {
    double best = static_cast<double>((tiles + sms - 1) / sms);
    for (int s = 2; s <= 4 && a.K / s >= 512; ++s) {
      const double cost = static_cast<double>((tiles * s + sms - 1) / sms) / s + 0.04 * (s - 1);  // + per-unit overhead
      if (cost < best - 1e-9) { best = cost; splits = s; }
    }
  }
  if (splits > 1) CRF_CUDA(cudaMemsetAsync(a.out0, 0, static_cast<size_t>(a.M) * a.N * sizeof(float), st));
  int grid = sms;
  if (grid > tiles * splits) grid = tiles * splits;
  KernelTimer tm(st, 2.0 * a.M * a.N * a.K, gemm_bytes(a, EPI), "gemm_%s_epi%d_M%d_N%d_K%d",
                 a.b_major ? "dgrad" : "fprop", EPI, a.M, a.N, a.K);
  launch_pdl(kern, grid, kThreads, kSmemBytes, st, m.tmA, m.tmB, m.tmO0, m.tmO1, m.tmAux, a.M, a.N, a.K, a.b_major,
             epi_params(a, 0, 0), splits);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace

// fprop / dgrad (A K-major), N a multiple of 128, no split-K (plan_gemm, crf_sched.h).
int launch_gemm_persistent(const crf_gemm_args& a, const GemmMaps& m, cudaStream_t st) {
  return with_epi(a.epilogue, [&](auto e) {
    constexpr int EPI = decltype(e)::value;
    if constexpr (EPI == CRF_EPI_SPLITK_F32) return set_error("crf_gemm: the persistent kernel has no split-K epilogue");
    else return launch_p<EPI>(m, a, st);
  });
}

}  // namespace crf
