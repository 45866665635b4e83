// CTA-pair (cta_group::2) variant of the persistent token-major GEMM for the wide decoder scales (C >= 512):
// one tcgen05.mma covers a 256 x 256 output tile on the two SMs of a TPC.
//
// Why: with 128 x 128 single-CTA tiles every 2.1 MFLOP of MMA needs 32 KB of operands from L2 and 8 KB of shared-memory
// reads per K step -- the C >= 512 GEMMs sit at 350-550 TFLOP/s, L2- and smem-bandwidth-bound (DESIGN.md section 8).
// A CTA pair shares both: each CTA loads its 128 rows of A and only HALF of the 256 N columns of B (32 KB per CTA for
// 8.4 MFLOP per pair: half the L2 traffic per flop), the tensor cores of both SMs read B from both shared memories,
// and each CTA keeps its 128 accumulator rows (x 256 columns, double-buffered: all 512 TMEM columns) in its own TMEM.
//
//   both CTAs    warp 8   TMA producer: its A rows + its B half into its own ring; the bytes are accounted on the LEADER's
//                         `full` barrier (cp.async.bulk.tensor ... cta_group::2, peer bit of the barrier address cleared)
//   leader only  warp 9   MMA issuer: tcgen05.mma.cta_group::2 (M = 256, N = 256, K = 16 per instruction); tcgen05.commit
//                         ... multicast::cluster frees the ring stage in BOTH CTAs and publishes the accumulator to both
//   both CTAs    warps 0-7  epilogue, two groups of four warps (column halves), thread = accumulator row, the same slab
//                         epilogues as the single-CTA kernel (crf_gemm_epi.cuh); TMEM hand-back = one remote mbarrier
//                         arrival per warp on the leader's `tmem_empty` barrier
#include "crf_gemm_epi.cuh"

namespace crf {

namespace {

constexpr int PM = 256, PN = 256, BK = 64;   // pair tile
constexpr int kThreads = 320;                // 8 epilogue warps + TMA warp + MMA warp
constexpr int kATile = 128 * 128, kBTile = 128 * 128, kStage = kATile + kBTile;  // per CTA: 16 KB + 16 KB
constexpr int kStages = 4;
constexpr int kSlab = 128 * 128;
constexpr int kRing = kStages * kStage;                 // 128 KB
constexpr int kSlabOff = kRing;                         // 2 groups x (out slab + aux / second-output slab)
constexpr int kBarOff = kSlabOff + 4 * kSlab;           // 192 KB
constexpr int kNumBars = 2 * kStages + 2 + 2 + 2;       // full, empty, tmem_full[2], tmem_empty[2], aux[2]
constexpr int kSmemBytes = kBarOff + 8 * kNumBars + 16 + 1024;
static_assert(kSmemBytes <= 232448, "shared-memory plan exceeds 227 KB");

// Pair p takes whole tiles p, p + npairs, ... in the producer, the MMA issuer and the epilogue alike.
template <int EPI>
__global__ void __launch_bounds__(kThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO0, const __grid_constant__ CUtensorMap tmO1,
                 const __grid_constant__ CUtensorMap tmAux, int M, int N, int K, int b_major, EpiParams ep) {
  pdl_launch_dependents();
  using TR = EpiTraits<EPI>;
  constexpr int kSlabCols = TR::kSlabCols;
  constexpr int kNumSlabs = 128 / kSlabCols;   // per epilogue group (128 of the 256 columns)

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // identical in both CTAs (same kernel, same layout)
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar0 = base + kBarOff;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * kStages + 2 + a); };
  auto aux_bar = [&](int g) { return bar0 + 8u * (2 * kStages + 4 + g); };
  const uint32_t tmem_ptr_addr = bar0 + 8u * kNumBars;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen + kBarOff + 8 * kNumBars);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();             // 0 = leader
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int n_tiles = N / PN;
  const int total_tiles = ((M + PM - 1) / PM) * n_tiles;
  const int nk_all = (K + BK - 1) / BK;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmO0);
    if (TR::kHasOut1) tma_prefetch_desc(&tmO1);
    if (TR::kHasAux) tma_prefetch_desc(&tmAux);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);      // the leader's producer arrives (expect_tx); both CTAs' TMA bytes complete it
      mbar_init(empty_bar(s), 1);     // multicast tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);     // multicast tcgen05.commit
      mbar_init(tempty_bar(a), 16);   // 8 epilogue warps x 2 CTAs (used on the leader only)
      mbar_init(aux_bar(a), 1);
    }
    fence_mbar_init();
  }
  if (warp == 9) {
    tmem_alloc_2sm(tmem_ptr_addr, 512);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  cluster_sync_all();   // barriers of BOTH CTAs are initialised before anything signals across the pair
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 8) {
    // ===== TMA producer (both CTAs): A rows [m0 + 128 rank, +128), B columns [n0 + 128 rank, +128) =====
    if (lane == 0) {
      int it = 0;
      for (int t = pair; t < total_tiles; t += npairs) {
        const int m0 = (t / n_tiles) * PM + 128 * static_cast<int>(rank);
        const int n0 = (t % n_tiles) * PN + 128 * static_cast<int>(rank);
        for (int kc = 0; kc < nk_all; ++kc, ++it) {
          const int s = it % kStages;
          if (it >= kStages) mbar_wait(empty_bar(s), ((it / kStages) - 1) & 1);
          const uint32_t a_dst = base + s * kStage, b_dst = a_dst + kATile;
          if (rank == 0) mbar_expect_tx(full_bar(s), 2 * kStage);   // the bytes of both CTAs land on the leader's barrier
          tma_load_2d_2sm(a_dst, &tmA, full_bar(s), kc * BK, m0);
          if (b_major == 0) {
            tma_load_2d_2sm(b_dst, &tmB, full_bar(s), kc * BK, n0);
          } else {
            tma_load_2d_2sm(b_dst, &tmB, full_bar(s), n0, kc * BK);
            tma_load_2d_2sm(b_dst + 8192, &tmB, full_bar(s), n0 + 64, kc * BK);
          }
        }
      }
    }
  } else if (warp == 9) {
    // ===== MMA issuer (leader CTA only) =====
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc(1u, 0u, static_cast<uint32_t>(b_major), PM, PN);
      int it = 0;
      for (int t = pair, i = 0; t < total_tiles; t += npairs, ++i) {
        const int a = i & 1;
        if (i >= 2) {
          mbar_wait(tempty_bar(a), ((i >> 1) - 1) & 1);   // both CTAs' epilogues have drained this accumulator
          tc_fence_after();
        }
        const uint32_t d_tmem = tmem_base + a * PN;
        for (int kc = 0; kc < nk_all; ++kc, ++it) {
          const int s = it % kStages;
          mbar_wait(full_bar(s), (it / kStages) & 1);
          tc_fence_after();
          const uint32_t a_src = base + s * kStage, b_src = a_src + kATile;
#pragma unroll
          for (int ks = 0; ks < BK / 16; ++ks) {
            const uint64_t ad = make_smem_desc(a_src + ks * 32, 16, 1024, kSwizzle128);
            const uint64_t bd = (b_major == 0) ? make_smem_desc(b_src + ks * 32, 16, 1024, kSwizzle128)
                                               : make_smem_desc(b_src + ks * 2048, 8192, 1024, kSwizzle128);
            umma_bf16_2sm(d_tmem, ad, bd, idesc, (kc > 0 || ks > 0) ? 1u : 0u);
          }
          umma_commit_2sm(empty_bar(s), 3);   // frees the stage in both CTAs
        }
        umma_commit_2sm(tfull_bar(a), 3);     // accumulator complete, in both CTAs' TMEM
      }
    }
  } else {
    // ===== epilogue (both CTAs): group e drains accumulator columns [128 e, 128 e + 128) of this CTA's 128 rows =====
    const int e = warp >> 2;
    const int r = threadIdx.x & 127;
    const uint32_t out0_s = base + kSlabOff + e * 2 * kSlab, x_s = out0_s + kSlab;
    uint8_t* o0 = gen + kSlabOff + e * 2 * kSlab;
    uint8_t* xb = o0 + kSlab;
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    int aux_cnt = 0;
    for (int t = pair, i = 0; t < total_tiles; t += npairs, ++i) {
      const int a = i & 1;
      const int m0 = (t / n_tiles) * PM + 128 * static_cast<int>(rank);
      const int n0 = (t % n_tiles) * PN + 128 * e;
      const uint32_t taddr = tmem_base + a * PN + e * 128 + lane_base;
      if (TR::kHasAux && r == 0) {
        mbar_expect_tx(aux_bar(e), kSlab);
        tma_load_2d(x_s, &tmAux, aux_bar(e), n0, m0);
      }
      mbar_wait(tfull_bar(a), (i >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int s = 0; s < kNumSlabs; ++s) {
        const int nc = n0 + s * kSlabCols;
        if (r == 0) bulk_wait_read<0>();
        named_bar_sync(1 + e, 128);
        if (TR::kHasAux) {
          mbar_wait(aux_bar(e), aux_cnt & 1);
          ++aux_cnt;
        }
#pragma unroll
        for (int half = 0; half < kSlabCols / 32; ++half) {
          uint32_t acc[32];
          tmem_ld32(taddr + s * kSlabCols + half * 32, acc);
          tmem_ld_wait();
          epi_group32<EPI>(acc, ep, nc + half * 32, r, half, o0, xb);
        }
        if (s == kNumSlabs - 1) {  // this warp has read its part of the accumulator: one arrival per warp on the leader
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(tempty_bar(a), 0);
        }
        fence_proxy_async_smem();
        named_bar_sync(1 + e, 128);
        if (r == 0) {
          if (EPI != CRF_EPI_BIAS_GELU || ep.store_out0) tma_store_2d(&tmO0, out0_s, nc, m0);
          if (TR::kHasOut1) tma_store_2d(&tmO1, x_s, nc, m0);
          bulk_commit();
          if (TR::kHasAux && s + 1 < kNumSlabs) {
            mbar_expect_tx(aux_bar(e), kSlab);
            tma_load_2d(x_s, &tmAux, aux_bar(e), nc + kSlabCols, m0);
          }
        }
      }
    }
    if (r == 0) bulk_wait_read<0>();
  }

  tc_fence_before();
  cluster_sync_all();   // nobody leaves (or frees TMEM) while the peer can still be read by an MMA or signalled
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

template <int EPI>
int launch_pair(const GemmMaps& m, const crf_gemm_args& a, cudaStream_t st) {
  auto kern = gemm_pair_kernel<EPI>;
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int tiles = ((a.M + PM - 1) / PM) * (a.N / PN);
  const int max_pairs = num_sms(a.device) / 2;
  int pairs = max_pairs;
  if (pairs > tiles) pairs = tiles;
  KernelTimer tm(st, 2.0 * a.M * a.N * a.K, gemm_bytes(a, EPI), "gemm2_%s_epi%d_M%d_N%d_K%d",
                 a.b_major ? "dgrad" : "fprop", EPI, a.M, a.N, a.K);
  CRF_CUDA(launch_pdl_cluster(2, kern, 2 * pairs, kThreads, kSmemBytes, st, m.tmA, m.tmB, m.tmO0, m.tmO1, m.tmAux, a.M, a.N,
                              a.K, a.b_major, epi_params(a, 0, 0)));
  note_launch();
  return 0;
}

}  // namespace

// fprop / dgrad (A K-major) with N a multiple of 256 and enough work for CTA pairs (plan_gemm, crf_sched.h).
int launch_gemm_pair(const crf_gemm_args& a, const GemmMaps& m, cudaStream_t st) {
  return with_epi(a.epilogue, [&](auto e) {
    constexpr int EPI = decltype(e)::value;
    if constexpr (EPI == CRF_EPI_SPLITK_F32) return set_error("crf_gemm: the CTA-pair kernel has no split-K epilogue");
    else return launch_pair<EPI>(m, a, st);
  });
}

}  // namespace crf
