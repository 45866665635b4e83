// TMA-fed tcgen05 GEMM used for every dense projection of the CRF block, forward and backward:
//   D[M,N] = sum_k A(m,k) * B(n,k),  bf16 operands, fp32 accumulation in TMEM.
//
//   fprop  (qk, proj, fc1, fc2)    : A = activations (tokens, Cin)  K-major, B = weight (Cout, Cin) K-major
//   dgrad  (dX = dY * W)           : A = dY (tokens, Cout)          K-major, B = weight (Cout, Cin) MN-major
//   wgrad  (dW = dY^T * X)         : A = dY (tokens, Cout) MN-major, B = X (tokens, Cin) MN-major, split-K over tokens
//
// Both orientations read the SAME smem tile format: rows of 64 bf16 (128 B) with the 128-byte swizzle, as
// written by a TMA box (64 cols x R rows).  A K-major operand uses one box of R = tile rows; an MN-major
// operand uses (tile MN extent / 64) boxes of 64 K-rows each, 8 KB apart (the descriptor's leading byte offset).
//
// CTA = 10 warps: warps 0-7 epilogue (two groups of four; thread = accumulator row = TMEM lane; the groups take
// alternate column slabs, which doubles the warps available to hide the GELU / conversion latency), warp 8 TMA
// producer, warp 9 MMA issuer + TMEM allocator.  One 128 x BN output tile per CTA, K streamed in 64-element chunks through a
// multi-stage mbarrier ring.  Two CTAs are co-resident per SM (<= 256 TMEM columns, <= ~100 KB smem each) so
// one CTA's epilogue overlaps the other's main loop.
//
// Epilogue: these GEMMs are HBM-bound at the small-C decoder scales, so output and auxiliary traffic goes through
// TMA as well.  The accumulator is drained in 128-byte-wide column slabs (64 bf16 or 32 fp32 columns): each thread
// writes its row of the slab into a swizzled smem tile (conflict-free), one thread issues a TMA store of the
// [128 x 128 B] box (rows beyond M are clipped by the tensor map), double-buffered.  Residual / pre-activation
// tiles the epilogue needs are TMA-loaded into the same kind of slab one step ahead.  The slabs alias the
// main-loop stages, which are dead once the accumulator barrier has fired.
//
// Split-K (weight gradients): each split stores its fp32 partial tile into a workspace [splits][Mpad][N] and a
// second kernel reduces the partials into dW (+=): deterministic, and no per-element L2 atomics.
#include <stdlib.h>

#include "crf_gemm_epi.cuh"
#include "crf_sched.h"

namespace crf {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kThreads = 320;  // 8 epilogue warps (two groups of 4), 1 TMA warp, 1 MMA warp
constexpr int kATileBytes = BM * 128;  // 16 KB
constexpr int kSlabBytes = BM * 128;   // 16 KB: 128 rows x 128 B

template <int BN, int EPI>
__global__ void __launch_bounds__(kThreads)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmO0, const __grid_constant__ CUtensorMap tmO1,
            const __grid_constant__ CUtensorMap tmAux, int M, int N, int total_chunks, int chunks_per_split, int stages,
            int a_major, int b_major, EpiParams ep, int chunks_per_part, int a_off, int b_off) {
  pdl_prologue();
  // chunks_per_part > 0: split-operand mode (crf_gemm_args.split3).  Both operands are stored as [hi | lo] halves side
  // by side and the K loop runs three times: chunk kc belongs to part kc / chunks_per_part = 0: hi*hi, 1: hi*lo(B),
  // 2: lo(A)*hi; the lo half of an operand is a_off / b_off elements further along its contiguous dimension.
  constexpr int kBTileBytes = BN * 128;
  constexpr int kStageBytes = kATileBytes + kBTileBytes;
  // Bias gradient for free: one extra N=16 MMA per K step against an all-ones B tile puts sum_k A(m,k) into 16
  // spare TMEM columns (every column holds the same sum); needs the next power of two of TMEM columns.
  const int kc_begin = blockIdx.z * chunks_per_split;
  const int kc_end = min(total_chunks, kc_begin + chunks_per_split);
  // split-operand mode: the column sums of A = hi + lo come from parts 0 (hi) and 2 (lo) only
  const bool cs_any = chunks_per_part == 0 || kc_begin < chunks_per_part || kc_end > 2 * chunks_per_part;
  const bool do_colsum = ep.colsum != nullptr && blockIdx.y == 0 && cs_any;
  const uint32_t kTmemCols = ep.colsum != nullptr ? 2u * BN : (BN < 32 ? 32u : static_cast<uint32_t>(BN));
  using TR = EpiTraits<EPI>;
  constexpr int kSlabCols = TR::kSlabCols;
  constexpr int kNumSlabs = BN / kSlabCols;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int nk = kc_end - kc_begin;
  if (nk <= 0) return;  // uniform for the whole CTA

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  // barriers live after the stage ring: full[stages], empty[stages], tmem_full, aux[2], tmem_ptr
  const uint32_t ring_bytes = static_cast<uint32_t>(stages) * kStageBytes < 4u * kSlabBytes
                                  ? 4u * kSlabBytes
                                  : static_cast<uint32_t>(stages) * kStageBytes;
  const uint32_t bar_base = smem_base + ring_bytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (stages + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * stages);
  auto aux_bar = [&](int s) { return bar_base + 8u * (2 * stages + 1 + s); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * stages + 3);
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + ring_bytes + 8 * (2 * stages + 3));
  const uint32_t ones_addr = bar_base + 8u * (2 * stages + 4);  // 1 KB of bf16 1.0 (any UMMA layout of it is all ones)
  if (ep.colsum != nullptr && threadIdx.x < 64) {
    *reinterpret_cast<uint4*>(smem_gen + ring_bytes + 8 * (2 * stages + 4) + 16 * threadIdx.x) =
        make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async_smem();
  }

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmO0);
    if (TR::kHasOut1) tma_prefetch_desc(&tmO1);
    if (TR::kHasAux) tma_prefetch_desc(&tmAux);
    for (int s = 0; s < stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(aux_bar(0), 1);
    mbar_init(aux_bar(1), 1);
    fence_mbar_init();
  }
  if (warp == 9) {
    tmem_alloc(tmem_ptr_addr, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 8) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int i = 0; i < nk; ++i) {
        const int s = i % stages;
        if (i >= stages) mbar_wait(empty_bar(s), ((i / stages) - 1) & 1);
        const uint32_t a_dst = smem_base + s * kStageBytes;
        const uint32_t b_dst = a_dst + kATileBytes;
        mbar_expect_tx(full_bar(s), kStageBytes);
        const int kc = kc_begin + i;
        const int part = chunks_per_part ? kc / chunks_per_part : 0;
        const int k0 = (kc - part * chunks_per_part) * BK;
        const int ao = part == 2 ? a_off : 0, bo = part == 1 ? b_off : 0;
        if (a_major == 0) {
          tma_load_2d(a_dst, &tmA, full_bar(s), k0 + ao, m0);
        } else {
#pragma unroll
          for (int j = 0; j < BM / 64; ++j) tma_load_2d(a_dst + j * 8192, &tmA, full_bar(s), m0 + 64 * j + ao, k0);
        }
        if (b_major == 0) {
          tma_load_2d(b_dst, &tmB, full_bar(s), k0 + bo, n0);
        } else {
#pragma unroll
          for (int j = 0; j < BN / 64; ++j) tma_load_2d(b_dst + j * 8192, &tmB, full_bar(s), n0 + 64 * j + bo, k0);
        }
      }
    }
  } else if (warp == 9) {
    // ===== MMA issuer =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc(1u, static_cast<uint32_t>(a_major), static_cast<uint32_t>(b_major), BM, BN);
      uint32_t cs_acc = 0u;
      for (int i = 0; i < nk; ++i) {
        const bool cs_part = chunks_per_part == 0 || (kc_begin + i) / chunks_per_part != 1;
        const int s = i % stages;
        mbar_wait(full_bar(s), (i / stages) & 1);
        tc_fence_after();
        const uint32_t a_src = smem_base + s * kStageBytes;
        const uint32_t b_src = a_src + kATileBytes;
#pragma unroll
        for (int ks = 0; ks < BK / 16; ++ks) {
          const uint64_t ad = (a_major == 0) ? make_smem_desc(a_src + ks * 32, 16, 1024, kSwizzle128)
                                             : make_smem_desc(a_src + ks * 2048, 8192, 1024, kSwizzle128);
          const uint64_t bd = (b_major == 0) ? make_smem_desc(b_src + ks * 32, 16, 1024, kSwizzle128)
                                             : make_smem_desc(b_src + ks * 2048, 8192, 1024, kSwizzle128);
          umma_bf16(tmem_base, ad, bd, idesc, (i > 0 || ks > 0) ? 1u : 0u);
          if (do_colsum && cs_part) {  // K-major, no swizzle: 8x16-byte core matrices, 128 B apart along K, 256 B along N
            umma_bf16(tmem_base + BN, ad, make_smem_desc(ones_addr, 128, 256, kSwizzleNone),
                      make_idesc(1u, static_cast<uint32_t>(a_major), 0u, BM, 16), cs_acc);
            cs_acc = 1u;
          }
        }
        umma_commit(empty_bar(s));  // frees the smem stage once these MMAs have read it
      }
      umma_commit(tmem_full_bar);  // accumulator complete (and every smem stage is dead from here on)
    }
  } else {
    // ===== epilogue: thread = accumulator row; slabs staged in smem, moved by TMA =====
    // Group e (warps 4e..4e+3) drains slabs e, e+2, ...; each group owns one output slab and one aux/out1 slab.
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const int e = warp >> 2;
    const int r = threadIdx.x & 127;
    const int buf = e;
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    const uint32_t out0_s = smem_base, x_s = smem_base + 2 * kSlabBytes;
    uint8_t* out0_g = smem_gen;
    uint8_t* x_g = smem_gen + 2 * kSlabBytes;
    const bool tma_red = (EPI == CRF_EPI_SPLITK_F32) && ep.tma_reduce != 0;
    const int out_row0 = (EPI == CRF_EPI_SPLITK_F32 && !tma_red) ? static_cast<int>(blockIdx.z) * ep.m_pad + m0 : m0;

    if (TR::kHasAux && r == 0 && e < kNumSlabs) {
      mbar_expect_tx(aux_bar(e), kSlabBytes);
      tma_load_2d(x_s + buf * kSlabBytes, &tmAux, aux_bar(e), n0 + e * kSlabCols, m0);
    }
#pragma unroll 1
    for (int s = e, it = 0; s < kNumSlabs; s += 2, ++it) {
      const int nc = n0 + s * kSlabCols;
      if (r == 0) bulk_wait_read<0>();  // this group's previous store has drained its slab buffers
      named_bar_sync(1 + e, 128);
      if (TR::kHasAux) mbar_wait(aux_bar(e), it & 1);
      uint8_t* o0 = out0_g + buf * kSlabBytes;
      uint8_t* xb = x_g + buf * kSlabBytes;
#pragma unroll
      for (int half = 0; half < kSlabCols / 32; ++half) {
        uint32_t acc[32];
        tmem_ld32(taddr + s * kSlabCols + half * 32, acc);
        tmem_ld_wait();
        epi_group32<EPI>(acc, ep, nc + half * 32, r, half, o0, xb);
      }
      fence_proxy_async_smem();
      named_bar_sync(3 + e, 128);
      if (r == 0) {
        if (tma_red) tma_reduce_add_2d(&tmO0, out0_s + buf * kSlabBytes, nc, out_row0);
        else if (EPI != CRF_EPI_BIAS_GELU || ep.store_out0) tma_store_2d(&tmO0, out0_s + buf * kSlabBytes, nc, out_row0);
        if (TR::kHasOut1) tma_store_2d(&tmO1, x_s + buf * kSlabBytes, nc, out_row0);
        bulk_commit();
        if (TR::kHasAux && s + 2 < kNumSlabs) {  // the aux slab was consumed before the barrier above: refill it
          mbar_expect_tx(aux_bar(e), kSlabBytes);
          tma_load_2d(x_s + buf * kSlabBytes, &tmAux, aux_bar(e), nc + 2 * kSlabCols, m0);
        }
      }
    }
    if (r == 0) bulk_wait_read<0>();
    if (do_colsum && e == 0) {  // warp-uniform: group 0 drains the spare accumulator columns
      uint32_t cs[32];
      tmem_ld32(taddr + BN, cs);
      tmem_ld_wait();
      if (m0 + r < M) atomicAdd(ep.colsum + m0 + r, __uint_as_float(cs[0]));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// dW[m,n] += sum_z part[z][m][n]
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ part, float* __restrict__ out, int M, int N, int m_pad, int splits) {
  pdl_prologue();
  const int64_t i4 = static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x;
  const int64_t total4 = static_cast<int64_t>(M) * N / 4;
  if (i4 >= total4) return;
  const int64_t e = i4 * 4;
  const int m = static_cast<int>(e / N), n = static_cast<int>(e - static_cast<int64_t>(m) * N);
  float4 acc = *reinterpret_cast<const float4*>(out + e);
  const float* p = part + static_cast<int64_t>(m) * N + n;
  const int64_t zs = static_cast<int64_t>(m_pad) * N;
#pragma unroll 4
  for (int z = 0; z < splits; ++z) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p + z * zs));
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(out + e) = acc;
}

struct Launch {
  int total_chunks, cps, splits, m_pad;
  int tma_reduce = 0;
  int chunks_per_part = 0, a_off = 0, b_off = 0;  // split-operand mode
};

template <int BN, int EPI>
int launch_one(const GemmMaps& m, const Launch& L, const crf_gemm_args& a, cudaStream_t st) {
  constexpr int kStageBytes = kATileBytes + BN * 128;
  // 2 co-resident CTAs/SM when K is short; one deep ring when K is long.
  // wgrad: one CTA per SM streams a long token range -> deep ring.  fprop/dgrad: these are epilogue-bound (GELU,
  // conversions, HBM stores), so favour residency: 128-wide tiles with a 2-stage ring = 3 CTAs per SM whose
  // main loops and epilogues interleave (measured: -0.5 ms per training step vs 256-wide tiles, 2 CTAs per SM).
  int stages = a.a_major == 1 ? ((L.cps >= 8) ? (BN == 256 ? 4 : 6) : (BN == 256 ? 2 : 3)) : 2;
  if (stages > L.cps) stages = L.cps < 2 ? 2 : L.cps;
  size_t ring = static_cast<size_t>(stages) * kStageBytes;
  if (ring < 4u * kSlabBytes) ring = 4u * kSlabBytes;
  const size_t smem = ring + 1024 + 8 * (2 * stages + 4) + 1024;  // + align slack, barriers, ones tile
  auto kern = gemm_kernel<BN, EPI>;
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const EpiParams ep = epi_params(a, L.m_pad, L.tma_reduce);
  dim3 grid((a.M + BM - 1) / BM, a.N / BN, L.splits);
  KernelTimer tm(st, 2.0 * a.M * a.N * a.K, gemm_bytes(a, EPI), "gemm%s_%s_epi%d_M%d_N%d_K%d", a.split3 ? "3" : "",
                 a.a_major ? "wgrad" : (a.b_major ? "dgrad" : "fprop"), EPI, a.M, a.N, a.K);
  launch_pdl(kern, grid, kThreads, smem, st, m.tmA, m.tmB, m.tmO0, m.tmO1, m.tmAux, a.M, a.N, L.total_chunks, L.cps, stages,
             a.a_major, a.b_major, ep, L.chunks_per_part, L.a_off, L.b_off);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

int launch_tiled(int BN, const GemmMaps& m, const Launch& L, const crf_gemm_args& a, int epi, cudaStream_t st) {
  return with_epi(epi, [&](auto e) {
    constexpr int EPI = decltype(e)::value;
    switch (BN) {
      case 256: return launch_one<256, EPI>(m, L, a, st);
      case 128: return launch_one<128, EPI>(m, L, a, st);
      default: return launch_one<64, EPI>(m, L, a, st);
    }
  });
}

}  // namespace

int gemm_maps(const crf_gemm_args& a, uint32_t b_rows, GemmMaps* m) {
  const uint64_t dup = a.split3 ? 2 : 1;  // split-operand matrices are twice as wide: [hi | lo]
  if (a.a_major == 0 ? make_tmap_bf16(&m->tmA, a.A, a.M, dup * a.K, BM) : make_tmap_bf16(&m->tmA, a.A, a.K, dup * a.M, 64))
    return 1;
  if (a.b_major == 0 ? make_tmap_bf16(&m->tmB, a.B, a.N, dup * a.K, b_rows) : make_tmap_bf16(&m->tmB, a.B, a.K, dup * a.N, 64))
    return 1;
  m->tmO0 = m->tmO1 = m->tmAux = m->tmA;
  const int epi = a.epilogue;
  if (epi == CRF_EPI_BIAS_GELU) {
    CRF_CHECK(a.out1 != nullptr, "crf_gemm: BIAS_GELU needs out1");
    if (a.out0 != nullptr && make_tmap_bf16(&m->tmO0, a.out0, a.M, a.N, BM)) return 1;
    if (make_tmap_bf16(&m->tmO1, a.out1, a.M, a.N, BM)) return 1;
  } else {
    CRF_CHECK(a.out0 != nullptr, "crf_gemm: out0 is null");
    const bool out_f32 = epi == CRF_EPI_STORE_F32 || epi == CRF_EPI_BIAS_RES_F32 || epi == CRF_EPI_SPLITK_F32;
    if (out_f32 ? make_tmap_f32(&m->tmO0, a.out0, a.M, a.N, BM) : make_tmap_bf16(&m->tmO0, a.out0, a.M, a.N, BM)) return 1;
  }
  if (epi == CRF_EPI_BIAS_RES_F32) {
    CRF_CHECK(a.aux1 != nullptr, "crf_gemm: BIAS_RES_F32 needs aux1 (residual)");
    if (make_tmap_f32(&m->tmAux, a.aux1, a.M, a.N, BM)) return 1;
  } else if (epi == CRF_EPI_MUL_DGELU) {
    CRF_CHECK(a.aux1 != nullptr, "crf_gemm: MUL_DGELU needs aux1 (pre-activation)");
    if (make_tmap_bf16(&m->tmAux, a.aux1, a.M, a.N, BM)) return 1;
  }
  return 0;
}

// Number of K splits a weight-gradient GEMM will use and the fp32 partial-tile workspace it needs.  The tile width is
// gemm_tile_n(N) without the cap plan_gemm applies to K-major A: the split-K GEMMs of the library have MN-major A.
size_t gemm_splitk_workspace_bytes(int M, int N, int K, int device, int* splits_out) {
  const int BN = gemm_tile_n(N);
  const int tiles = ((M + BM - 1) / BM) * (N / BN);
  const int chunks = (K + BK - 1) / BK;
  int s = num_sms(device) / tiles;  // about one CTA per SM, each with a deep pipeline over its token range
  if (s > chunks) s = chunks;
  if (s < 1) s = 1;
  if (splits_out) *splits_out = s;
  if (s == 1) return 0;
  const size_t m_pad = static_cast<size_t>((M + BM - 1) / BM) * BM;
  return static_cast<size_t>(s) * m_pad * N * sizeof(float);
}

int launch_gemm(const crf_gemm_args& a, cudaStream_t st) {
  CRF_CHECK(a.M > 0 && a.N > 0 && a.K > 0, "crf_gemm: empty problem M=%d N=%d K=%d", a.M, a.N, a.K);
  CRF_CHECK(a.N % 64 == 0, "crf_gemm: N=%d must be a multiple of 64", a.N);
  CRF_CHECK(a.a_major == 0 || a.a_major == 1, "crf_gemm: bad a_major");
  CRF_CHECK(a.b_major == 0 || a.b_major == 1, "crf_gemm: bad b_major");
  CRF_CHECK(a.a_major == 1 || a.K % 8 == 0, "crf_gemm: K-major A needs K %% 8 == 0 (K=%d)", a.K);
  CRF_CHECK(a.a_major == 0 || a.M % 8 == 0, "crf_gemm: MN-major A needs M %% 8 == 0 (M=%d)", a.M);
  CRF_CHECK(a.ld_out == a.N, "crf_gemm: outputs must be dense (ld_out == N)");
  if (a.split3) {
    CRF_CHECK((a.a_major == 1 || a.K % BK == 0) && (a.b_major == 1 || a.K % BK == 0),
              "crf_gemm: split3 with a K-major operand needs K %% 64 == 0 (K=%d)", a.K);
    CRF_CHECK((a.a_major == 0 || a.M % 64 == 0), "crf_gemm: split3 with MN-major A needs M %% 64 == 0 (M=%d)", a.M);
    CRF_CHECK(a.epilogue == CRF_EPI_STORE_F32 || a.epilogue == CRF_EPI_BIAS_RES_F32 || a.epilogue == CRF_EPI_SPLITK_F32,
              "crf_gemm: split3 supports the fp32 epilogues only");
  }
  const GemmPlan plan = plan_gemm(a.M, a.N, a.K, a.a_major, a.epilogue, a.split3);
  GemmMaps m;
  // the pair and persistent kernels load 128 rows of B per CTA and K step
  if (gemm_maps(a, plan.kernel == kGemmTiled ? plan.bn : 128, &m)) return 1;
  if (plan.kernel == kGemmPair) return launch_gemm_pair(a, m, st);
  if (plan.kernel == kGemmPersistent) return launch_gemm_persistent(a, m, st);

  Launch L{};
  L.total_chunks = (a.K + BK - 1) / BK;
  if (a.split3) {
    L.chunks_per_part = L.total_chunks;
    L.total_chunks *= 3;
    L.a_off = a.a_major == 0 ? a.K : a.M;
    L.b_off = a.b_major == 0 ? a.K : a.N;
  }
  L.splits = 1;
  L.cps = L.total_chunks;
  L.m_pad = (a.M + BM - 1) / BM * BM;
  const int epi = a.epilogue;

  if (epi == CRF_EPI_SPLITK_F32) {
    // out0 (M,N) f32 += A^T B.  One split: in-place accumulate (residual = out0).  Otherwise partials + reduce.
    int splits = 1;
    gemm_splitk_workspace_bytes(a.M, a.N, a.split3 ? 3 * a.K : a.K, a.device, &splits);
    if (a.split_k > 0 && a.split_k < splits) splits = a.split_k;
    const size_t per_split = static_cast<size_t>(L.m_pad) * a.N * sizeof(float);
    static const bool deterministic = getenv("CRF_WGRAD_DETERMINISTIC") != nullptr && atoi(getenv("CRF_WGRAD_DETERMINISTIC")) != 0;
    if (splits > 1 && deterministic) {  // the partial tiles must fit the caller's workspace
      const size_t fit = a.workspace == nullptr ? 0 : a.workspace_bytes / per_split;
      if (fit < static_cast<size_t>(splits)) splits = fit < 1 ? 1 : static_cast<int>(fit);
    }
    crf_gemm_args b = a;
    b.bias = nullptr;
    if (splits <= 1) {
      m.tmAux = m.tmO0;
      return launch_tiled(plan.bn, m, L, b, CRF_EPI_BIAS_RES_F32, st);
    }
    L.cps = (L.total_chunks + splits - 1) / splits;
    L.splits = (L.total_chunks + L.cps - 1) / L.cps;  // no empty split
    // Default: every split ADDS its fp32 tile into dW with a TMA reduction (cp.reduce.async.bulk.tensor .add): no
    // partial buffer, no reduce kernel; the sum over splits is formed by the L2 in arrival order (fp32 round-off
    // depends on it).  CRF_WGRAD_DETERMINISTIC=1 keeps the partial tiles + fixed-order reduce kernel.
    if (!deterministic) {
      L.tma_reduce = 1;
      return launch_tiled(plan.bn, m, L, b, epi, st);
    }
    if (make_tmap_f32(&m.tmO0, a.workspace, static_cast<uint64_t>(L.splits) * L.m_pad, a.N, BM)) return 1;
    if (launch_tiled(plan.bn, m, L, b, epi, st)) return 1;
    const int64_t total4 = static_cast<int64_t>(a.M) * a.N / 4;
    KernelTimer tm(st, 0.0, 4.0 * a.M * a.N * (L.splits + 2), "splitk_reduce_M%d_N%d_S%d", a.M, a.N, L.splits);
    launch_pdl(splitk_reduce_kernel, static_cast<unsigned>((total4 + 255) / 256), 256, 0, st, 
        reinterpret_cast<const float*>(a.workspace), reinterpret_cast<float*>(a.out0), a.M, a.N, L.m_pad, L.splits);
    CRF_CUDA(cudaGetLastError());
    note_launch();
    return 0;
  }
  return launch_tiled(plan.bn, m, L, a, epi, st);
}

}  // namespace crf
