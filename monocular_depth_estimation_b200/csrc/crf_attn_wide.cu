// Window-attention core for WIDE heads: head_dim 64 and 128 (BASELINE.json configs[2] sweeps heads 4-32 at embed
// 64-512, i.e. head_dim up to 128; the four decoder scales of the model all have head_dim 32 and run on
// crf_attn_async.cu).
//
// STATUS: written after the Python-side GPU budget of round 1 was spent; verified on a B200 through the C ABI by the
// Python-free harness tools/hwcheck.cu (profiles/r01_hwcheck.txt: forward o / lse and backward dq / dk / dv / d_table /
// d_bias against a double-precision C++ reference, head_dim 64 and 128, padded + shifted, one and two heads, several
// CTAs per head: rel-L2 2.3e-3 / 2.4e-3 / 1.7e-3, the same figures as the head_dim-32 kernels on the same inputs).
// The pytest cases that drive it through Python (`*_wide*`) have not run yet and sit in tests/test_zz_gpu_unverified.py.
//
// Same mathematics and index maps as crf_attn_async.cu (newcrf_layers.py:121-146, :212-249, :332-350): pad, roll,
// partition, bias gather, shift mask, softmax, P V, reverse, un-roll and crop never exist in HBM.  A head of width
// hd = 32 * NS is processed as NS 32-wide SLICES, every slice tile having exactly the shape, swizzle and descriptors
// of the head_dim-32 kernels:
//   S   = sum_s Q_s [K_A;K_B]_s^T                   (2 NS accumulating K=16 MMAs into the same 128 x 128 accumulator)
//   O_s = P V_s                                     (own 64 TMEM columns per slice: window A | window B)
//   dP  = sum_s dO_s V_s^T,  dV_s = Pbd^T dO_s,  dK_s = dSbd^T Q_s,  dQ_s = dSbd [K_A;K_B]_s
// Structure: the synchronous single-buffer form (one thread per tile row, one MMA-issuing thread, __syncthreads
// between the phases of a window pair) -- the first generation of the head_dim-32 kernels, which was verified on
// B200 before the pipelined generations replaced it; chosen here because every barrier is a __syncthreads or one of
// two mbarriers, so the protocol cannot deadlock.  Throughput is not tuned (one thread per 64-byte row is L1TEX-tag
// bound, no overlap between gather, MMA and softmax of different pairs).
#include <stdlib.h>

#include "crf_attn_common.cuh"

namespace crf {

namespace {

constexpr int kWideThreads = 160;  // warps 0-3: one thread per tile row; warp 4: MMA issuer / TMEM owner
constexpr int kTile = 8192;        // one 128-row x 64-byte SW64 slice tile

// Token index of tile row r of a window pair: >= 0 real token, -1 zero-pad token, -2 dead row.
template <int WS>
__device__ __forceinline__ int row_token(const AttnParams& P, int pair, int r, int& window_global, int& pos) {
  const int half = r >> 6;
  pos = r & 63;
  window_global = 2 * pair + half;
  if (pos >= WS * WS || window_global >= P.total_windows) return -2;
  const int b = window_global / P.gm.nW;
  const int win = window_global - b * P.gm.nW;
  const int src = P.gm.source(win, pos);
  return src < 0 ? -1 : b * P.gm.H * P.gm.W + src;
}

// copy one 64-byte slice (32 bf16) of a token row into row r of a SW64 tile
__device__ __forceinline__ void gather_row64(uint32_t tile, int r, const __nv_bfloat16* src) {
#pragma unroll
  for (int c = 0; c < 4; ++c) cp_async16(tile + sw64_offset(r, c), src + 8 * c);
}
__device__ __forceinline__ void zero_row64(uint8_t* tile_gen, int r) {
#pragma unroll
  for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(tile_gen + sw64_offset(r, c)) = make_uint4(0, 0, 0, 0);
}
__device__ __forceinline__ void bias_row64(uint8_t* tile_gen, int r, const float* bias32) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(bias32 + 8 * c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(bias32 + 8 * c + 4));
    *reinterpret_cast<uint4*>(tile_gen + sw64_offset(r, c)) =
        make_uint4(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w), pack_bf16(b.x, b.y), pack_bf16(b.z, b.w));
  }
}

template <int NS, int WS>
struct WideFwd {
  static constexpr int kQ = 0, kK = NS * kTile, kV = 2 * NS * kTile, kP = 3 * NS * kTile;  // P: 128 x 128 B SW128
  static constexpr int kMisc = kP + 16384;                                                  // tbl | rid | bars | tmem ptr
  static constexpr int kTbl = rpb_table_padded(WS);                                         // 176 floats at WS = 7
  static constexpr int kTmemCols = NS == 2 ? 256 : 512;  // S [0,128) + O_s [128 + 64 s, 128 + 64 s + 64)
  // head_dim 64: pad the request to 80 KB so that at most two CTAs (2 x 256 TMEM columns) share an SM
  static constexpr int kSmem = (kMisc + kTbl * 4 + 128 + 32 + 1024) < 81920 ? 81920 : (kMisc + kTbl * 4 + 128 + 32 + 1024);
};

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int NS, int WS>
__global__ void __launch_bounds__(kWideThreads)
attn_fwd_wide_kernel(const AttnParams P) {
  using L = WideFwd<NS, WS>;
  constexpr int kNTok = WS * WS;
  constexpr int HD = 32 * NS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t Qs = base + L::kQ, Ks = base + L::kK, Vs = base + L::kV, Ps = base + L::kP;
  uint8_t* Ps_gen = gen + L::kP;
  float* tbl = reinterpret_cast<float*>(gen + L::kMisc);  // L::kTbl floats
  uint8_t* rid = gen + L::kMisc + L::kTbl * 4;                // 128 bytes
  const uint32_t bar_s = base + L::kMisc + L::kTbl * 4 + 128;
  const uint32_t bar_o = bar_s + 8;
  const uint32_t tmem_ptr_addr = bar_s + 16;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen + L::kMisc + L::kTbl * 4 + 128 + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const int C = P.C;

  if (warp == 4) {
    if (lane == 0) {
      mbar_init(bar_s, 1);
      mbar_init(bar_o, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_ptr_addr, L::kTmemCols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < rpb_table_size(WS); i += kWideThreads) tbl[i] = __ldg(P.table + i * P.nH + h);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_gen;

  const uint32_t idesc_s = make_idesc(1u, 0u, 0u, 128, 128);
  const uint32_t idesc_o = make_idesc(1u, 0u, 1u, 128, 32);

  int it = 0;
  for (int pair = blockIdx.x; pair < P.npairs; pair += gridDim.x, ++it) {
    int tok = -2, wg = 0, pos = 0;
    const int r = threadIdx.x;
    // ---- phase 0: gather the NS slices of this head's Q, K, V rows ----
    if (warp < 4) {
      tok = row_token<WS>(P, pair, r, wg, pos);
      if (tok >= 0) {
        const __nv_bfloat16* qrow = P.qk + static_cast<int64_t>(tok) * 2 * C + h * HD;
        const __nv_bfloat16* vrow = P.vb + static_cast<int64_t>(tok) * C + h * HD;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          gather_row64(Qs + s * kTile, r, qrow + 32 * s);
          gather_row64(Ks + s * kTile, r, qrow + C + 32 * s);
          gather_row64(Vs + s * kTile, r, vrow + 32 * s);
        }
      } else {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          zero_row64(gen + L::kQ + s * kTile, r);
          zero_row64(gen + L::kV + s * kTile, r);
          // zero-padded token: k = bias (LayerNorm'd zero row through qk), v = 0 (newcrf_layers.py:215-217)
          if (tok == -1) bias_row64(gen + L::kK + s * kTile, r, P.qk_bias + C + h * HD + 32 * s);
          else zero_row64(gen + L::kK + s * kTile, r);
        }
      }
      int region = 0;
      if (tok != -2 && P.gm.shift > 0) {
        const int b = wg / P.gm.nW;
        region = P.gm.region(wg - b * P.gm.nW, pos);
      }
      rid[r] = static_cast<uint8_t>(region);
      cp_async_commit();
      cp_async_wait_all();
      fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    // ---- phase 1: S = sum over slices of Q_s K_s^T ----
    if (warp == 4 && lane == 0) {
      tc_fence_after();
#pragma unroll
      for (int s = 0; s < NS; ++s) {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma_bf16(tmem, make_smem_desc(Qs + s * kTile + ks * 32, 16, 512, kSwizzle64),
                    make_smem_desc(Ks + s * kTile + ks * 32, 16, 512, kSwizzle64), idesc_s, (s > 0 || ks > 0) ? 1u : 0u);
      }
      umma_commit(bar_s);
    }
    // ---- phase 2: softmax, one thread per row ----
    if (warp < 4) {
      mbar_wait(bar_s, it & 1);
      tc_fence_after();
      const int half = r >> 6;
      const uint32_t taddr = tmem + (static_cast<uint32_t>(warp * 32) << 16) + half * 64;
      uint32_t s0[32], s1[32];
      tmem_ld32(taddr, s0);
      tmem_ld32(taddr + 32, s1);
      tmem_ld_wait();
      float p[64];
      if (tok != -2) {
        const int bi = rpb_base<WS>(pos);
        const uint8_t* rrow = rid + half * 64;
        const int my_region = rrow[pos];
        const bool masked = P.gm.shift > 0 && !P.ext_replaces;
        const float* xmask = P.ext_mask != nullptr
                                 ? P.ext_mask + (static_cast<int64_t>(wg % P.ext_mask_nw) * kNTok + pos) * kNTok
                                 : nullptr;
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          float s = __uint_as_float(j < 32 ? s0[j & 31] : s1[j & 31]) + tbl[bi - rpb_col<WS>(j)];
          if (masked && rrow[j] != my_region) s += -100.0f;
          if (xmask != nullptr) s += __ldg(xmask + j);
          p[j] = s;
          mx = fmaxf(mx, s);
        }
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          p[j] = __expf(p[j] - mx);
          sum += p[j];
        }
        const float inv = 1.0f / sum;
#pragma unroll
        for (int j = 0; j < kNTok; ++j) p[j] *= inv;
#pragma unroll
        for (int j = kNTok; j < 64; ++j) p[j] = 0.f;
        if (P.lse != nullptr) P.lse[(static_cast<int64_t>(wg) * P.nH + h) * 64 + pos] = mx + __logf(sum);
      } else {
#pragma unroll
        for (int j = 0; j < 64; ++j) p[j] = 0.f;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c)
        *reinterpret_cast<uint4*>(Ps_gen + sw128_offset(r, c)) =
            make_uint4(pack_bf16(p[8 * c], p[8 * c + 1]), pack_bf16(p[8 * c + 2], p[8 * c + 3]),
                       pack_bf16(p[8 * c + 4], p[8 * c + 5]), pack_bf16(p[8 * c + 6], p[8 * c + 7]));
      fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    // ---- phase 3: O_s = P V_s (window A -> cols [0,32), window B -> cols [32,64) of the slice's 64 columns) ----
    if (warp == 4 && lane == 0) {
      tc_fence_after();
#pragma unroll
      for (int s = 0; s < NS; ++s) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_bf16(tmem + 128 + s * 64 + half * 32, make_smem_desc(Ps + ks * 32, 16, 1024, kSwizzle128),
                      make_smem_desc(Vs + s * kTile + half * 4096 + ks * 1024, 512, 512, kSwizzle64), idesc_o,
                      ks > 0 ? 1u : 0u);
        }
      }
      umma_commit(bar_o);
    }
    // ---- phase 4: store O rows in token order (window_reverse + un-roll + crop) ----
    if (warp < 4) {
      mbar_wait(bar_o, it & 1);
      tc_fence_after();
      const int half = r >> 6;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        uint32_t o[32];
        tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16) + 128 + s * 64 + half * 32, o);
        tmem_ld_wait();
        if (tok >= 0) {
          uint4* dst = reinterpret_cast<uint4*>(P.o + static_cast<int64_t>(tok) * C + h * HD + 32 * s);
#pragma unroll
          for (int c = 0; c < 4; ++c)
            dst[c] = make_uint4(pack_bf16(__uint_as_float(o[8 * c]), __uint_as_float(o[8 * c + 1])),
                                pack_bf16(__uint_as_float(o[8 * c + 2]), __uint_as_float(o[8 * c + 3])),
                                pack_bf16(__uint_as_float(o[8 * c + 4]), __uint_as_float(o[8 * c + 5])),
                                pack_bf16(__uint_as_float(o[8 * c + 6]), __uint_as_float(o[8 * c + 7])));
        }
      }
    }
    // the next iteration's first __syncthreads (preceded by tcgen05.fence::before_thread_sync) orders these TMEM
    // reads and the smem reads of the finished MMAs before they are overwritten.
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem, L::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
template <int NS, int WS>
struct WideBwd {
  // Q, K, V, dO: NS slice tiles each; Pbd, dSbd: 2 x 16 KB each (two SW128 column chunks of 128 rows)
  static constexpr int kQ = 0, kK = NS * kTile, kV = 2 * NS * kTile, kG = 3 * NS * kTile;
  static constexpr int kPb = 4 * NS * kTile, kDb = kPb + 32768;
  static constexpr int kMisc = kDb + 32768;
  static constexpr int kTbl = rpb_table_padded(WS);      // 176 floats at WS = 7
  static constexpr int kTmemCols = NS == 2 ? 256 : 512;  // S [0,128), dP [128,256); then dV_s | dK_s | dQ_s at 96 s
  static constexpr int kSmem = kMisc + kTbl * 4 + 128 + 32 + 1024;
  static_assert(kSmem <= 232448, "shared-memory plan exceeds 227 KB");
  static_assert(96 * NS <= kTmemCols, "second-stage results do not fit the TMEM allocation");
};

template <int NS, int WS>
__global__ void __launch_bounds__(kWideThreads)
attn_bwd_wide_kernel(const AttnParams P) {
  using L = WideBwd<NS, WS>;
  constexpr int kNTok = WS * WS;
  constexpr int HD = 32 * NS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t Qs = base + L::kQ, Ks = base + L::kK, Vs = base + L::kV, Gs = base + L::kG;
  const uint32_t Pb = base + L::kPb, Db = base + L::kDb;
  float* tbl = reinterpret_cast<float*>(gen + L::kMisc);  // L::kTbl floats
  uint8_t* rid = gen + L::kMisc + L::kTbl * 4;                // 128 bytes
  const uint32_t bar_s = base + L::kMisc + L::kTbl * 4 + 128;
  const uint32_t bar_o = bar_s + 8;
  const uint32_t tmem_ptr_addr = bar_s + 16;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen + L::kMisc + L::kTbl * 4 + 128 + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const int C = P.C;

  if (warp == 4) {
    if (lane == 0) {
      mbar_init(bar_s, 1);
      mbar_init(bar_o, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_ptr_addr, L::kTmemCols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < rpb_table_size(WS); i += kWideThreads) tbl[i] = __ldg(P.table + i * P.nH + h);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_gen;

  const uint32_t idesc_s = make_idesc(1u, 0u, 0u, 128, 128);  // S, dP : K-major x K-major
  const uint32_t idesc_t = make_idesc(1u, 1u, 1u, 128, 32);   // dV, dK: MN-major x MN-major
  const uint32_t idesc_q = make_idesc(1u, 0u, 1u, 128, 32);   // dQ    : K-major x MN-major

  float dtab[kNTok];  // sum over all my pairs of dS[my row][j]
#pragma unroll
  for (int j = 0; j < kNTok; ++j) dtab[j] = 0.f;
  const int my_pos = threadIdx.x & 63;

  int it = 0;
  for (int pair = blockIdx.x; pair < P.npairs; pair += gridDim.x, ++it) {
    int tok = -2, wg = 0, pos = 0;
    const int r = threadIdx.x;
    if (warp < 4) {
      tok = row_token<WS>(P, pair, r, wg, pos);
      if (tok >= 0) {
        const __nv_bfloat16* qrow = P.qk + static_cast<int64_t>(tok) * 2 * C + h * HD;
        const __nv_bfloat16* vrow = P.vb + static_cast<int64_t>(tok) * C + h * HD;
        const __nv_bfloat16* grow = P.dout + static_cast<int64_t>(tok) * C + h * HD;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          gather_row64(Qs + s * kTile, r, qrow + 32 * s);
          gather_row64(Ks + s * kTile, r, qrow + C + 32 * s);
          gather_row64(Vs + s * kTile, r, vrow + 32 * s);
          gather_row64(Gs + s * kTile, r, grow + 32 * s);
        }
      } else {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          zero_row64(gen + L::kQ + s * kTile, r);
          zero_row64(gen + L::kV + s * kTile, r);
          zero_row64(gen + L::kG + s * kTile, r);
          if (tok == -1) bias_row64(gen + L::kK + s * kTile, r, P.qk_bias + C + h * HD + 32 * s);
          else zero_row64(gen + L::kK + s * kTile, r);
        }
      }
      int region = 0;
      if (tok != -2 && P.gm.shift > 0) {
        const int b = wg / P.gm.nW;
        region = P.gm.region(wg - b * P.gm.nW, pos);
      }
      rid[r] = static_cast<uint8_t>(region);
      cp_async_commit();
      cp_async_wait_all();
      fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    // ---- S = sum_s Q_s K_s^T -> cols [0,128);  dP = sum_s dO_s V_s^T -> cols [128,256) ----
    if (warp == 4 && lane == 0) {
      tc_fence_after();
#pragma unroll
      for (int s = 0; s < NS; ++s) {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma_bf16(tmem, make_smem_desc(Qs + s * kTile + ks * 32, 16, 512, kSwizzle64),
                    make_smem_desc(Ks + s * kTile + ks * 32, 16, 512, kSwizzle64), idesc_s, (s > 0 || ks > 0) ? 1u : 0u);
      }
#pragma unroll
      for (int s = 0; s < NS; ++s) {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma_bf16(tmem + 128, make_smem_desc(Gs + s * kTile + ks * 32, 16, 512, kSwizzle64),
                    make_smem_desc(Vs + s * kTile + ks * 32, 16, 512, kSwizzle64), idesc_s, (s > 0 || ks > 0) ? 1u : 0u);
      }
      umma_commit(bar_s);
    }
    // ---- P, dS per row; block-diagonal bf16 tiles ----
    if (warp < 4) {
      mbar_wait(bar_s, it & 1);
      tc_fence_after();
      const int half = r >> 6;
      const uint32_t taddr = tmem + (static_cast<uint32_t>(warp * 32) << 16) + half * 64;
      float p[64], ds[64];
      {
        uint32_t s0[32], s1[32];
        tmem_ld32(taddr, s0);
        tmem_ld32(taddr + 32, s1);
        tmem_ld_wait();
        if (tok >= 0) {
          const float lse = __ldg(P.lse + (static_cast<int64_t>(wg) * P.nH + h) * 64 + pos);
          const int bi = rpb_base<WS>(pos);
          const uint8_t* rrow = rid + half * 64;
          const int my_region = rrow[pos];
          const bool masked = P.gm.shift > 0 && !P.ext_replaces;
          const float* xmask = P.ext_mask != nullptr
                                   ? P.ext_mask + (static_cast<int64_t>(wg % P.ext_mask_nw) * kNTok + pos) * kNTok
                                   : nullptr;
#pragma unroll
          for (int j = 0; j < kNTok; ++j) {
            float s = __uint_as_float(j < 32 ? s0[j & 31] : s1[j & 31]) + tbl[bi - rpb_col<WS>(j)];
            if (masked && rrow[j] != my_region) s += -100.0f;
            if (xmask != nullptr) s += __ldg(xmask + j);
            p[j] = __expf(s - lse);
          }
        } else {
#pragma unroll
          for (int j = 0; j < kNTok; ++j) p[j] = 0.f;
        }
#pragma unroll
        for (int j = kNTok; j < 64; ++j) p[j] = 0.f;
      }
      {
        uint32_t g0[32], g1[32];
        tmem_ld32(taddr + 128, g0);
        tmem_ld32(taddr + 128 + 32, g1);
        tmem_ld_wait();
        float dsum = 0.f;
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          ds[j] = __uint_as_float(j < 32 ? g0[j & 31] : g1[j & 31]);
          dsum += p[j] * ds[j];
        }
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          ds[j] = p[j] * (ds[j] - dsum);
          dtab[j] += ds[j];
        }
#pragma unroll
        for (int j = kNTok; j < 64; ++j) ds[j] = 0.f;
      }
      // row r of the 128 x 128 block-diagonal tiles: own window's 64 columns carry data, the other 64 are zero
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint32_t own = static_cast<uint32_t>(half) * 16384u + sw128_offset(r, c);
        const uint32_t oth = static_cast<uint32_t>(half ^ 1) * 16384u + sw128_offset(r, c);
        *reinterpret_cast<uint4*>(gen + L::kPb + own) =
            make_uint4(pack_bf16(p[8 * c], p[8 * c + 1]), pack_bf16(p[8 * c + 2], p[8 * c + 3]),
                       pack_bf16(p[8 * c + 4], p[8 * c + 5]), pack_bf16(p[8 * c + 6], p[8 * c + 7]));
        *reinterpret_cast<uint4*>(gen + L::kPb + oth) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(gen + L::kDb + own) =
            make_uint4(pack_bf16(ds[8 * c], ds[8 * c + 1]), pack_bf16(ds[8 * c + 2], ds[8 * c + 3]),
                       pack_bf16(ds[8 * c + 4], ds[8 * c + 5]), pack_bf16(ds[8 * c + 6], ds[8 * c + 7]));
        *reinterpret_cast<uint4*>(gen + L::kDb + oth) = make_uint4(0, 0, 0, 0);
      }
      fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    // ---- per slice s: dV_s -> cols [96 s, +32), dK_s -> [96 s + 32, +32), dQ_s -> [96 s + 64, +32) ----
    // (S and dP have been consumed by every row thread before the barrier above, so their columns are reused)
    if (warp == 4 && lane == 0) {
      tc_fence_after();
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const uint32_t t0 = tmem + 96 * s;
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)  // K = 128 query rows, 16 per step
          umma_bf16(t0, make_smem_desc(Pb + ks * 2048, 16384, 1024, kSwizzle128),
                    make_smem_desc(Gs + s * kTile + ks * 1024, 512, 512, kSwizzle64), idesc_t, ks > 0 ? 1u : 0u);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
          umma_bf16(t0 + 32, make_smem_desc(Db + ks * 2048, 16384, 1024, kSwizzle128),
                    make_smem_desc(Qs + s * kTile + ks * 1024, 512, 512, kSwizzle64), idesc_t, ks > 0 ? 1u : 0u);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)  // K = 128 stacked keys: column chunk ks / 4, 32 B per step inside it
          umma_bf16(t0 + 64, make_smem_desc(Db + (ks >> 2) * 16384 + (ks & 3) * 32, 16, 1024, kSwizzle128),
                    make_smem_desc(Ks + s * kTile + ks * 1024, 512, 512, kSwizzle64), idesc_q, ks > 0 ? 1u : 0u);
      }
      umma_commit(bar_o);
    }
    if (warp < 4) {
      mbar_wait(bar_o, it & 1);
      tc_fence_after();
      const uint32_t trow = tmem + (static_cast<uint32_t>(warp * 32) << 16);
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        uint32_t a[32];
        // dV (row = key)
        tmem_ld32(trow + 96 * s, a);
        tmem_ld_wait();
        if (tok >= 0) {
          float4* dst = reinterpret_cast<float4*>(P.dv + static_cast<int64_t>(tok) * C + h * HD + 32 * s);
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            float4 v = make_float4(__uint_as_float(a[4 * c]), __uint_as_float(a[4 * c + 1]),
                                   __uint_as_float(a[4 * c + 2]), __uint_as_float(a[4 * c + 3]));
            if (P.dv_acc) {  // a token belongs to exactly one window of a block: no other thread touches this row
              const float4 o = dst[c];
              v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
            }
            dst[c] = v;
          }
        }
        // dK (row = key)
        tmem_ld32(trow + 96 * s + 32, a);
        tmem_ld_wait();
        if (tok >= 0) {
          uint4* dst = reinterpret_cast<uint4*>(P.dqk + static_cast<int64_t>(tok) * 2 * C + C + h * HD + 32 * s);
#pragma unroll
          for (int c = 0; c < 4; ++c)
            dst[c] = make_uint4(pack_bf16(__uint_as_float(a[8 * c]), __uint_as_float(a[8 * c + 1])),
                                pack_bf16(__uint_as_float(a[8 * c + 2]), __uint_as_float(a[8 * c + 3])),
                                pack_bf16(__uint_as_float(a[8 * c + 4]), __uint_as_float(a[8 * c + 5])),
                                pack_bf16(__uint_as_float(a[8 * c + 6]), __uint_as_float(a[8 * c + 7])));
        } else if (tok == -1) {  // zero-padded key: k == bias, so its gradient goes to the k half of qk.bias
#pragma unroll
          for (int j = 0; j < 32; ++j) atomicAdd(P.d_qk_bias + C + h * HD + 32 * s + j, __uint_as_float(a[j]));
        }
        // dQ (row = query); d(xW+b) = dq * scale because q was stored pre-scaled
        tmem_ld32(trow + 96 * s + 64, a);
        tmem_ld_wait();
        if (tok >= 0) {
          uint4* dst = reinterpret_cast<uint4*>(P.dqk + static_cast<int64_t>(tok) * 2 * C + h * HD + 32 * s);
          const float sc = P.scale;
#pragma unroll
          for (int c = 0; c < 4; ++c)
            dst[c] = make_uint4(pack_bf16(sc * __uint_as_float(a[8 * c]), sc * __uint_as_float(a[8 * c + 1])),
                                pack_bf16(sc * __uint_as_float(a[8 * c + 2]), sc * __uint_as_float(a[8 * c + 3])),
                                pack_bf16(sc * __uint_as_float(a[8 * c + 4]), sc * __uint_as_float(a[8 * c + 5])),
                                pack_bf16(sc * __uint_as_float(a[8 * c + 6]), sc * __uint_as_float(a[8 * c + 7])));
        }
      }
    }
  }

  // flush the relative-position-bias gradient: dTable[idx(i,j), h] += sum_windows dS[i][j]
  __syncthreads();
  float* dt = tbl;  // reuse as the CTA-level accumulator
  for (int i = threadIdx.x; i < L::kTbl; i += kWideThreads) dt[i] = 0.f;
  __syncthreads();
  if (warp < 4 && my_pos < kNTok) {
    const int bi = rpb_base<WS>(my_pos);
#pragma unroll
    for (int j = 0; j < kNTok; ++j) atomicAdd(dt + bi - rpb_col<WS>(j), dtab[j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < rpb_table_size(WS); i += kWideThreads) atomicAdd(P.d_table + i * P.nH + h, dt[i]);

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem, L::kTmemCols);
  }
}

int wide_grid_x(const AttnParams& P, const crf_block_desc& d, int ctas_per_sm) {
  int gx = (num_sms(d.device) * ctas_per_sm + P.nH - 1) / P.nH;
  if (gx > P.npairs) gx = P.npairs;
  return gx < 1 ? 1 : gx;
}

template <int NS, int WS>
int launch_fwd(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  auto kern = attn_fwd_wide_kernel<NS, WS>;
  constexpr int smem = WideFwd<NS, WS>::kSmem;
  const double N = WS * WS;
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const double TC = static_cast<double>(d.B) * d.H * d.W * d.C;
  KernelTimer tm(st, 4.0 * N * N * d.C * P.total_windows, 8.0 * TC, "attn_fwd_wide_B%d_%dx%d_C%d_h%d_s%d", d.B, d.H,
                 d.W, d.C, P.nH, d.shift);
  kern<<<dim3(wide_grid_x(P, d, NS == 2 ? 2 : 1), P.nH), kWideThreads, smem, st>>>(P);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

template <int NS, int WS>
int launch_bwd(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  auto kern = attn_bwd_wide_kernel<NS, WS>;
  constexpr int smem = WideBwd<NS, WS>::kSmem;
  const double N = WS * WS;
  CRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const double TC = static_cast<double>(d.B) * d.H * d.W * d.C;
  KernelTimer tm(st, 10.0 * N * N * d.C * P.total_windows, 16.0 * TC, "attn_bwd_wide_B%d_%dx%d_C%d_h%d_s%d", d.B,
                 d.H, d.W, d.C, P.nH, d.shift);
  kern<<<dim3(wide_grid_x(P, d, 1), P.nH), kWideThreads, smem, st>>>(P);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace

int launch_attn_fwd_wide(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  if (P.hd != 64 && P.hd != 128) return set_error("wide attention core: head_dim must be 64 or 128 (got %d)", P.hd);
  const int rc = with_window(P.gm.ws, [&](auto w) {
    return P.hd == 64 ? launch_fwd<2, decltype(w)::value>(P, d, st) : launch_fwd<4, decltype(w)::value>(P, d, st);
  });
  return rc >= 0 ? rc : set_error("wide attention core: no kernel for window %d", P.gm.ws);
}

int launch_attn_bwd_wide(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  if (P.hd != 64 && P.hd != 128) return set_error("wide attention core: head_dim must be 64 or 128 (got %d)", P.hd);
  const int rc = with_window(P.gm.ws, [&](auto w) {
    return P.hd == 64 ? launch_bwd<2, decltype(w)::value>(P, d, st) : launch_bwd<4, decltype(w)::value>(P, d, st);
  });
  return rc >= 0 ? rc : set_error("wide attention core: no kernel for window %d", P.gm.ws);
}

}  // namespace crf
