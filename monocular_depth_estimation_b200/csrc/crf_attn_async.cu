// Window-attention core of the CRF block on tcgen05, forward and backward.
//
// Replaces, without materialising any of them in HBM: F.pad, torch.roll, window_partition of x and v, the
// relative-position-bias gather, the shifted-window mask, softmax, attn @ v, window_reverse, the reverse roll and
// the crop (newcrf_layers.py:121-146, :212-249, :332-350).
//
// Work decomposition: a CTA owns one head and loops over PAIRS of windows.  The two N-token windows of a pair
// (N = ws^2 <= 64; the kernels are instantiated per window size 2..8, and the prose below uses ws = 7, N = 49) are
// stacked into one 128-row UMMA tile (rows 0..N-1 = window A, 64..64+N-1 = window B, the rest zero):
//   S  [128 x 128] = bias + Q[128 x hd] * [K_A ; K_B]^T     -- row r only uses the 64 columns of its own window
//   O  [128 x 2hd] = P~[128 x 64] * [V_A | V_B]             -- row r reads the hd columns of its window
// Token rows are gathered straight from the token-major q/k/v tensors with the closed-form pad+roll index map
// (cp.async 16-byte copies into the swizzled UMMA layout); zero-padded tokens get k = bias, v = 0 exactly as the
// reference's pad-after-LayerNorm produces.  Softmax runs one thread per accumulator row (TMEM lane), fp32.
// Backward recomputes S and P from q, k and the saved row log-sum-exp:
//   dP = dO * [V_A;V_B]^T,  dS = P o (dP - rowsum(P o dP)),  per window w: dV_w = P_w^T dO_w, dK_w = dS_w^T Q_w,
//   dQ_w = dS_w K_w;  the relative-position-bias gradient is accumulated in registers across all pairs a CTA
//   processes (each thread owns one query row) and flushed once per CTA.
//
// This is the third generation of these kernels (single-buffer -> warp-specialised double-buffered -> this one),
// restructured after per-phase cycle counts (CRF_ATTN_PROF=1) showed where a window pair's time goes.  Nothing on the
// per-pair chain
//   gather -> S (/dP) MMA -> softmax (/dS) math -> second-stage MMAs -> stores
// waits for something it does not depend on, and the issue-bound softmax warps do less per element:
//
//   * loaders never block on their own gathers: each loader thread hands its 64-byte head slices to the LSU with
//     cp.async and lets the hardware arrive on the slot's `full` mbarrier (cp.async.mbarrier.arrive.noinc) when they
//     land, so up to four window pairs of gathers are in flight per SM;
//   * two MMA-issuing warps instead of one: warp 12 issues the first stage (S, dP) of every pair, warp 13 the second
//     stage (P V / dV, dK, dQ), each a plain in-order loop -- a single issuing thread spent 60 % of the kernel's
//     duration issuing and was the bottleneck;
//   * the relative-position bias is pre-loaded into the S accumulator: after a compute thread has drained its TMEM
//     lane it writes its row's 49 bias values (fp32, exact) there with tcgen05.st, and the next S = Q K^T accumulates
//     on top -- 16 LDS.128 + 2 tcgen05.st per row and pair, off the critical path, replace 49 LDS + 49 FADD on it;
//   * softmax numerator only: P~ = 2^((S - max) log2e) goes to the tensor core unnormalised and the O row is divided
//     by the row sum when it comes back; max / sum / dsum are four-way interleaved chains;
//   * compute threads derive their row's token, window and shifted-window mask themselves (closed form, a 49-bit
//     mask per row that is non-zero only for windows on the roll seam), so no metadata travels through shared memory;
//   * backward: P and dS are stored as COMPACT 128 x 64 tiles (row = query, 64 keys of its own window) and the
//     second stage runs per window as M=64 tcgen05 MMAs (dV = P_w^T dO_w, dK = dS_w^T Q_w, dQ = dS_w K_w; the two
//     windows of a pair land on the two 16-lane halves of every TMEM sub-partition), which halves the P / dS tiles
//     and gives the backward two input slots per lane like the forward; the row log-sum-exp is fetched before the
//     wait on S, and dv is accumulated with fire-and-forget red.global.add.v4.f32.
//
// Roles (512 threads, 1 CTA / SM, CTA = one head x a strided set of window pairs, two "lanes" g = pair parity):
//   warps 0-3 / 4-7  compute group of lane 0 / 1 (thread = tile row = TMEM lane)
//   warps 8-11       loaders (four threads per tile row, see loader_loop)
//   warp 12 / 13     first- / second-stage MMA issuer (one thread each); warp 12 owns the TMEM allocation
// mbarriers: full[g][slot] (256 loader arrivals: one per thread + one made by the LSU for its cp.asyncs) -> s_done[g] (commit) -> p_ready[g] (128)
// -> o_done[g] (commit) -> t_free[g] (128: TMEM drained and bias pre-loaded);  in_free[g][slot] (commit).
#include "crf_attn_common.cuh"

namespace crf {

namespace {

constexpr int kThreads = 512;
constexpr int HD = 32;
constexpr float kLog2e = 1.4426950408889634f;

constexpr uint32_t kSlot = 32768;                       // Q | K | V | (dO): 4 x 8 KB
constexpr uint32_t kFwdTiles = 4 * kSlot;               // P tiles: 2 lanes x 16 KB
constexpr uint32_t kFwdMisc = kFwdTiles + 2 * 16384;
constexpr uint32_t kBwdTiles = 4 * kSlot;               // P | dS tiles: 2 lanes x (16 + 16) KB
constexpr uint32_t kBwdMisc = kBwdTiles + 2 * 32768;
constexpr int kBiasStride = 68;                         // floats per bias row (272 B: conflict-free LDS.128 per quarter warp)
constexpr uint32_t kScratchWarp = 32 * 80;

// The misc region behind the tiles, for window size WS (N = WS^2 tokens per window):
//   tbl[rpb_table_padded(WS)] f32 | bias rows [N][68] f32 | 8 compute warps x (32 rows x 80 B) scratch | 16 mbarriers |
//   TMEM address.  At WS = 7: tbl[176], bias rows [49][68].
// The WS = 8 backward keeps no bias rows: its 196 KB of tiles plus 64 rows of 272 B would exceed the 227 KB a CTA may
// use, so it pre-loads the bias straight from the table (64 scalar LDS per row and pair instead of 16 LDS.128).
template <int WS, bool BWD>
struct Misc {
  static constexpr int kN = WS * WS;
  static constexpr bool kBiasRows = !(BWD && WS == 8);
  static constexpr int kTblFloats = rpb_table_padded(WS);
  static constexpr uint32_t kTbl = 0;
  static constexpr uint32_t kBias = kTblFloats * 4;
  static constexpr uint32_t kScratch = kBias + (kBiasRows ? kN * kBiasStride * 4 : 0);
  static constexpr uint32_t kBar = kScratch + 8 * kScratchWarp;
  static constexpr uint32_t kTmem = kBar + 16 * 8;
  static constexpr uint32_t kBytes = kTmem + 16;
  static_assert(kBias % 16 == 0 && kBar % 8 == 0, "bias-row / mbarrier alignment");
  static_assert(WS >= kMinWindow && WS <= kMaxWindow, "a window's N = WS^2 tokens must fit 64 tile rows");
};

struct Bars {
  uint32_t base;
  __device__ uint32_t full(int g, int slot) const { return base + 8u * (2 * g + slot); }
  __device__ uint32_t s_done(int g) const { return base + 8u * (4 + g); }
  __device__ uint32_t p_ready(int g) const { return base + 8u * (6 + g); }
  __device__ uint32_t o_done(int g) const { return base + 8u * (8 + g); }
  __device__ uint32_t t_free(int g) const { return base + 8u * (10 + g); }
  __device__ uint32_t in_free(int g, int slot) const { return base + 8u * (12 + 2 * g + slot); }
};

__device__ __forceinline__ void init_bars(const Bars& b) {
  for (int g = 0; g < 2; ++g) {
    for (int slot = 0; slot < 2; ++slot) {
      mbar_init(b.full(g, slot), 256);  // every loader thread: one arrive of its own + one made by its cp.asyncs
      mbar_init(b.in_free(g, slot), 1);
    }
    mbar_init(b.s_done(g), 1);
    mbar_init(b.p_ready(g), 128);
    mbar_init(b.o_done(g), 1);
    mbar_init(b.t_free(g), 128);
  }
  fence_mbar_init();
}

// Exact floor(a / d) for 0 <= a < 2^22 from a float reciprocal (the two integer divisions per row were a visible
// part of the XU-pipe load: 52 % busy in the second-generation kernels).
__device__ __forceinline__ int fast_div(int a, int d, float rd) {
  int q = __float2int_rz((static_cast<float>(a) + 0.5f) * rd);
  const int r = a - q * d;
  if (r < 0) --q;
  else if (r >= d) ++q;
  return q;
}
// global window -> (image, window row, window column)
struct WinPos {
  int b, wh, ww;
  bool hsplit, wsplit;  // the window straddles the roll seam in h / w (shifted-window mask separates positions)
};
template <int WS>
__device__ __forceinline__ WinPos window_pos(const AttnParams& P, int wg) {
  WinPos w;
  w.b = fast_div(wg, P.gm.nW, P.rcp_nW);
  const int win = wg - w.b * P.gm.nW;
  w.wh = fast_div(win, P.gm.nWw, P.rcp_nWw);
  w.ww = win - w.wh * P.gm.nWw;
  w.hsplit = P.gm.shift > 0 && (w.wh + 1) * WS == P.gm.Hp;
  w.wsplit = P.gm.shift > 0 && (w.ww + 1) == P.gm.nWw;
  return w;
}
// Closed-form geometry of tile position (pi, pj) of a window (newcrf_layers.py:212-233 folded): token index (>= 0),
// or -1 for a zero-pad position.
template <int WS>
__device__ __forceinline__ int window_token(const AttnParams& P, const WinPos& w, int pi, int pj) {
  int hh = w.wh * WS + pi + P.gm.shift, wx = w.ww * WS + pj + P.gm.shift;
  if (hh >= P.gm.Hp) hh -= P.gm.Hp;
  if (wx >= P.gm.Wp) wx -= P.gm.Wp;
  return (hh < P.gm.H && wx < P.gm.W) ? (w.b * P.gm.H + hh) * P.gm.W + wx : -1;
}

// Per-row view a compute thread needs: token (-2 dead row), global window, and the N-bit set of key positions j the
// shifted-window mask separates from this row (region(i) != region(j)  <=>  they lie on different sides of a seam).
struct RowView {
  int tok, wg;
  uint32_t m_lo, m_hi;
};
template <int WS>
__device__ __forceinline__ RowView row_view(const AttnParams& P, int pair, int half, int pos, int pi, int pj,
                                            uint64_t far_h, uint64_t far_w) {
  constexpr int kN = WS * WS;
  RowView v;
  v.wg = 2 * pair + half;
  v.tok = -2;
  v.m_lo = v.m_hi = 0u;
  if (pos < kN && v.wg < P.total_windows) {
    const WinPos w = window_pos<WS>(P, v.wg);
    v.tok = window_token<WS>(P, w, pi, pj);
    const int lo = WS - P.gm.shift;
    uint64_t m = 0;
    if (w.hsplit) m |= (pi >= lo) ? ~far_h : far_h;
    if (w.wsplit) m |= (pj >= lo) ? ~far_w : far_w;
    m &= kN < 64 ? (1ull << (kN & 63)) - 1 : ~0ull;  // (a shift by 64 would be undefined)
    if (P.ext_replaces) m = 0;
    v.m_lo = static_cast<uint32_t>(m);
    v.m_hi = static_cast<uint32_t>(m >> 32);
  }
  return v;
}
#define CRF_MASKED(v, j) ((((j) < 32 ? (v).m_lo >> ((j) & 31) : (v).m_hi >> ((j) & 31)) & 1u) != 0u)

// key positions on the far side of the seam: rows i >= WS - shift (far_h), columns j >= WS - shift (far_w)
template <int WS>
__device__ __forceinline__ void seam_sets(int shift, uint64_t& far_h, uint64_t& far_w) {
  far_h = far_w = 0;
  const int lo = WS - shift;
#pragma unroll
  for (int j = 0; j < WS * WS; ++j) {
    if (j / WS >= lo) far_h |= 1ull << j;
    if (j % WS >= lo) far_w |= 1ull << j;
  }
}

// bias rows: brow[i][j] = table[relative_position_index[i][j], h] (newcrf_layers.py:124-127), 0 for j >= N
template <int WS>
__device__ __forceinline__ void build_bias_rows(float* brow, const float* tbl) {
  constexpr int kN = WS * WS;
  for (int idx = threadIdx.x; idx < kN * 64; idx += kThreads) {
    const int i = idx >> 6, j = idx & 63;
    brow[i * kBiasStride + j] = j < kN ? tbl[rpb_base<WS>(i) - rpb_col<WS>(j)] : 0.f;
  }
}
// Write this thread's bias row into the 64 S columns of its TMEM lane (whole warp; dead rows write row 0's values,
// which nobody reads), so that the next S MMA accumulates Q K^T on top of it.
template <int WS>
__device__ __forceinline__ void preload_bias(const float* brow, int pos, uint32_t taddr) {
  const float4* src = reinterpret_cast<const float4*>(brow + (pos < WS * WS ? pos : 0) * kBiasStride);
#pragma unroll
  for (int hlf = 0; hlf < 2; ++hlf) {
    uint32_t v[32];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float4 b = src[hlf * 8 + c];
      v[4 * c] = __float_as_uint(b.x); v[4 * c + 1] = __float_as_uint(b.y);
      v[4 * c + 2] = __float_as_uint(b.z); v[4 * c + 3] = __float_as_uint(b.w);
    }
    tmem_st32(taddr + hlf * 32, v);
  }
  tmem_st_wait();
}
// The same row gathered from the table itself (the WS = 8 backward, which has no room for bias rows).  Every column
// j < N of a live row gets its bias; the columns j >= N of this N = 64 window do not exist.
template <int WS>
__device__ __forceinline__ void preload_bias_from_table(const float* tbl, int pos, uint32_t taddr) {
  constexpr int kN = WS * WS;
  const int bi = rpb_base<WS>(pos < kN ? pos : 0);
#pragma unroll
  for (int hlf = 0; hlf < 2; ++hlf) {
    uint32_t v[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      const int j = hlf * 32 + c;
      v[c] = j < kN ? __float_as_uint(tbl[bi - rpb_col<WS>(j)]) : 0u;
    }
    tmem_st32(taddr + hlf * 32, v);
  }
  tmem_st_wait();
}
template <int WS, bool BWD>
__device__ __forceinline__ void preload_row_bias(const float* brow, const float* tbl, int pos, uint32_t taddr) {
  if constexpr (Misc<WS, BWD>::kBiasRows) preload_bias<WS>(brow, pos, taddr);
  else preload_bias_from_table<WS>(tbl, pos, taddr);
}

// Loaders: FOUR threads per tile row (thread t: 16-byte chunk t & 3 of rows (t >> 2) + 32 k), so one warp-level
// cp.async covers 8 rows x 64 contiguous bytes = 8 cache lines.  With one thread per row every instruction touched 32
// lines and the L1TEX tag stage (one line per cycle) was the kernel's limiter: ~1500 (fwd) / ~4100 (bwd, with the
// equally scattered stores) tag cycles per pair against 2800 / 6100 measured cycles per pair.
template <bool BWD>
__device__ __forceinline__ void load_chunk(const AttnParams& P, int tok, int r, int c, int h, uint32_t in_s,
                                           uint8_t* in_g, bool& any_async) {
  const int C = P.C;
  const uint32_t off = sw64_offset(r, c);
  const bool live_c = 8 * c < P.hd;  // head_dim 16: chunks 2, 3 of the 32-wide tiles stay zero
  if (tok >= 0 && live_c) {
    const __nv_bfloat16* qrow = P.qk + static_cast<int64_t>(tok) * 2 * C + h * P.hd + 8 * c;
    cp_async16(in_s + off, qrow);
    cp_async16(in_s + 8192 + off, qrow + C);
    cp_async16(in_s + 16384 + off, P.vb + static_cast<int64_t>(tok) * C + h * P.hd + 8 * c);
    if (BWD) cp_async16(in_s + 24576 + off, P.dout + static_cast<int64_t>(tok) * C + h * P.hd + 8 * c);
    any_async = true;
  } else {
    const uint4 z = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<uint4*>(in_g + off) = z;
    *reinterpret_cast<uint4*>(in_g + 16384 + off) = z;
    if (BWD) *reinterpret_cast<uint4*>(in_g + 24576 + off) = z;
    uint4 kv = z;
    if (tok == -1 && live_c) {  // zero-padded token: k = bias (LayerNorm'd zero row through qk), v = 0
      const float* bk = P.qk_bias + C + h * P.hd + 8 * c;
      const float4 a = __ldg(reinterpret_cast<const float4*>(bk));
      const float4 b = __ldg(reinterpret_cast<const float4*>(bk + 4));
      kv = make_uint4(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w), pack_bf16(b.x, b.y), pack_bf16(b.z, b.w));
    }
    *reinterpret_cast<uint4*>(in_g + 8192 + off) = kv;
  }
}

template <int WS, bool BWD>
__device__ __forceinline__ void loader_loop(const AttnParams& P, const Bars& bars, uint32_t base, uint8_t* gen, int h,
                                            int niter) {
  constexpr int kN = WS * WS;
  const int t = threadIdx.x - 256;
  const int c = t & 3, rb = t >> 2;           // rows rb, rb + 32 (window A) and rb + 64, rb + 96 (window B)
  const int pi0 = rb / WS, pj0 = rb % WS;     // position rb (always live when N > 32)
  const int pi1 = (rb + 32) / WS, pj1 = (rb + 32) % WS;
  const bool live0 = kN > 32 || rb < kN;      // dead rows (-2) are written as zeros
  const bool live1 = rb + 32 < kN;
  int pair = blockIdx.x;
  const bool prof = P.prof && blockIdx.x == 0 && blockIdx.y == 0 && t == 0;
  long long t_wait = 0, t_begin = prof ? clock64() : 0;
  for (int i = 0; i < niter; ++i, pair += gridDim.x) {
    const int g = i & 1, n = i >> 1, slot = n & 1, b4 = 2 * g + slot;
    int tok[4];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int wg = 2 * pair + half;
      tok[2 * half] = tok[2 * half + 1] = -2;
      if (wg < P.total_windows) {
        const WinPos w = window_pos<WS>(P, wg);
        if (live0) tok[2 * half] = window_token<WS>(P, w, pi0, pj0);
        if (live1) tok[2 * half + 1] = window_token<WS>(P, w, pi1, pj1);
      }
    }
    const long long t0 = prof ? clock64() : 0;
    if (n >= 2) mbar_wait(bars.in_free(g, slot), ((n >> 1) - 1) & 1);
    if (prof) t_wait += clock64() - t0;
    bool any_async = false;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      load_chunk<BWD>(P, tok[k], rb + 32 * k, c, h, base + b4 * kSlot, gen + b4 * kSlot, any_async);
    fence_proxy_async_smem();
    mbar_arrive(bars.full(g, slot));                // releases this thread's st.shared rows
    cp_async_mbar_arrive_noinc(bars.full(g, slot));  // the LSU arrives when this thread's copies have landed
  }
  if (prof)
    printf("crf prof loader: niter %d total %lld cyc, waiting for a free slot %lld cyc\n", niter, clock64() - t_begin,
           t_wait);
}

// Warp-cooperative store of one 64-byte slice per tile row.  Thread `lane` holds the slice of ITS row (v[4]); the
// slices are transposed through a warp-private scratch (32 rows x 80 B) so that four consecutive threads write the
// four 16-byte chunks of one row: 8 cache lines per warp-level store instead of 32.  tokq[k] = token of row
// (lane >> 2) + 8 k (< 0: not stored).  RED: fp32 accumulate with red.global.add.v4.f32.
template <bool RED>
__device__ __forceinline__ void warp_store_rows64(uint8_t* scratch, int lane, const uint4 (&v)[4], const int (&tokq)[4],
                                                  uint8_t* gbase, int64_t row_bytes, int nchunks = 4) {
#pragma unroll
  for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(scratch + lane * 80 + 16 * c) = v[c];
  __syncwarp();
  const int c = lane & 3;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint4 d = *reinterpret_cast<const uint4*>(scratch + ((lane >> 2) + 8 * k) * 80 + 16 * c);
    if (tokq[k] >= 0 && c < nchunks) {
      uint8_t* dst = gbase + static_cast<int64_t>(tokq[k]) * row_bytes + 16 * c;
      if (RED)
        red_add_f32x4(reinterpret_cast<float*>(dst), make_float4(__uint_as_float(d.x), __uint_as_float(d.y),
                                                                 __uint_as_float(d.z), __uint_as_float(d.w)));
      else
        *reinterpret_cast<uint4*>(dst) = d;
    }
  }
  __syncwarp();
}

#define CRF_PROF_DECL(N)                                                                        \
  const bool prof = P.prof && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0;          \
  long long ph[N], tp = prof ? clock64() : 0;                                                   \
  for (int k_ = 0; k_ < N; ++k_) ph[k_] = 0
#define CRF_PROF_MARK(k) do { if (prof) { const long long t_ = clock64(); ph[k] += t_ - tp; tp = t_; } } while (0)

// =====================================================================================================
// forward
// =====================================================================================================
template <int WS>
__global__ void __launch_bounds__(kThreads, 1)
attn_fwd_async_kernel(const AttnParams P) {
  using M = Misc<WS, false>;
  constexpr int kNTok = WS * WS;
  pdl_launch_dependents();   // (the relative-position table below is a parameter: read before pdl_wait)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* misc = gen + kFwdMisc;
  float* tbl = reinterpret_cast<float*>(misc + M::kTbl);
  float* brow = reinterpret_cast<float*>(misc + M::kBias);
  const Bars bars{base + kFwdMisc + M::kBar};
  const uint32_t tmem_ptr_addr = base + kFwdMisc + M::kTmem;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(misc + M::kTmem);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const int C = P.C;
  const int niter = (P.npairs - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 12) {
    if (lane == 0) init_bars(bars);
    __syncwarp();
    tmem_alloc(tmem_ptr_addr, 256);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < M::kTblFloats; i += kThreads)
    tbl[i] = i < rpb_table_size(WS) ? __ldg(P.table + i * P.nH + h) : 0.f;
  __syncthreads();
  build_bias_rows<WS>(brow, tbl);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem = *tmem_ptr_gen;

  if (warp >= 12) {
    reg_dealloc<56>();
    if (warp == 12 && lane == 0) {
      // ================= first-stage MMA issuer: S = bias (pre-loaded) + Q [K_A;K_B]^T =================
      const uint32_t idesc_s = make_idesc(1u, 0u, 0u, 128, 128);
      for (int i = 0; i < niter; ++i) {
        const int g = i & 1, n = i >> 1, slot = n & 1;
        mbar_wait(bars.full(g, slot), (n >> 1) & 1);
        mbar_wait(bars.t_free(g), n & 1);
        tc_fence_after();
        const SmemDescBase dq = make_smem_desc_base(base + (2 * g + slot) * kSlot, 16, 512, kSwizzle64);
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks)
          umma_bf16(tmem + g * 128, smem_desc_at(dq, ks * 32), smem_desc_at(dq, 8192 + ks * 32), idesc_s, 1u);
        umma_commit(bars.s_done(g));
      }
    } else if (warp == 13 && lane == 0) {
      // ================= second-stage MMA issuer: O = P~ V =================
      // one N = 64 MMA per K step: B = [V_A | V_B], two 32-wide MN-major SW64 panels 4096 B apart (LBO), so columns
      // [0,hd) hold P~ V_A and [hd,2hd) hold P~ V_B for all 128 rows; row r reads the half of its own window
      const uint32_t idesc_o = make_idesc(1u, 0u, 1u, 128, 2 * HD);
      for (int i = 0; i < niter; ++i) {
        const int g = i & 1, n = i >> 1, slot = n & 1;
        mbar_wait(bars.p_ready(g), n & 1);
        tc_fence_after();
        const SmemDescBase dv = make_smem_desc_base(base + (2 * g + slot) * kSlot + 16384, 4096, 512, kSwizzle64);
        const SmemDescBase dp = make_smem_desc_base(base + kFwdTiles + g * 16384, 16, 1024, kSwizzle128);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          umma_bf16(tmem + g * 128, smem_desc_at(dp, ks * 32), smem_desc_at(dv, ks * 1024), idesc_o, ks > 0 ? 1u : 0u);
        umma_commit(bars.o_done(g));
        umma_commit(bars.in_free(g, slot));
      }
    }
  } else if (warp >= 8) {
    reg_dealloc<56>();
    loader_loop<WS, false>(P, bars, base, gen, h, niter);
  } else {
    // ================= compute groups =================
    reg_alloc<200>();
    const int g = warp >> 2;
    const int r = threadIdx.x & 127;
    const int half = r >> 6, pos = r & 63;
    const int pi = pos / WS, pj = pos % WS;
    const uint32_t t0 = tmem + g * 128 + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    uint8_t* Ps_g = gen + kFwdTiles + g * 16384;
    uint8_t* scratch = misc + M::kScratch + warp * kScratchWarp;
    uint64_t far_h, far_w;
    seam_sets<WS>(P.gm.shift, far_h, far_w);
    CRF_PROF_DECL(8);

    preload_bias<WS>(brow, pos, t0 + half * 64);
    tc_fence_before();
    mbar_arrive(bars.t_free(g));

    RowView rv = row_view<WS>(P, blockIdx.x + g * gridDim.x, half, pos, pi, pj, far_h, far_w);
    for (int i = g, n = 0; i < niter; i += 2, ++n) {
      const int pair = blockIdx.x + i * gridDim.x;
      const float* xmask = (P.ext_mask != nullptr && rv.tok != -2)
                               ? P.ext_mask + (static_cast<int64_t>(rv.wg % P.ext_mask_nw) * kNTok + pos) * kNTok
                               : nullptr;
      CRF_PROF_MARK(7);
      mbar_wait(bars.s_done(g), n & 1);
      CRF_PROF_MARK(0);
      tc_fence_after();
      uint32_t s0[32], s1[32];
      tmem_ld32(t0 + half * 64, s0);
      tmem_ld32(t0 + half * 64 + 32, s1);
      tmem_ld_wait();
      CRF_PROF_MARK(1);
      float p[64];
      float inv = 0.f, lse = 0.f;
      if (rv.tok != -2) {
#pragma unroll
        for (int j = 0; j < kNTok; ++j) p[j] = __uint_as_float(j < 32 ? s0[j & 31] : s1[j & 31]);
        if ((rv.m_lo | rv.m_hi) != 0u) {  // only windows on the roll seam
#pragma unroll
          for (int j = 0; j < kNTok; ++j)
            if (CRF_MASKED(rv, j)) p[j] += -100.0f;
        }
        if (xmask != nullptr) {
#pragma unroll
          for (int j = 0; j < kNTok; ++j) p[j] += __ldg(xmask + j);
        }
        float m4[4] = {p[0], p[1], p[2], p[3]};
#pragma unroll
        for (int j = 4; j < kNTok; ++j) m4[j & 3] = fmaxf(m4[j & 3], p[j]);
        const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
        const float mxl = mx * kLog2e;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          p[j] = ex2_approx(fmaf(p[j], kLog2e, -mxl));
          s4[j & 3] += p[j];
        }
        const float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
        inv = __fdividef(1.0f, sum);
        lse = mx + __logf(sum);
#pragma unroll
        for (int j = kNTok; j < 64; ++j) p[j] = 0.f;
      } else {
#pragma unroll
        for (int j = 0; j < 64; ++j) p[j] = 0.f;
      }
      CRF_PROF_MARK(2);
#pragma unroll
      for (int c = 0; c < 8; ++c)
        *reinterpret_cast<uint4*>(Ps_g + sw128_offset(r, c)) =
            make_uint4(pack_bf16(p[8 * c], p[8 * c + 1]), pack_bf16(p[8 * c + 2], p[8 * c + 3]),
                       pack_bf16(p[8 * c + 4], p[8 * c + 5]), pack_bf16(p[8 * c + 6], p[8 * c + 7]));
      CRF_PROF_MARK(3);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bars.p_ready(g));
      CRF_PROF_MARK(4);
      if (P.lse != nullptr && rv.tok != -2) P.lse[(static_cast<int64_t>(rv.wg) * P.nH + h) * 64 + pos] = lse;
      // geometry of this lane's next pair, computed while the tensor core works on O
      const RowView rv_next = row_view<WS>(P, pair + 2 * gridDim.x, half, pos, pi, pj, far_h, far_w);

      mbar_wait(bars.o_done(g), n & 1);
      CRF_PROF_MARK(5);
      tc_fence_after();
      uint32_t o[32];
      tmem_ld32(t0 + half * HD, o);
      tmem_ld_wait();
      preload_bias<WS>(brow, pos, t0 + half * 64);  // the next S of this lane accumulates on top of the bias
      tc_fence_before();
      mbar_arrive(bars.t_free(g));
      CRF_PROF_MARK(6);
      {
        uint4 v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c)
          v[c] = make_uint4(pack_bf16(inv * __uint_as_float(o[8 * c]), inv * __uint_as_float(o[8 * c + 1])),
                            pack_bf16(inv * __uint_as_float(o[8 * c + 2]), inv * __uint_as_float(o[8 * c + 3])),
                            pack_bf16(inv * __uint_as_float(o[8 * c + 4]), inv * __uint_as_float(o[8 * c + 5])),
                            pack_bf16(inv * __uint_as_float(o[8 * c + 6]), inv * __uint_as_float(o[8 * c + 7])));
        int tq[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) tq[k] = __shfl_sync(0xffffffffu, rv.tok, (lane >> 2) + 8 * k);
        warp_store_rows64<false>(scratch, lane, v, tq, reinterpret_cast<uint8_t*>(P.o) + h * P.hd * 2,
                                 static_cast<int64_t>(C) * 2, P.hd / 8);
      }
      rv = rv_next;
    }
    if (prof)
      printf("crf prof fwd compute (lane 0): pairs %d | wait S %lld | ld S %lld | math %lld | P tile %lld | fence+arrive "
             "%lld | wait O %lld | ld O + bias preload %lld | store + next row view %lld cyc\n",
             (niter + 1) / 2, ph[0], ph[1], ph[2], ph[3], ph[4], ph[5], ph[6], ph[7]);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 12) {
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

// =====================================================================================================
// backward
// =====================================================================================================
template <int WS>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_async_kernel(const AttnParams P) {
  using M = Misc<WS, true>;
  constexpr int kNTok = WS * WS;
  pdl_launch_dependents();   // (the relative-position table below is a parameter: read before pdl_wait)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* misc = gen + kBwdMisc;
  float* tbl = reinterpret_cast<float*>(misc + M::kTbl);
  float* brow = reinterpret_cast<float*>(misc + M::kBias);
  const Bars bars{base + kBwdMisc + M::kBar};
  const uint32_t tmem_ptr_addr = base + kBwdMisc + M::kTmem;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(misc + M::kTmem);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const int C = P.C;
  const int niter = (P.npairs - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 12) {
    if (lane == 0) init_bars(bars);
    __syncwarp();
    tmem_alloc(tmem_ptr_addr, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < M::kTblFloats; i += kThreads)
    tbl[i] = i < rpb_table_size(WS) ? __ldg(P.table + i * P.nH + h) : 0.f;
  __syncthreads();
  if constexpr (M::kBiasRows) build_bias_rows<WS>(brow, tbl);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem = *tmem_ptr_gen;

  if (warp >= 12) {
    reg_dealloc<56>();
    if (warp == 12 && lane == 0) {
      // ================= first-stage MMA issuer: S (on the pre-loaded bias) and dP, M = 128 =================
      const uint32_t idesc_s = make_idesc(1u, 0u, 0u, 128, 128);
      for (int i = 0; i < niter; ++i) {
        const int g = i & 1, n = i >> 1, slot = n & 1;
        mbar_wait(bars.full(g, slot), (n >> 1) & 1);
        mbar_wait(bars.t_free(g), n & 1);
        tc_fence_after();
        const SmemDescBase din = make_smem_desc_base(base + (2 * g + slot) * kSlot, 16, 512, kSwizzle64);
        const uint32_t t0 = tmem + g * 256;
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks)  // S += Q K^T -> cols [0,128)
          umma_bf16(t0, smem_desc_at(din, ks * 32), smem_desc_at(din, 8192 + ks * 32), idesc_s, 1u);
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks)  // dP = dO V^T -> cols [128,256)
          umma_bf16(t0 + 128, smem_desc_at(din, 24576 + ks * 32), smem_desc_at(din, 16384 + ks * 32), idesc_s,
                    ks > 0 ? 1u : 0u);
        umma_commit(bars.s_done(g));
      }
    } else if (warp == 13 && lane == 0) {
      // ================= second-stage MMA issuer: per window, M = 64 =================
      const uint32_t idesc_t = make_idesc(1u, 1u, 1u, 64, HD);    // dV, dK: MN-major x MN-major
      const uint32_t idesc_q = make_idesc(1u, 0u, 1u, 64, HD);    // dQ    : K-major x MN-major
      for (int i = 0; i < niter; ++i) {
        const int g = i & 1, n = i >> 1, slot = n & 1;
        mbar_wait(bars.p_ready(g), n & 1);
        tc_fence_after();
        const SmemDescBase din = make_smem_desc_base(base + (2 * g + slot) * kSlot, 512, 512, kSwizzle64);  // MN-major B
        const SmemDescBase dtA = make_smem_desc_base(base + kBwdTiles + g * 32768, 8192, 1024, kSwizzle128);  // MN-major A
        const SmemDescBase dtK = make_smem_desc_base(base + kBwdTiles + g * 32768, 16, 1024, kSwizzle128);    // K-major A
#pragma unroll
        for (int w = 0; w < 2; ++w) {  // window w: tile rows [64w, 64w+64), TMEM lanes 16w + {0..15} + 32k
          const uint32_t t0 = tmem + g * 256 + (static_cast<uint32_t>(16 * w) << 16);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)  // dV_w = P_w^T dO_w : K = 64 query rows
            umma_bf16(t0, smem_desc_at(dtA, w * 8192 + ks * 2048), smem_desc_at(din, 24576 + w * 4096 + ks * 1024),
                      idesc_t, ks > 0 ? 1u : 0u);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)  // dK_w = dS_w^T Q_w
            umma_bf16(t0 + 32, smem_desc_at(dtA, 16384 + w * 8192 + ks * 2048), smem_desc_at(din, w * 4096 + ks * 1024),
                      idesc_t, ks > 0 ? 1u : 0u);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)  // dQ_w = dS_w K_w : K = 64 keys
            umma_bf16(t0 + 64, smem_desc_at(dtK, 16384 + w * 8192 + ks * 32),
                      smem_desc_at(din, 8192 + w * 4096 + ks * 1024), idesc_q, ks > 0 ? 1u : 0u);
        }
        umma_commit(bars.o_done(g));
        umma_commit(bars.in_free(g, slot));
      }
    }
  } else if (warp >= 8) {
    reg_dealloc<56>();
    loader_loop<WS, true>(P, bars, base, gen, h, niter);
  } else {
    // ================= compute groups =================
    reg_alloc<200>();
    const int g = warp >> 2;
    const int r = threadIdx.x & 127;
    const int half = r >> 6, pos = r & 63;
    const int pi = pos / WS, pj = pos % WS;
    // second-stage results (M = 64 per window): this thread's TMEM lane holds row epos of window ehalf
    const int ehalf = lane >> 4, epos = 16 * (warp & 3) + (lane & 15);
    const int epi_i = epos / WS, epi_j = epos % WS;
    const uint32_t t0 = tmem + g * 256 + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    uint8_t* Pb_g = gen + kBwdTiles + g * 32768;
    uint8_t* Db_g = Pb_g + 16384;
    uint8_t* scratch = misc + M::kScratch + warp * kScratchWarp;
    const int bi = rpb_base<WS>(pos < kNTok ? pos : 0);
    uint64_t far_h, far_w;
    seam_sets<WS>(P.gm.shift, far_h, far_w);
    float dtab[kNTok];
#pragma unroll
    for (int j = 0; j < kNTok; ++j) dtab[j] = 0.f;
    CRF_PROF_DECL(8);

    preload_row_bias<WS, true>(brow, tbl, pos, t0 + half * 64);
    tc_fence_before();
    mbar_arrive(bars.t_free(g));

    // per-pair row state, always computed one pair ahead (while the tensor core runs the second stage)
    auto row_state = [&](int pr, RowView& v, float& l, int& et) {
      v = row_view<WS>(P, pr, half, pos, pi, pj, far_h, far_w);
      l = 0.f;
      if (v.tok >= 0) l = __ldg(P.lse + (static_cast<int64_t>(v.wg) * P.nH + h) * 64 + pos);
      et = -2;
      const int ewg = 2 * pr + ehalf;
      if (epos < kNTok && ewg < P.total_windows) et = window_token<WS>(P, window_pos<WS>(P, ewg), epi_i, epi_j);
    };
    RowView rv;
    float lse;
    int etok;
    row_state(blockIdx.x + g * gridDim.x, rv, lse, etok);
    for (int i = g, n = 0; i < niter; i += 2, ++n) {
      const int pair = blockIdx.x + i * gridDim.x;
      const float* xmask = (P.ext_mask != nullptr && rv.tok != -2)
                               ? P.ext_mask + (static_cast<int64_t>(rv.wg % P.ext_mask_nw) * kNTok + pos) * kNTok
                               : nullptr;
      CRF_PROF_MARK(7);
      mbar_wait(bars.s_done(g), n & 1);
      CRF_PROF_MARK(0);
      tc_fence_after();
      float p[64], ds[64];
      {
        uint32_t s0[32], s1[32];
        tmem_ld32(t0 + half * 64, s0);
        tmem_ld32(t0 + half * 64 + 32, s1);
        tmem_ld_wait();
        CRF_PROF_MARK(1);
        if (rv.tok >= 0) {
#pragma unroll
          for (int j = 0; j < kNTok; ++j) p[j] = __uint_as_float(j < 32 ? s0[j & 31] : s1[j & 31]);
          if ((rv.m_lo | rv.m_hi) != 0u) {  // only windows on the roll seam
#pragma unroll
            for (int j = 0; j < kNTok; ++j)
              if (CRF_MASKED(rv, j)) p[j] += -100.0f;
          }
          if (xmask != nullptr) {
#pragma unroll
            for (int j = 0; j < kNTok; ++j) p[j] += __ldg(xmask + j);
          }
          const float lsel = lse * kLog2e;
#pragma unroll
          for (int j = 0; j < kNTok; ++j) p[j] = ex2_approx(fmaf(p[j], kLog2e, -lsel));
        } else {
#pragma unroll
          for (int j = 0; j < kNTok; ++j) p[j] = 0.f;
        }
#pragma unroll
        for (int j = kNTok; j < 64; ++j) p[j] = 0.f;
      }
      {
        uint32_t g0[32], g1[32];
        tmem_ld32(t0 + 128 + half * 64, g0);
        tmem_ld32(t0 + 128 + half * 64 + 32, g1);
        tmem_ld_wait();
        float d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          ds[j] = __uint_as_float(j < 32 ? g0[j & 31] : g1[j & 31]);
          d4[j & 3] = fmaf(p[j], ds[j], d4[j & 3]);
        }
        const float dsum = (d4[0] + d4[1]) + (d4[2] + d4[3]);
#pragma unroll
        for (int j = 0; j < kNTok; ++j) {
          ds[j] = p[j] * (ds[j] - dsum);
          dtab[j] += ds[j];
        }
#pragma unroll
        for (int j = kNTok; j < 64; ++j) ds[j] = 0.f;
      }
      CRF_PROF_MARK(2);
#pragma unroll
      for (int c = 0; c < 8; ++c) {  // compact tiles: row r = query, 64 key columns of its own window
        const uint32_t off = sw128_offset(r, c);
        *reinterpret_cast<uint4*>(Pb_g + off) =
            make_uint4(pack_bf16(p[8 * c], p[8 * c + 1]), pack_bf16(p[8 * c + 2], p[8 * c + 3]),
                       pack_bf16(p[8 * c + 4], p[8 * c + 5]), pack_bf16(p[8 * c + 6], p[8 * c + 7]));
        *reinterpret_cast<uint4*>(Db_g + off) =
            make_uint4(pack_bf16(ds[8 * c], ds[8 * c + 1]), pack_bf16(ds[8 * c + 2], ds[8 * c + 3]),
                       pack_bf16(ds[8 * c + 4], ds[8 * c + 5]), pack_bf16(ds[8 * c + 6], ds[8 * c + 7]));
      }
      CRF_PROF_MARK(3);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bars.p_ready(g));
      CRF_PROF_MARK(4);
      RowView rv_next;
      float lse_next;
      int etok_next;
      row_state(pair + 2 * gridDim.x, rv_next, lse_next, etok_next);

      mbar_wait(bars.o_done(g), n & 1);
      CRF_PROF_MARK(5);
      tc_fence_after();
      uint32_t a[32], b[32], c2[32];
      tmem_ld32(t0, a);
      tmem_ld32(t0 + 32, b);
      tmem_ld32(t0 + 64, c2);
      tmem_ld_wait();
      {
        int tq[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) tq[k] = __shfl_sync(0xffffffffu, etok, (lane >> 2) + 8 * k);
        uint4 v[4];
        uint8_t* dvb = reinterpret_cast<uint8_t*>(P.dv) + h * P.hd * 4;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {  // dv: 4 * head_dim bytes per row, 64-byte passes
          if (16 * hf >= P.hd) break;
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = make_uint4(a[16 * hf + 4 * c], a[16 * hf + 4 * c + 1], a[16 * hf + 4 * c + 2], a[16 * hf + 4 * c + 3]);
          if (P.dv_acc) warp_store_rows64<true>(scratch, lane, v, tq, dvb + 64 * hf, static_cast<int64_t>(C) * 4);
          else warp_store_rows64<false>(scratch, lane, v, tq, dvb + 64 * hf, static_cast<int64_t>(C) * 4);
        }
        uint8_t* dqb = reinterpret_cast<uint8_t*>(P.dqk) + h * P.hd * 2;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          v[c] = make_uint4(pack_bf16(__uint_as_float(b[8 * c]), __uint_as_float(b[8 * c + 1])),
                            pack_bf16(__uint_as_float(b[8 * c + 2]), __uint_as_float(b[8 * c + 3])),
                            pack_bf16(__uint_as_float(b[8 * c + 4]), __uint_as_float(b[8 * c + 5])),
                            pack_bf16(__uint_as_float(b[8 * c + 6]), __uint_as_float(b[8 * c + 7])));
        warp_store_rows64<false>(scratch, lane, v, tq, dqb + C * 2, static_cast<int64_t>(C) * 4, P.hd / 8);  // dk
        // zero-padded keys: k == bias, so their gradient goes to the k half of qk.bias (warp-reduced, one atomic/lane)
        if (__any_sync(0xffffffffu, etok == -1)) {
          float mine = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float s = warp_sum(etok == -1 ? __uint_as_float(b[j]) : 0.f);
            if (lane == j) mine = s;
          }
          if (lane < P.hd) atomicAdd(P.d_qk_bias + C + h * P.hd + lane, mine);
        }
        // dv and dk are on their way (64 of the 96 result registers are dead): pre-load the bias and hand the TMEM
        // columns back BEFORE the last store, so the next first-stage MMAs of this lane run under it
        preload_row_bias<WS, true>(brow, tbl, pos, t0 + half * 64);
        tc_fence_before();
        mbar_arrive(bars.t_free(g));
        const float sc = P.scale;  // d(xW+b) = dq * scale because q was stored pre-scaled
#pragma unroll
        for (int c = 0; c < 4; ++c)
          v[c] = make_uint4(pack_bf16(sc * __uint_as_float(c2[8 * c]), sc * __uint_as_float(c2[8 * c + 1])),
                            pack_bf16(sc * __uint_as_float(c2[8 * c + 2]), sc * __uint_as_float(c2[8 * c + 3])),
                            pack_bf16(sc * __uint_as_float(c2[8 * c + 4]), sc * __uint_as_float(c2[8 * c + 5])),
                            pack_bf16(sc * __uint_as_float(c2[8 * c + 6]), sc * __uint_as_float(c2[8 * c + 7])));
        warp_store_rows64<false>(scratch, lane, v, tq, dqb, static_cast<int64_t>(C) * 4, P.hd / 8);  // dq
      }
      CRF_PROF_MARK(6);
      rv = rv_next;
      lse = lse_next;
      etok = etok_next;
    }
    if (prof)
      printf("crf prof bwd compute (lane 0): pairs %d | wait S,dP %lld | ld S %lld | math %lld | P,dS tiles %lld | "
             "fence+arrive %lld | wait 2nd stage %lld | ld + stores + bias preload %lld | next row view %lld cyc\n",
             (niter + 1) / 2, ph[0], ph[1], ph[2], ph[3], ph[4], ph[5], ph[6], ph[7]);

    // relative-position-bias gradient: dTable[idx(i,j), h] += sum over my pairs of dS[i][j]
    named_bar_sync(1, 256);  // both compute groups are past their last read of tbl
    if (threadIdx.x < M::kTblFloats) tbl[threadIdx.x] = 0.f;
    named_bar_sync(1, 256);
    if (pos < kNTok) {
#pragma unroll
      for (int j = 0; j < kNTok; ++j) atomicAdd(tbl + bi - rpb_col<WS>(j), dtab[j]);
    }
    named_bar_sync(1, 256);
    if (threadIdx.x < rpb_table_size(WS)) atomicAdd(P.d_table + threadIdx.x * P.nH + h, tbl[threadIdx.x]);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 12) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

int grid_x(const AttnParams& P, const crf_block_desc& d) {
  int gx = num_sms(d.device) / P.nH;  // one 512-thread CTA per SM, never a partial second wave
  if (gx > (P.npairs + 1) / 2) gx = (P.npairs + 1) / 2;  // at least two pairs per CTA so both lanes work
  return gx < 1 ? 1 : gx;
}

template <int WS>
int launch_fwd(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  constexpr size_t smem = kFwdMisc + Misc<WS, false>::kBytes + 1024;
  static_assert(smem <= 232448, "shared-memory plan exceeds 227 KB");
  CRF_CUDA(cudaFuncSetAttribute(attn_fwd_async_kernel<WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const double TC = static_cast<double>(d.B) * d.H * d.W * d.C;
  const double N = WS * WS;
  KernelTimer tm(st, 4.0 * N * N * d.C * P.total_windows, 8.0 * TC, "attn_fwd_B%d_%dx%d_C%d_s%d", d.B, d.H, d.W, d.C,
                 d.shift);
  launch_pdl(attn_fwd_async_kernel<WS>, dim3(grid_x(P, d), P.nH), kThreads, smem, st, P);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

template <int WS>
int launch_bwd(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  constexpr size_t smem = kBwdMisc + Misc<WS, true>::kBytes + 1024;
  static_assert(smem <= 232448, "shared-memory plan exceeds 227 KB");
  CRF_CUDA(cudaFuncSetAttribute(attn_bwd_async_kernel<WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const double TC = static_cast<double>(d.B) * d.H * d.W * d.C;
  const double N = WS * WS;
  KernelTimer tm(st, 10.0 * N * N * d.C * P.total_windows, 16.0 * TC, "attn_bwd_B%d_%dx%d_C%d_s%d", d.B, d.H, d.W,
                 d.C, d.shift);
  launch_pdl(attn_bwd_async_kernel<WS>, dim3(grid_x(P, d), P.nH), kThreads, smem, st, P);
  CRF_CUDA(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace

int launch_attn_fwd_async(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  const int rc = with_window(P.gm.ws, [&](auto w) { return launch_fwd<decltype(w)::value>(P, d, st); });
  return rc >= 0 ? rc : set_error("attention core: no kernel for window %d", P.gm.ws);
}

int launch_attn_bwd_async(const AttnParams& P, const crf_block_desc& d, cudaStream_t st) {
  const int rc = with_window(P.gm.ws, [&](auto w) { return launch_bwd<decltype(w)::value>(P, d, st); });
  return rc >= 0 ? rc : set_error("attention core: no kernel for window %d", P.gm.ws);
}

}  // namespace crf
