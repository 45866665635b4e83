// Epilogue building blocks shared by the GEMM kernels: per-thread processing of 32 accumulator columns of one row
// (bias, scale, residual, exact-erf GELU, GELU derivative) and the swizzled slab stores that feed the TMA stores.
#pragma once
#include <type_traits>

#include "crf_host.h"
#include "crf_ptx.cuh"

namespace crf {

struct EpiParams {
  const float* bias;
  float scale;
  int scale_cols;
  int m_pad;       // split-K: rows per split in the partial buffer
  int store_out0;  // BIAS_GELU: 0 -> skip the pre-activation output (inference)
  float* colsum;   // wgrad only: colsum[m] += sum_k A(m,k)  (the bias gradient), or nullptr
  int tma_reduce;  // split-K: 1 -> every split adds its tile into the output with a TMA reduction (no partial buffer)
};

__device__ __forceinline__ void add_bias32(float (&v)[32], const float* bias, int n) {
  if (bias == nullptr) return;
  const float4* b4 = reinterpret_cast<const float4*>(bias + n);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 b = __ldg(b4 + j);
    v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
  }
}
// 32 fp32 values -> 4 x 16-byte chunks of bf16 at chunk index c0.. of row r of a swizzled slab
__device__ __forceinline__ void store_bf16_32(uint8_t* slab, int r, int c0, const float (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    *reinterpret_cast<uint4*>(slab + sw128_offset(r, c0 + j)) =
        make_uint4(pack_bf16(v[8 * j], v[8 * j + 1]), pack_bf16(v[8 * j + 2], v[8 * j + 3]),
                   pack_bf16(v[8 * j + 4], v[8 * j + 5]), pack_bf16(v[8 * j + 6], v[8 * j + 7]));
}

// One thread, one accumulator row, 32 consecutive columns starting at global column n.  `half` selects the 64-byte
// half of a bf16 slab row; fp32 slabs hold exactly these 32 columns.  o0 / xb are the (generic-address) slab buffers.
template <int EPI>
__device__ __forceinline__ void epi_group32(const uint32_t (&acc)[32], const EpiParams& ep, int n, int r, int half,
                                            uint8_t* o0, uint8_t* xb) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
  if constexpr (EPI == CRF_EPI_STORE_F32 || EPI == CRF_EPI_SPLITK_F32) {
    add_bias32(v, ep.bias, n);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      *reinterpret_cast<float4*>(o0 + sw128_offset(r, j)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  } else if constexpr (EPI == CRF_EPI_BIAS_RES_F32) {
    add_bias32(v, ep.bias, n);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 q = *reinterpret_cast<const float4*>(xb + sw128_offset(r, j));
      *reinterpret_cast<float4*>(o0 + sw128_offset(r, j)) =
          make_float4(v[4 * j] + q.x, v[4 * j + 1] + q.y, v[4 * j + 2] + q.z, v[4 * j + 3] + q.w);
    }
  } else if constexpr (EPI == CRF_EPI_STORE_BF16) {
    add_bias32(v, ep.bias, n);
    if (n < ep.scale_cols) {  // scale_cols is a multiple of 32: a 32-column group is on one side
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] *= ep.scale;
    }
    store_bf16_32(o0, r, half * 4, v);
  } else if constexpr (EPI == CRF_EPI_BIAS_GELU) {
    add_bias32(v, ep.bias, n);
    if (ep.store_out0) store_bf16_32(o0, r, half * 4, v);
#pragma unroll
    for (int j = 0; j < 16; ++j) gelu_erf2(v[2 * j], v[2 * j + 1]);   // packed fp32x2, bit-identical to gelu_erf
    store_bf16_32(xb, r, half * 4, v);
  } else if constexpr (EPI == CRF_EPI_MUL_DGELU) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 p = *reinterpret_cast<const uint4*>(xb + sw128_offset(r, half * 4 + j));
      const uint32_t pw[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int q = 0; q < 4; ++q)   // packed fp32x2: same operations, same order as dgelu_erf on each value
        f2_unpack(f2_mul(f2_pack(v[8 * j + 2 * q], v[8 * j + 2 * q + 1]), dgelu_erf2(bf16_lo(pw[q]), bf16_hi(pw[q]))),
                  v[8 * j + 2 * q], v[8 * j + 2 * q + 1]);
    }
    store_bf16_32(o0, r, half * 4, v);
  }
}

template <int EPI>
struct EpiTraits {
  static constexpr bool kOutF32 = (EPI == CRF_EPI_STORE_F32 || EPI == CRF_EPI_BIAS_RES_F32 || EPI == CRF_EPI_SPLITK_F32);
  static constexpr bool kHasAux = (EPI == CRF_EPI_BIAS_RES_F32 || EPI == CRF_EPI_MUL_DGELU);
  static constexpr bool kHasOut1 = (EPI == CRF_EPI_BIAS_GELU);
  static constexpr int kSlabCols = kOutF32 ? 32 : 64;
};

// Calls f(std::integral_constant<int, EPI>()) for a GEMM epilogue (the kernels are instantiated per epilogue) and
// returns its result.
template <typename F>
int with_epi(int epi, F&& f) {
  switch (epi) {
    case CRF_EPI_STORE_F32: return f(std::integral_constant<int, CRF_EPI_STORE_F32>());
    case CRF_EPI_STORE_BF16: return f(std::integral_constant<int, CRF_EPI_STORE_BF16>());
    case CRF_EPI_BIAS_RES_F32: return f(std::integral_constant<int, CRF_EPI_BIAS_RES_F32>());
    case CRF_EPI_BIAS_GELU: return f(std::integral_constant<int, CRF_EPI_BIAS_GELU>());
    case CRF_EPI_MUL_DGELU: return f(std::integral_constant<int, CRF_EPI_MUL_DGELU>());
    case CRF_EPI_SPLITK_F32: return f(std::integral_constant<int, CRF_EPI_SPLITK_F32>());
    default: return set_error("crf_gemm: unknown epilogue %d", epi);
  }
}

// m_pad and tma_reduce: the tiled kernel's split-K (0 for the other kernels and epilogues)
inline EpiParams epi_params(const crf_gemm_args& a, int m_pad, int tma_reduce) {
  EpiParams ep;
  ep.bias = a.bias;
  ep.scale = a.scale;
  ep.scale_cols = a.scale_cols;
  ep.m_pad = m_pad;
  ep.store_out0 = a.out0 != nullptr ? 1 : 0;
  ep.colsum = a.a_major == 1 ? a.colsum : nullptr;
  ep.tma_reduce = tma_reduce;
  return ep;
}

// Algorithmic HBM bytes of a GEMM with epilogue epi (KernelTimer): both operands once (twice as wide with split3), the
// outputs once, the aux input once.
inline double gemm_bytes(const crf_gemm_args& a, int epi) {
  const double mn = static_cast<double>(a.M) * a.N;
  const double out_bytes = epi == CRF_EPI_STORE_BF16 ? 2 * mn
                           : epi == CRF_EPI_BIAS_RES_F32 ? 8 * mn
                           : epi == CRF_EPI_BIAS_GELU ? (a.out0 != nullptr ? 4 * mn : 2 * mn)
                           : 4 * mn;
  return (a.split3 ? 2.0 : 1.0) * 2.0 * (static_cast<double>(a.M) + a.N) * a.K + out_bytes;
}

}  // namespace crf
