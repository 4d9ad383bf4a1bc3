// Host-side setup shared by the tcgen05 kernels: TMA tensor maps and UMMA instruction descriptors.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace b200 {

// Encodes a tiled TMA map with the options every tcgen05 kernel here uses: no interleave, 128-byte swizzle, L2 256-byte promotion,
// no out-of-bounds fill, element strides 1.  `dims` and `box` have `rank` entries, `strides` (bytes) rank - 1.  Binds the primary
// context first (see bind_primary_context).  On failure records "cuTensorMapEncodeTiled (<who>) ..." as the last error and returns false.
bool encode_tiled(CUtensorMap* out, CUtensorMapDataType type, uint32_t rank, const void* ptr, const cuuint64_t* dims,
                  const cuuint64_t* strides, const cuuint32_t* box, const char* who);

namespace gemm {
// 3-D map {inner (contiguous), rows, batch} of a bf16 / fp16 operand (2-byte elements) or, with dtype kF32, of an fp32 output (TMA-store
// maps); box {box_inner, box_rows, 1}.  Cached by all its arguments.  Defined in gemm_sm100.cu.
bool make_map(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t rows, uint64_t batch, uint64_t ld, uint64_t bstride,
              uint32_t box_inner, uint32_t box_rows, int dtype);
}  // namespace gemm

// UMMA instruction descriptor (cute::UMMA::InstrDescriptor bit layout) for an M x N tile with fp32 accumulation.
//   a_fmt / b_fmt  kind::f16: F16 = 0, BF16 = 1;  kind::f8f6f4 / mxf8f6f4: E4M3 = 0, E5M2 = 1
//   a_mn / b_mn    operand is MN-major (1) or K-major (0)
//   block_scaled   cute::UMMA::InstrDescriptorBlockScaled: no c_format (always fp32); bits [4,6) b_sf_id, 23 scale format
//                  (1 = E8M0), [29,31) a_sf_id - the issuer ORs the two ids in per MMA
inline uint32_t umma_idesc(uint32_t a_fmt, uint32_t b_fmt, bool a_mn, bool b_mn, int m, int n, bool block_scaled) {
  uint32_t d = 0;
  if (!block_scaled) d |= 1u << 4;                // c_format = F32
  d |= a_fmt << 7;                                // a_format
  d |= b_fmt << 10;                               // b_format
  d |= (a_mn ? 1u : 0u) << 15;                    // a_major
  d |= (b_mn ? 1u : 0u) << 16;                    // b_major
  d |= (uint32_t)(n >> 3) << 17;                  // n_dim
  if (block_scaled) d |= 1u << 23;                // scale format E8M0
  d |= (uint32_t)(m >> 4) << 24;                  // m_dim
  return d;
}

}  // namespace b200
