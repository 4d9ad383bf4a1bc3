// FP8 (E4M3 / E5M2) GEMM for sm_100a: same persistent warp-specialised structure as gemm_sm100.cu (TMA -> 128B-swizzled smem
// ring -> tcgen05.mma -> TMEM double-buffered accumulators -> tcgen05.ld epilogue), with `kind::f8f6f4` MMAs (K = 32 per
// instruction, 2x the bf16 rate), fp32 accumulation and a per-tensor dequantisation scale (+ bias / activation) fused in the
// epilogue.  Both operands are K-major ("TN" GEMM): A [M,K], B [N,K], 1 byte per element.
//
// MX variant (`MX = true`, BN = 128): OCP microscaling - one E8M0 (power-of-two) scale per 32 consecutive K elements of every A row
// and B row.  The scale bytes travel as 512-byte blocks (128 rows x 4 k-blocks, byte = (row % 32) * 16 + (row / 32) * 4 + k-block: the
// layout tcgen05.cp.32x128b.warpx4 scatters into 4 TMEM columns of every lane quadrant), one bulk copy per operand and stage; the issuer
// copies them smem -> TMEM in front of the stage's four `tcgen05.mma.kind::mxf8f6f4.block_scale` (the k-block is selected by the
// a_sf_id / b_sf_id fields of the instruction descriptor), so dequantisation costs no epilogue work and no extra pass.
//
// Parity (behaviour): fp8_fp8_half_gemm_fused (paddle/phi/kernels/fusion/fp8_gemm/fp8_gemm_with_cublasLt/*) which calls cuBLASLt.
#include <cuda.h>
#include <cstdio>

#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_ptx.cuh"
#include "include/b200_tcgen05_host.h"

namespace b200 {
namespace gemm8 {
using namespace ptx;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 128;  // 128 x 1B = 128B = one swizzle atom row
constexpr int UMMA_K = 32;    // kind::f8f6f4: 32 elements (32 bytes) per MMA along K
constexpr int kStages = 4;
constexpr int kThreads = 256;
constexpr int kAccStages = 2;
constexpr uint32_t A_STAGE_BYTES = BLOCK_M * BLOCK_K;      // 16 KB

constexpr uint32_t SF_BLOCK_BYTES = 512;   // scale bytes of 128 rows x 128 k (4 blocks of 32)

template <int BN, bool MX = false> struct Cfg {
  static constexpr uint32_t B_STAGE_BYTES = BN * BLOCK_K;
  static constexpr uint32_t SF_BYTES = MX ? 2048u : 0u;          // [SFA 512 | SFB 512 per 128 columns] behind the operand tiles
  static constexpr uint32_t SF_TX = MX ? SF_BLOCK_BYTES * (1 + BN / 128) : 0u;
  static constexpr uint32_t STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES + SF_BYTES;
  static constexpr uint32_t TX_BYTES = A_STAGE_BYTES + B_STAGE_BYTES + SF_TX;
  // MX at BN = 256 keeps ONE accumulator (256 columns) so that the scale columns fit: a 128-wide tile reads A and B from shared memory
  // at 128 B/clk for full-rate fp8 MMAs - all the pipe has, before the TMA writes - and tops out at ~1.5 PFLOP/s; the 256-wide tile
  // needs 96 B/clk and wins even without the epilogue overlap.
  static constexpr int ACC = (MX && BN == 256) ? 1 : kAccStages;
  static constexpr uint32_t SF_COL0 = ACC * BN;                  // MX: per smem stage 4 columns SFA + BN / 32 columns SFB after the accumulators
  static constexpr uint32_t SF_STAGE_COLS = BN == 256 ? 16 : 8;
  static constexpr uint32_t TMEM_COLS = MX ? 512u : kAccStages * BN;  // powers of two >= 32
  static constexpr uint32_t SMEM_BYTES = kStages * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(!MX || ACC * BN + kStages * SF_STAGE_COLS <= 512, "MX: TMEM budget");
  static_assert(SMEM_BYTES <= 232448, "fp8 gemm: shared memory budget");
};

struct Params {
  int m, n, k, batch;
  void* d;
  const void* bias;
  int64_t ldd, stride_d;
  int in_dtype, out_dtype;
  int has_bias, act, accumulate;
  float scale;
  const float* scale_a;   // optional device scalars (per-tensor dequantisation factors produced by quantize_fp8): no host round trip
  const float* scale_b;
  const uint8_t* sfa;     // MX: E8M0 scale blocks [m / 128][k / 128][512] of A, same for B over n
  const uint8_t* sfb;
  uint32_t idesc;
};

template <int BN, bool MX>
__global__ void __launch_bounds__(kThreads, 1)
gemm_fp8_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const Params p) {
  using C = Cfg<BN, MX>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // SWIZZLE_128B needs 1024B alignment
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + kStages * C::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStages + kAccStages + s); };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_gen + kStages * C::STAGE_BYTES + 8 * (2 * kStages + 2 * kAccStages));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (p.m + BLOCK_M - 1) / BLOCK_M, num_n = (p.n + BN - 1) / BN;
  const int tiles_per_batch = num_m * num_n;
  const int num_tiles = tiles_per_batch * p.batch;
  const int num_kb = (p.k + BLOCK_K - 1) / BLOCK_K;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < kAccStages; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 4); }
    fence_barrier_init();
    fence_proxy_async();
  } else if (warp == 2) {
    tmem_alloc(smem_u32((const void*)tmem_ptr_smem), C::TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // tile order: groups of 8 M-tiles sweep N (operand panels stay L2-resident across the wave)
  auto tile_coords = [&](int tile, int& bz, int& mb, int& nb) {
    bz = tile / tiles_per_batch;
    const int t = tile - bz * tiles_per_batch;
    constexpr int GROUP_M = 8;
    const int in_group = GROUP_M * num_n;
    const int g = t / in_group;
    const int first_m = g * GROUP_M;
    const int gsz = min(num_m - first_m, GROUP_M);
    const int r = t - g * in_group;
    mb = first_m + r % gsz;
    nb = r / gsz;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ================= TMA producer =================
      int stage = 0;
      uint32_t phase = 0;
      const uint64_t hint = 0x1000000000000000ull;  // EVICT_NORMAL
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int bz, mb, nb;
        tile_coords(tile, bz, mb, nb);
        const int m0 = mb * BLOCK_M, n0 = nb * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
          mbar_expect_tx(full_bar(stage), C::TX_BYTES);
          const int k0 = kb * BLOCK_K;
          tma_load_3d(sa, &map_a, full_bar(stage), k0, m0, bz, hint);  // box {128 k bytes, 128 m}
          tma_load_3d(sb, &map_b, full_bar(stage), k0, n0, bz, hint);  // box {128 k bytes, BN n}
          if constexpr (MX) {
            bulk_load(sb + C::B_STAGE_BYTES, p.sfa + ((int64_t)mb * num_kb + kb) * SF_BLOCK_BYTES, SF_BLOCK_BYTES, full_bar(stage));
#pragma unroll
            for (int h = 0; h < BN / 128; ++h)
              bulk_load(sb + C::B_STAGE_BYTES + (1 + h) * SF_BLOCK_BYTES, p.sfb + ((int64_t)(nb * (BN / 128) + h) * num_kb + kb) * SF_BLOCK_BYTES, SF_BLOCK_BYTES, full_bar(stage));
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ================= MMA issuer =================
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      const uint64_t desc_a0 = make_smem_desc(smem_base, 16, 1024), desc_b0 = make_smem_desc(smem_base + A_STAGE_BYTES, 16, 1024);
      const uint64_t desc_sf0 = make_sf_desc(smem_base + A_STAGE_BYTES + C::B_STAGE_BYTES);
      (void)desc_sf0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++local) {
        const int as = local % C::ACC;
        const uint32_t aphase = (local / C::ACC) & 1;
        mbar_wait(tempty_bar(as), aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          // descriptors are built once (desc_a0 / desc_b0 / desc_sf0 below the loop head) and advanced by adding to the address field
          const uint64_t soff = (uint64_t)((stage * C::STAGE_BYTES) >> 4);
          uint32_t tsfa = 0, tsfb = 0;
          if constexpr (MX) {      // scale bytes smem -> TMEM; tcgen05.cp and tcgen05.mma execute in issue order
            tsfa = tmem_base + C::SF_COL0 + stage * C::SF_STAGE_COLS;
            tsfb = tsfa + 4;
            tmem_cp_sf(tsfa, desc_sf0 + soff);
#pragma unroll
            for (int h = 0; h < BN / 128; ++h) tmem_cp_sf(tsfb + 4 * h, desc_sf0 + soff + (uint64_t)(((1 + h) * SF_BLOCK_BYTES) >> 4));
          }
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = desc_a0 + soff + 2 * k, bdesc = desc_b0 + soff + 2 * k;   // K-major: 32 fp8 elements = 32 B per step
            if constexpr (MX) umma_mxf8(tmem_d, adesc, bdesc, p.idesc | ((uint32_t)k << 29) | ((uint32_t)k << 4), tsfa, tsfb, (kb | k) != 0);   // a_sf_id, b_sf_id = k-block
            else umma_f8(tmem_d, adesc, bdesc, p.idesc, (kb | k) != 0);
          }
          umma_commit(empty_bar(stage));  // frees the smem slot once these MMAs retire
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(tfull_bar(as));      // accumulator complete -> epilogue
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue =================
    const int ew = warp - 4;  // TMEM lane quadrant (warp id % 4)
    int local = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++local) {
      int bz, mb, nb;
      tile_coords(tile, bz, mb, nb);
      const int as = local % C::ACC;
      const uint32_t aphase = (local / C::ACC) & 1;
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const int row = mb * BLOCK_M + ew * 32 + lane;
      const bool row_ok = row < p.m;
      const float dq = p.scale * (p.scale_a ? *p.scale_a : 1.f) * (p.scale_b ? *p.scale_b : 1.f);
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const int col0 = nb * BN + c * 32;
        if (col0 >= p.n) break;  // warp-uniform
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BN + c * 32, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        const int valid = min(32, p.n - col0);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] *= dq;           // per-tensor dequantisation scale (scale_a * scale_b)
        if (p.has_bias) {
          if (p.out_dtype == kBF16) {
            const __nv_bfloat16* b = (const __nv_bfloat16*)p.bias + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j) if (j < valid) v[j] += __bfloat162float(b[j]);
          } else if (p.out_dtype == kF16) {
            const __half* b = (const __half*)p.bias + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j) if (j < valid) v[j] += __half2float(b[j]);
          } else {
            const float* b = (const float*)p.bias + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j) if (j < valid) v[j] += b[j];
          }
        }
        if (p.act == 1) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
        } else if (p.act == 2) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (row_ok) {
          void* dptr = p.d;
          int64_t off = (int64_t)bz * p.stride_d + (int64_t)row * p.ldd + col0;
          if (p.out_dtype == kBF16) store_row_chunk((__nv_bfloat16*)dptr + off, v, valid, p.accumulate);
          else if (p.out_dtype == kF16) store_row_chunk((__half*)dptr + off, v, valid, p.accumulate);
          else store_row_chunk((float*)dptr + off, v, valid, p.accumulate);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------- host side
// 3-D byte map {k (contiguous), rows, batch}
static bool make_map8(CUtensorMap* out, const void* ptr, uint64_t k, uint64_t rows, uint64_t batch, uint64_t ld, uint64_t bstride, uint32_t box_rows) {
  cuuint64_t dims[3] = {k, rows, batch};
  cuuint64_t strides[2] = {ld, batch > 1 ? bstride : rows * ld};
  cuuint32_t box[3] = {(cuuint32_t)BLOCK_K, box_rows, 1};
  return encode_tiled(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, ptr, dims, strides, box, "fp8 gemm");
}

template <int BN, bool MX>
static int launch(const GemmFp8Args& g, cudaStream_t s) {
  using C = Cfg<BN, MX>;
  CUtensorMap ma, mb;
  const uint64_t batch = g.batch > 1 ? g.batch : 1;
  if (!make_map8(&ma, g.a, g.k, g.m, batch, g.lda, g.stride_a, BLOCK_M)) return 2;
  if (!make_map8(&mb, g.b, g.k, g.n, batch, g.ldb, g.stride_b, BN)) return 2;
  Params p;
  p.m = g.m; p.n = g.n; p.k = g.k; p.batch = (int)batch;
  p.d = g.d; p.bias = g.bias; p.ldd = g.ldd; p.stride_d = g.stride_d;
  p.in_dtype = 0; p.out_dtype = g.out_dtype;
  p.has_bias = g.bias ? 1 : 0;
  p.act = g.act;
  p.accumulate = 0;
  p.scale = g.scale;
  p.scale_a = g.scale_a_dev; p.scale_b = g.scale_b_dev;
  p.sfa = g.sfa; p.sfb = g.sfb;
  p.idesc = umma_idesc(g.a_e5m2 ? 1u : 0u, g.b_e5m2 ? 1u : 0u, false, false, BLOCK_M, BN, MX);   // E4M3 = 0, E5M2 = 1
  static bool attr_set = false;
  auto kern = gemm_fp8_kernel<BN, MX>;
  if (!attr_set) {
    B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  const int num_tiles = ((g.m + BLOCK_M - 1) / BLOCK_M) * ((g.n + BN - 1) / BN) * (int)batch;
  const int grid = num_tiles < sm_count() ? num_tiles : sm_count();
  kern<<<grid, kThreads, C::SMEM_BYTES, s>>>(ma, mb, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_last_error(__FILE__, __LINE__, cudaGetErrorString(e)); return 3; }
  return 0;
}

}  // namespace gemm8

int gemm_fp8_tcgen05(const GemmFp8Args& g, cudaStream_t s) {
  if (g.m <= 0 || g.n <= 0 || g.k <= 0 || g.k % 16 || g.lda % 16 || g.ldb % 16) return 1;   // TMA strides: multiples of 16 bytes
  if ((reinterpret_cast<uintptr_t>(g.a) | reinterpret_cast<uintptr_t>(g.b)) & 15) return 1;
  if (g.sfa || g.sfb) {
    // MX: whole 128 x 128 x 128 scale blocks only
    if (!g.sfa || !g.sfb || g.m % 128 || g.n % 128 || g.k % 128 || g.batch > 1) return 1;
    if ((reinterpret_cast<uintptr_t>(g.sfa) | reinterpret_cast<uintptr_t>(g.sfb)) & 15) return 1;
    return g.n % 256 == 0 ? gemm8::launch<256, true>(g, s) : gemm8::launch<128, true>(g, s);
  }
  if (g.n <= 128) return gemm8::launch<128, false>(g, s);
  return gemm8::launch<256, false>(g, s);
}

}  // namespace b200
