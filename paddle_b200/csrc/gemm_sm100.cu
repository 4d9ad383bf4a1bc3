// Persistent warp-specialised GEMM for sm_100a: TMA (cp.async.bulk.tensor) -> 128B-swizzled smem ring ->
// tcgen05.mma (kind::f16, fp32 accumulate in TMEM, double-buffered accumulators) -> tcgen05.ld epilogue with fused
// bias / activation / accumulate.  Hand-written PTX; no CUTLASS.
//
// Parity (behaviour): phi MatmulKernel / fused_gemm_epilogue (paddle/phi/kernels/fusion/gpu/fused_gemm_epilogue_kernel.cu)
// which call cuBLASLt in the reference.
//
// Operand layouts (all four combinations, selected by descriptor "major" bits, no transposition copies):
//   A: [M,K] row-major (K-major)  or  [K,M] row-major (MN-major, "a_is_km")  -> needed for dW = X^T dY
//   B: [N,K] row-major (K-major, "b_is_nk")  or  [K,N] row-major (MN-major)  -> paddle Linear weight is [in,out]
// Warp roles (256 threads): w0 TMA producer | w1 MMA issuer | w2 TMEM allocator | w4..w7 epilogue (TMEM lane quadrants).
#include <cuda.h>
#include <cstdio>
#include <mutex>
#include <unordered_map>

#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_ptx.cuh"
#include "include/b200_tcgen05_host.h"

namespace b200 {
namespace gemm {
using namespace ptx;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;   // 64 x 2B = 128B = one swizzle atom row
constexpr int UMMA_K = 16;
constexpr int kStages = 4;
constexpr int kThreads = 256;
constexpr int kAccStages = 2;
constexpr uint32_t A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB

template <int BN> struct Cfg {
  static constexpr uint32_t B_STAGE_BYTES = BN * BLOCK_K * 2;
  static constexpr uint32_t STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr uint32_t TMEM_COLS = kAccStages * BN;  // 512 / 256 / 128: powers of two >= 32
  static constexpr uint32_t SMEM_BYTES = kStages * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

struct Params {
  int m, n, k, batch;
  void* d;
  const void* bias;
  int64_t ldd, stride_d;
  int in_dtype, out_dtype;
  int has_bias, act, accumulate;
  uint32_t idesc;
  int rs_world, rs_rows;   // fused reduce-scatter push (see GemmArgs)
  void* rs_dst[8];
};

template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const Params p) {
  using C = Cfg<BN>;
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
          mbar_expect_tx(full_bar(stage), C::STAGE_BYTES);
          const int k0 = kb * BLOCK_K;
          if constexpr (!A_MN) {
            tma_load_3d(sa, &map_a, full_bar(stage), k0, m0, bz, hint);  // box {64 k, 128 m}
          } else {
#pragma unroll
            for (int i = 0; i < BLOCK_M / 64; ++i)                      // box {64 m, 64 k}
              tma_load_3d(sa + i * 8192, &map_a, full_bar(stage), m0 + i * 64, k0, bz, hint);
          }
          if constexpr (!B_MN) {
            tma_load_3d(sb, &map_b, full_bar(stage), k0, n0, bz, hint);  // box {64 k, BN n}
          } else {
#pragma unroll
            for (int i = 0; i < BN / 64; ++i)                           // box {64 n, 64 k}
              tma_load_3d(sb + i * 8192, &map_b, full_bar(stage), n0 + i * 64, k0, bz, hint);
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
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++local) {
        const int as = local & 1;
        const uint32_t aphase = (local >> 1) & 1;
        mbar_wait(tempty_bar(as), aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // K-major: advance 16 elem = 32 B inside the swizzle row; MN-major: advance 16 k-rows = 2048 B
            const uint64_t adesc = A_MN ? make_smem_desc(sa + k * 2048, 8192, 1024) : make_smem_desc(sa + k * 32, 16, 1024);
            const uint64_t bdesc = B_MN ? make_smem_desc(sb + k * 2048, 8192, 1024) : make_smem_desc(sb + k * 32, 16, 1024);
            umma_f16(tmem_d, adesc, bdesc, p.idesc, (kb | k) != 0);
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
      const int as = local & 1;
      const uint32_t aphase = (local >> 1) & 1;
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const int row = mb * BLOCK_M + ew * 32 + lane;
      const bool row_ok = row < p.m;
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
        if (p.has_bias) {
          if (p.in_dtype == kBF16) {
            const __nv_bfloat16* b = (const __nv_bfloat16*)p.bias + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j) if (j < valid) v[j] += __bfloat162float(b[j]);
          } else if (p.in_dtype == kF16) {
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
          if (p.rs_world > 1) {   // fused reduce-scatter: push this row's partial into its owner's staging slot (peer HBM)
            const int owner = row / p.rs_rows;
            dptr = p.rs_dst[owner];
            off = (int64_t)(row - owner * p.rs_rows) * p.ldd + col0;
          }
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
struct MapKey {
  const void* ptr; uint64_t inner, rows, batch, ld, bstride; uint32_t box_inner, box_rows; int dtype;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && inner == o.inner && rows == o.rows && batch == o.batch && ld == o.ld && bstride == o.bstride &&
           box_inner == o.box_inner && box_rows == o.box_rows && dtype == o.dtype;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = std::hash<const void*>()(k.ptr);
    auto mix = [&](uint64_t v) { h ^= std::hash<uint64_t>()(v) + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
    mix(k.inner); mix(k.rows); mix(k.batch); mix(k.ld); mix(k.bstride); mix(k.box_inner); mix(k.box_rows); mix((uint64_t)k.dtype);
    return h;
  }
};

bool make_map(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t rows, uint64_t batch, uint64_t ld, uint64_t bstride,
              uint32_t box_inner, uint32_t box_rows, int dtype) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  MapKey key{ptr, inner, rows, batch, ld, bstride, box_inner, box_rows, dtype};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return true; }
  }
  cuuint64_t dims[3] = {inner, rows, batch};
  const uint64_t es = dtype == kF32 ? 4 : 2;
  cuuint64_t strides[2] = {ld * es, (batch > 1 ? bstride : rows * ld) * es};
  cuuint32_t box[3] = {box_inner, box_rows, 1};
  const CUtensorMapDataType type =
      dtype == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : (dtype == kF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
  if (!encode_tiled(out, type, 3, ptr, dims, strides, box, "gemm")) return false;
  std::lock_guard<std::mutex> g(mu);
  if (cache.size() > 8192) cache.clear();
  cache.emplace(key, *out);
  return true;
}

template <int BN, bool A_MN, bool B_MN>
static int launch(const GemmArgs& g, cudaStream_t s) {
  using C = Cfg<BN>;
  CUtensorMap ma, mb;
  const uint64_t batch = g.batch > 1 ? g.batch : 1;
  bool ok;
  if (!A_MN) ok = make_map(&ma, g.a, g.k, g.m, batch, g.lda, g.stride_a, BLOCK_K, BLOCK_M, g.dtype);
  else       ok = make_map(&ma, g.a, g.m, g.k, batch, g.lda, g.stride_a, 64, BLOCK_K, g.dtype);
  if (!ok) return 2;
  if (!B_MN) ok = make_map(&mb, g.b, g.k, g.n, batch, g.ldb, g.stride_b, BLOCK_K, BN, g.dtype);
  else       ok = make_map(&mb, g.b, g.n, g.k, batch, g.ldb, g.stride_b, 64, BLOCK_K, g.dtype);
  if (!ok) return 2;
  Params p;
  p.m = g.m; p.n = g.n; p.k = g.k; p.batch = (int)batch;
  p.d = g.d; p.bias = g.bias; p.ldd = g.ldd; p.stride_d = g.stride_d;
  p.in_dtype = g.dtype; p.out_dtype = g.out_dtype;
  p.has_bias = (g.epilogue >= 1 && g.epilogue <= 3 && g.bias) ? 1 : 0;
  p.act = g.epilogue == 2 ? 1 : (g.epilogue == 3 ? 2 : 0);
  p.accumulate = g.epilogue == 4 ? 1 : 0;
  p.rs_world = g.rs_world > 1 ? g.rs_world : 0;
  p.rs_rows = g.rs_rows;
  for (int i = 0; i < 8; ++i) p.rs_dst[i] = g.rs_dst[i];
  if (p.rs_world) p.ldd = g.n;
  const uint32_t f = g.dtype == kBF16 ? 1u : 0u;
  p.idesc = umma_idesc(f, f, A_MN, B_MN, BLOCK_M, BN, false);
  static bool attr_set = false;
  auto kern = gemm_kernel<BN, A_MN, B_MN>;
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

template <int BN>
static int launch_layout(const GemmArgs& g, cudaStream_t s) {
  if (g.a_is_km) return g.b_is_nk ? launch<BN, true, false>(g, s) : launch<BN, true, true>(g, s);
  return g.b_is_nk ? launch<BN, false, false>(g, s) : launch<BN, false, true>(g, s);
}

}  // namespace gemm

int gemm_tcgen05_supported(int m, int n, int k, int64_t lda, int64_t ldb, int64_t ldd, int a_is_km, int b_is_nk) {
  if (m <= 0 || n <= 0 || k <= 0) return 0;
  if (lda % 8 || ldb % 8) return 0;            // TMA global strides must be multiples of 16 bytes
  // inner (contiguous) extents must also keep 16-byte granularity for the tensor map
  const int a_inner = a_is_km ? m : k, b_inner = b_is_nk ? k : n;
  if (a_inner % 8 || b_inner % 8) return 0;
  (void)ldd;
  return 1;
}

int gemm_tcgen05(const GemmArgs& g, cudaStream_t s) {
  if (!gemm_tcgen05_supported(g.m, g.n, g.k, g.lda, g.ldb, g.ldd, g.a_is_km, g.b_is_nk)) return 1;
  if ((reinterpret_cast<uintptr_t>(g.a) & 15) || (reinterpret_cast<uintptr_t>(g.b) & 15)) return 1;
  if (g.dtype != kBF16 && g.dtype != kF16) return 1;
  if (g.ag_world > 1) return gemm_tcgen05_2cta(g, s);   // the fused all-gather lives in the CTA-pair kernel only
  // large problems: CTA-pair kernel (cta_group::2, 256x256 cluster tile)
  if (g.m >= 256 && g.n >= 256) return gemm_tcgen05_2cta(g, s);
  // tile-N choice: widest tile that keeps the last wave reasonably full
  const int sms = sm_count();
  auto waves_eff = [&](int bn) {
    const int64_t tiles = (int64_t)((g.m + 127) / 128) * ((g.n + bn - 1) / bn) * (g.batch > 1 ? g.batch : 1);
    const int64_t waves = (tiles + sms - 1) / sms;
    return (double)tiles / (double)(waves * sms);
  };
  int bn = 256;
  if (g.n <= 64) bn = 64;
  else if (g.n <= 128) bn = 128;
  else if (waves_eff(256) < 0.75 && waves_eff(128) > waves_eff(256) + 0.08) bn = 128;
  if (bn == 256) return gemm::launch_layout<256>(g, s);
  if (bn == 128) return gemm::launch_layout<128>(g, s);
  return gemm::launch_layout<64>(g, s);
}

}  // namespace b200
