// 2-CTA (cta_group::2) variant of the persistent tcgen05 GEMM: a cluster of two CTAs (one TPC) computes one 256x256
// output tile.  Each CTA stages its own 128 rows of A and its own 128-column half of B, the leader CTA issues
// tcgen05.mma.cta_group::2 (UMMA M=256, N=256) which reads both CTAs' shared memory, and every CTA drains its own
// 128x256 accumulator half from its TMEM.  Versus the 1-CTA kernel this halves the B traffic through each SM's
// shared memory (96 -> 64 B/clk/SM at full MMA rate), which is what limits the long-K shapes.
//
// Barrier protocol (per pipeline stage s; leader = cluster rank 0):
//   full[s]   (leader only)  : 1 arrival (leader producer, expect_tx = bytes of BOTH CTAs) + complete_tx from the TMA
//                              loads of both CTAs (cp.async.bulk.tensor.cta_group::2 signals the leader's barrier)
//   empty[s]  (both CTAs)    : tcgen05.commit.cta_group::2 ... multicast -> each producer waits on its own copy
//   tfull[a]  (both CTAs)    : multicast commit after the last k-block -> each CTA's epilogue waits on its own copy
//   tempty[a] (leader only)  : 8 arrivals = 4 epilogue warps x 2 CTAs (the peer arrives remotely through mapa)
#include <cuda.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_ptx.cuh"
#include "include/b200_tcgen05_host.h"

namespace b200 {
namespace gemm2 {
using namespace ptx;

constexpr int BLOCK_M = 128;      // per CTA (cluster tile M = 256)
constexpr int BLOCK_N = 256;      // cluster tile N; each CTA stages BLOCK_N/2 columns of B
constexpr int HALF_N = BLOCK_N / 2;
constexpr int BLOCK_K = 64;
constexpr int UMMA_K = 16;
constexpr int kStages = 6;
constexpr int kThreads = 256;
constexpr int kAccStages = 2;
constexpr uint32_t A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;   // 16 KB
constexpr uint32_t B_STAGE_BYTES = HALF_N * BLOCK_K * 2;    // 16 KB
constexpr uint32_t STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr uint32_t TMEM_COLS = kAccStages * BLOCK_N;        // 512
// TMA-store epilogue: every epilogue warp stages [32 rows x 128 B] boxes (128B-swizzled) in two alternating 4 KB buffers
constexpr uint32_t STG_BOX_BYTES = 32 * 128;
constexpr uint32_t STG_OFF = kStages * STAGE_BYTES + 1024;                 // after the barrier page (1024-aligned)
constexpr uint32_t STG_BYTES = 4 * 2 * STG_BOX_BYTES;                      // 32 KB
constexpr uint32_t SMEM_BYTES = STG_OFF + STG_BYTES + 1024;                // + alignment slack = 231424 <= 232448 (227 KB)

struct DMaps { CUtensorMap m[8]; };   // TMA-store maps of the output: [0] = D, or one per reduce-scatter owner slot

struct Params {
  int tma_store;           // epilogue goes TMEM -> registers -> swizzled smem -> cp.async.bulk.tensor (UTMASTG), also to peer HBM;
                           // 0: registers -> global stores (output rows that are not 16-byte aligned)
  int m, n, k, batch;
  void* d;
  const void* bias;
  int64_t ldd, stride_d;
  int in_dtype, out_dtype;
  int has_bias, act, accumulate;
  uint32_t idesc;
  // grouped GEMM (MoE experts, see GemmArgs::grouped): 1 = rows grouped by expert (tile -> expert table), 2 = per-expert weight gradient
  int grouped;
  const int* tile_expert;
  const int* expert_k0;
  const int* expert_kb;
  int rs_world, rs_rows;   // fused reduce-scatter push (see GemmArgs)
  void* rs_dst[8];
  // fused all-gather -> GEMM (see GemmArgs): warp 3 of every CTA pulls the peers' row shards into the local A buffer
  int ag_world, ag_rank, ag_rows, ag_chunks;
  const char* ag_src[8];
  char* ag_dst;
  uint32_t* ag_flags;
  uint32_t* ag_pad[8];
  uint32_t ag_epoch;
};

constexpr int kAgChunkBytes = 16384;
constexpr int kAgReadySlot = 4, kAgDoneSlot = 5, kPadRanks = 8;

// the all-gather's cross-rank waits; a peer that stalls traps with a message naming this protocol
__device__ __forceinline__ void ag_wait(const uint32_t* p, uint32_t epoch, const char* what) {
  spin_sys_ge(p, epoch, "b200 gemm2 all-gather: timeout waiting for %s\n", what);
}
// bounded spin on a gathered row block's chunk counter (bumped by the copy warps of this GPU)
__device__ __forceinline__ void spin_gpu_ge(const uint32_t* p, uint32_t target) {
  const uint64_t t0 = globaltimer_ns();
  while (ld_acquire_gpu_u32(p) < target) {
    if (globaltimer_ns() - t0 > kSpinTimeoutNs) { printf("b200 gemm2 all-gather: timeout waiting for a gathered row block\n"); __trap(); }
  }
}

// Copy role of the fused all-gather: chunk g of the remote data is handled by warp (g % #CTAs); finished chunks bump the
// counter of their 128-row block, which the TMA producers poll before loading A rows of that block.
__device__ __forceinline__ void ag_copy_role(const Params& p, int lane) {
  const int nwarps = gridDim.x, wid = blockIdx.x;
  const int blocks_per_rank = p.ag_rows / BLOCK_M;
  const int64_t block_bytes = (int64_t)BLOCK_M * p.k * 2;
  const int64_t per_src = (int64_t)blocks_per_rank * p.ag_chunks;
  const int64_t total = (int64_t)(p.ag_world - 1) * per_src;
  uint32_t* my_pad = p.ag_pad[p.ag_rank];
  if (wid == 0 && lane < p.ag_world && lane != p.ag_rank)        // my shard is in place (stream order before this kernel)
    st_release_sys_u32(p.ag_pad[lane] + kAgReadySlot * kPadRanks + p.ag_rank, p.ag_epoch);
  int cur_src = -1;
  for (int64_t g = wid; g < total; g += nwarps) {
    const int pr = (int)(g / per_src) + 1;
    const int src = (p.ag_rank + pr) % p.ag_world;
    const int64_t rem = g - (int64_t)(pr - 1) * per_src;
    const int blk_in = (int)(rem / p.ag_chunks), ch = (int)(rem % p.ag_chunks);
    if (src != cur_src) {
      if (lane == 0) ag_wait(my_pad + kAgReadySlot * kPadRanks + src, p.ag_epoch, "a peer shard");
      __syncwarp();
      cur_src = src;
    }
    const uint4* sp = reinterpret_cast<const uint4*>(p.ag_src[src] + blk_in * block_bytes + (int64_t)ch * kAgChunkBytes);
    uint4* dp = reinterpret_cast<uint4*>(p.ag_dst + ((int64_t)src * blocks_per_rank + blk_in) * block_bytes + (int64_t)ch * kAgChunkBytes);
#pragma unroll
    for (int it = 0; it < kAgChunkBytes / 16 / 32 / 8; ++it) {
      uint4 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = sp[(it * 8 + j) * 32 + lane];     // 8 independent 16 B loads over NVLink in flight
#pragma unroll
      for (int j = 0; j < 8; ++j) dp[(it * 8 + j) * 32 + lane] = v[j];
    }
    __syncwarp();
    if (lane == 0) {
      __threadfence();
      atomicAdd(p.ag_flags + src * blocks_per_rank + blk_in, 1u);
    }
  }
  __syncwarp();
  if (lane == 0) {
    __threadfence();
    const int done_idx = p.ag_world * blocks_per_rank;
    if (atomicAdd(p.ag_flags + done_idx, 1u) == (uint32_t)nwarps - 1) {    // every pull of this rank has completed
      for (int r = 0; r < p.ag_world; ++r)
        if (r != p.ag_rank) st_release_sys_u32(p.ag_pad[r] + kAgDoneSlot * kPadRanks + p.ag_rank, p.ag_epoch);
    }
  }
  if (wid == 0 && lane < p.ag_world && lane != p.ag_rank)        // peers finished reading my shard: it may be reused after exit
    ag_wait(my_pad + kAgDoneSlot * kPadRanks + lane, p.ag_epoch, "a peer to finish reading");
}

template <bool A_MN, bool B_MN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ DMaps dmaps,
             const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + kStages * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStages + kAccStages + s); };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_gen + kStages * STAGE_BYTES + 8 * (2 * kStages + 2 * kAccStages));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int num_m = (p.m + 2 * BLOCK_M - 1) / (2 * BLOCK_M), num_n = (p.n + BLOCK_N - 1) / BLOCK_N;
  const int tiles_per_batch = num_m * num_n;
  const int num_tiles = tiles_per_batch * p.batch;
  const int num_kb = (p.k + BLOCK_K - 1) / BLOCK_K;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < kAccStages; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 8); }
    fence_barrier_init();
    fence_proxy_async();
  }
  cluster_sync();  // barriers of both CTAs are initialised before any remote arrive / TMA completion can target them
  if (warp == 2) {
    tmem_alloc<2>(smem_u32((const void*)tmem_ptr_smem), TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  auto tile_coords = [&](int tile, int& bz, int& mb, int& nb) {
    bz = tile / tiles_per_batch;
    const int t = tile - bz * tiles_per_batch;
    constexpr int GROUP_M = 4;  // 4 x 256 rows
    const int in_group = GROUP_M * num_n;
    const int g = t / in_group;
    const int first_m = g * GROUP_M;
    const int gsz = min(num_m - first_m, GROUP_M);
    const int r = t - g * in_group;
    mb = first_m + r % gsz;
    nb = r / gsz;
    if (p.ag_world > 1) {   // fused all-gather: start with the row blocks that are already local
      mb += p.ag_rank * (p.ag_rows / (2 * BLOCK_M));
      if (mb >= num_m) mb -= num_m;
    }
  };

  // grouped modes: which batch index each operand uses for this tile, the reduction range, and whether the tile exists at all
  auto tile_group = [&](int bz, int mb, int& za, int& zb, int& zd, int& kbeg, int& nkb) -> bool {
    za = zb = zd = bz; kbeg = 0; nkb = num_kb;
    if (p.grouped == 1) {
      const int e = p.tile_expert[mb];
      if (e < 0) return false;           // padding tile beyond the last expert's rows
      za = 0; zb = e; zd = 0;
    } else if (p.grouped == 2) {
      nkb = p.expert_kb[bz];
      if (nkb <= 0) return false;        // expert received no rows: its weight gradient gets nothing added
      kbeg = p.expert_k0[bz];
      za = 0; zb = 0; zd = bz;
    }
    return true;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ================= TMA producer (both CTAs: own A rows, own half of B) =================
      int stage = 0;
      uint32_t phase = 0;
      const uint64_t hint = 0x1000000000000000ull;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        int bz, mb, nb;
        tile_coords(tile, bz, mb, nb);
        int za, zb, zd, kbeg, nkb;
        if (!tile_group(bz, mb, za, zb, zd, kbeg, nkb)) continue;
        const int m0 = mb * 2 * BLOCK_M + (int)cta_rank * BLOCK_M;
        const int n0 = nb * BLOCK_N + (int)cta_rank * HALF_N;
        if (p.ag_world > 1) {
          const int blk = m0 / BLOCK_M;
          if (blk / (p.ag_rows / BLOCK_M) != p.ag_rank) {        // rows owned by a peer: wait until the copy warps landed them
            spin_gpu_ge(p.ag_flags + blk, (uint32_t)p.ag_chunks);
            asm volatile("fence.proxy.async;" ::: "memory");     // generic-proxy writes (other SMs) -> TMA (async proxy) reads
          }
        }
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
          if (leader) mbar_expect_tx(full_bar(stage), 2 * STAGE_BYTES);
          const int k0 = kbeg + kb * BLOCK_K;
          if constexpr (!A_MN) {
            tma_load_3d_2sm(sa, &map_a, full_bar(stage), k0, m0, za, hint);
          } else {
#pragma unroll
            for (int i = 0; i < BLOCK_M / 64; ++i) tma_load_3d_2sm(sa + i * 8192, &map_a, full_bar(stage), m0 + i * 64, k0, za, hint);
          }
          if constexpr (!B_MN) {
            tma_load_3d_2sm(sb, &map_b, full_bar(stage), k0, n0, zb, hint);
          } else {
#pragma unroll
            for (int i = 0; i < HALF_N / 64; ++i) tma_load_3d_2sm(sb + i * 8192, &map_b, full_bar(stage), n0 + i * 64, k0, zb, hint);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      // ================= MMA issuer (leader CTA only) =================
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        int nkb = num_kb;
        if (p.grouped) {
          int bz, mb, nb, za, zb, zd, kbeg;
          tile_coords(tile, bz, mb, nb);
          if (!tile_group(bz, mb, za, zb, zd, kbeg, nkb)) continue;
        }
        const int as = local & 1;
        const uint32_t aphase = (local >> 1) & 1;
        ++local;
        mbar_wait(tempty_bar(as), aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BLOCK_N;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = A_MN ? make_smem_desc(sa + k * 2048, 8192, 1024) : make_smem_desc(sa + k * 32, 16, 1024);
            const uint64_t bdesc = B_MN ? make_smem_desc(sb + k * 2048, 8192, 1024) : make_smem_desc(sb + k * 32, 16, 1024);
            umma_f16_2sm(tmem_d, adesc, bdesc, p.idesc, (kb | k) != 0);
          }
          umma_commit_2sm(empty_bar(stage));
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(tfull_bar(as));
      }
    }
  } else if (warp == 3) {
    if (p.ag_world > 1) ag_copy_role(p, lane);
  } else if (warp >= 4) {
    // ================= epilogue (both CTAs: own 128 rows x 256 columns) =================
    const int ew = warp - 4;
    int local = 0;
    int tma_buf = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
      int bz, mb, nb;
      tile_coords(tile, bz, mb, nb);
      {
        int za, zb, zd, kbeg, nkb;
        if (!tile_group(bz, mb, za, zb, zd, kbeg, nkb)) continue;
        bz = zd;                            // batch index of the OUTPUT for this tile
      }
      const int as = local & 1;
      const uint32_t aphase = (local >> 1) & 1;
      ++local;
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const int row = mb * 2 * BLOCK_M + (int)cta_rank * BLOCK_M + ew * 32 + lane;
      const bool row_ok = row < p.m;
      if (p.tma_store) {
        // ---- TMA-store epilogue: [32 rows x 128 B] boxes through 128B-swizzled smem, one cp.async.bulk.tensor per box ----
        const int row0 = mb * 2 * BLOCK_M + (int)cta_rank * BLOCK_M + ew * 32;      // first row of this warp's 32-row strip
        const int owner = p.rs_world > 1 ? row0 / p.rs_rows : 0;
        const int row_rel = p.rs_world > 1 ? row0 - owner * p.rs_rows : row0;
        const int cpb = p.out_dtype == kF32 ? 32 : 64;                              // columns per 128-byte box row
        const uint32_t stg = smem_base + STG_OFF + (uint32_t)ew * 2 * STG_BOX_BYTES;
#pragma unroll 1
        for (int c = 0; c < BLOCK_N / cpb; ++c) {
          const int col0 = nb * BLOCK_N + c * cpb;
          if (col0 >= p.n || row0 >= p.m) break;
          if (lane == 0) bulk_wait_read<1>();       // the box stored two iterations ago has been read out of this buffer
          __syncwarp();
          const uint32_t dst = stg + (uint32_t)tma_buf * STG_BOX_BYTES + (uint32_t)lane * 128;
          const uint32_t sw = (uint32_t)(lane & 7);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (h * 32 >= cpb) break;
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BLOCK_N + c * cpb + h * 32, r);
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
            if (p.has_bias) {
              const int cb = col0 + h * 32;
              if (p.in_dtype == kBF16) {
                const __nv_bfloat16* b = (const __nv_bfloat16*)p.bias + cb;
#pragma unroll
                for (int j = 0; j < 32; ++j) if (cb + j < p.n) v[j] += __bfloat162float(b[j]);
              } else {
                const __half* b = (const __half*)p.bias + cb;
#pragma unroll
                for (int j = 0; j < 32; ++j) if (cb + j < p.n) v[j] += __half2float(b[j]);
              }
            }
            if (p.act == 1) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
            } else if (p.act == 2) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (p.out_dtype == kF32) {
#pragma unroll
              for (int q = 0; q < 8; ++q)
                st_shared_v4(dst + (((uint32_t)q ^ sw) << 4), __float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]),
                             __float_as_uint(v[4 * q + 2]), __float_as_uint(v[4 * q + 3]));
            } else if (p.out_dtype == kBF16) {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                st_shared_v4(dst + (((uint32_t)(h * 4 + q) ^ sw) << 4), pack2<__nv_bfloat16>(v[8 * q], v[8 * q + 1]),
                             pack2<__nv_bfloat16>(v[8 * q + 2], v[8 * q + 3]), pack2<__nv_bfloat16>(v[8 * q + 4], v[8 * q + 5]),
                             pack2<__nv_bfloat16>(v[8 * q + 6], v[8 * q + 7]));
            } else {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                st_shared_v4(dst + (((uint32_t)(h * 4 + q) ^ sw) << 4), pack2<__half>(v[8 * q], v[8 * q + 1]), pack2<__half>(v[8 * q + 2], v[8 * q + 3]),
                             pack2<__half>(v[8 * q + 4], v[8 * q + 5]), pack2<__half>(v[8 * q + 6], v[8 * q + 7]));
            }
          }
          fence_proxy_async();                      // generic-proxy smem writes -> visible to the TMA (async proxy)
          __syncwarp();
          if (lane == 0) {
            if (p.accumulate) tma_reduce_add_3d(&dmaps.m[owner], stg + (uint32_t)tma_buf * STG_BOX_BYTES, col0, row_rel, bz);
            else tma_store_3d(&dmaps.m[owner], stg + (uint32_t)tma_buf * STG_BOX_BYTES, col0, row_rel, bz);
            bulk_commit();
          }
          tma_buf ^= 1;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty_bar(as), 0);
        continue;
      }
#pragma unroll 1
      for (int c = 0; c < BLOCK_N / 32; ++c) {
        const int col0 = nb * BLOCK_N + c * 32;
        if (col0 >= p.n) break;
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BLOCK_N + c * 32, r);
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        const int valid = min(32, p.n - col0);
        if (p.has_bias) {
          if (p.in_dtype == kBF16) {
            const __nv_bfloat16* b = (const __nv_bfloat16*)p.bias + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j) if (j < valid) v[j] += __bfloat162float(b[j]);
          } else {
            const __half* b = (const __half*)p.bias + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j) if (j < valid) v[j] += __half2float(b[j]);
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
      if (lane == 0) mbar_arrive_cluster(tempty_bar(as), 0);  // leader's barrier counts both CTAs' epilogue warps
    }
    if (p.tma_store && lane == 0) bulk_wait<0>();    // every box has been written before the CTA may exit
  }

  tc_fence_before();
  cluster_sync();  // peer smem / TMEM stay valid until every MMA and remote arrive has retired
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2>(tmem_base, TMEM_COLS);
  }
}

template <bool A_MN, bool B_MN>
static int launch(const GemmArgs& g, cudaStream_t s) {
  CUtensorMap ma, mb;
  uint64_t batch = g.batch > 1 ? g.batch : 1;
  uint64_t batch_a = batch, batch_b = batch;
  if (g.grouped == 1) { batch_a = 1; batch_b = g.groups; batch = 1; }             // rows grouped by expert: B = stacked expert weights
  else if (g.grouped == 2) { batch_a = 1; batch_b = 1; batch = g.groups; }        // per-expert weight gradient: D = stacked [E, m, n]
  bool ok;
  if (!A_MN) ok = gemm::make_map(&ma, g.a, g.k, g.m, batch_a, g.lda, g.stride_a, BLOCK_K, BLOCK_M, g.dtype);
  else       ok = gemm::make_map(&ma, g.a, g.m, g.k, batch_a, g.lda, g.stride_a, 64, BLOCK_K, g.dtype);
  if (!ok) return 2;
  if (!B_MN) ok = gemm::make_map(&mb, g.b, g.k, g.n, batch_b, g.ldb, g.stride_b, BLOCK_K, HALF_N, g.dtype);
  else       ok = gemm::make_map(&mb, g.b, g.n, g.k, batch_b, g.ldb, g.stride_b, 64, BLOCK_K, g.dtype);
  if (!ok) return 2;
  Params p;
  p.m = g.m; p.n = g.n; p.k = g.k; p.batch = (int)batch;
  p.d = g.d; p.bias = g.bias; p.ldd = g.ldd; p.stride_d = g.stride_d;
  p.in_dtype = g.dtype; p.out_dtype = g.out_dtype;
  p.has_bias = (g.epilogue >= 1 && g.epilogue <= 3 && g.bias) ? 1 : 0;
  p.act = g.epilogue == 2 ? 1 : (g.epilogue == 3 ? 2 : 0);
  p.accumulate = g.epilogue == 4 ? 1 : 0;
  p.grouped = g.grouped; p.tile_expert = g.tile_expert; p.expert_k0 = g.expert_k0; p.expert_kb = g.expert_kb;
  p.rs_world = g.rs_world > 1 ? g.rs_world : 0;
  p.rs_rows = g.rs_rows;
  for (int i = 0; i < 8; ++i) p.rs_dst[i] = g.rs_dst[i];
  if (p.rs_world) p.ldd = g.n;
  p.ag_world = 0;
  if (g.ag_world > 1) {
    // preconditions of the fused all-gather (checked by the caller as well): A is K-major with lda == k, whole 256-row tiles per rank
    if (A_MN || g.lda != g.k || g.ag_rows % (2 * BLOCK_M) || g.m != g.ag_world * g.ag_rows || batch != 1 ||
        ((int64_t)BLOCK_M * g.k * 2) % kAgChunkBytes) {
      set_last_error(__FILE__, __LINE__, "gemm_tcgen05_2cta: unsupported shape for the fused all-gather");
      return 4;
    }
    p.ag_world = g.ag_world; p.ag_rank = g.ag_rank; p.ag_rows = g.ag_rows;
    p.ag_chunks = (int)(((int64_t)BLOCK_M * g.k * 2) / kAgChunkBytes);
    for (int i = 0; i < 8; ++i) { p.ag_src[i] = (const char*)g.ag_src[i]; p.ag_pad[i] = (uint32_t*)g.ag_pad[i]; }
    p.ag_dst = (char*)const_cast<void*>(g.a);
    p.ag_flags = (uint32_t*)g.ag_flags;
    p.ag_epoch = g.ag_epoch;
  }
  // TMA-store epilogue whenever the output rows are 16-byte aligned; accumulate (D += AB, the fused weight-gradient path) becomes a
  // TMA reduce-add (UTMAREDG): the addition happens in L2 and D is never read by the SMs
  DMaps dm;
  memset(&dm, 0, sizeof(dm));
  {
    const int es = g.out_dtype == kF32 ? 4 : 2;
    const uint32_t cpb = 128 / es;
    bool ok2 = true;
    if (p.rs_world) {
      ok2 = (g.n * es) % 16 == 0 && g.rs_rows % 32 == 0;
      for (int r = 0; r < p.rs_world && ok2; ++r)
        ok2 = ((uintptr_t)g.rs_dst[r] % 16 == 0) && gemm::make_map(&dm.m[r], g.rs_dst[r], g.n, g.rs_rows, 1, g.n, 0, cpb, 32, g.out_dtype);
    } else {
      ok2 = (g.ldd * es) % 16 == 0 && ((uintptr_t)g.d % 16 == 0) && (batch == 1 || (g.stride_d * es) % 16 == 0) &&
            gemm::make_map(&dm.m[0], g.d, g.n, g.m, batch, g.ldd, g.stride_d, cpb, 32, g.out_dtype);
    }
    if (!ok2) take_last_error();     // an odd leading dimension just keeps the register-store epilogue
    p.tma_store = ok2 ? 1 : 0;
  }
  const uint32_t f = g.dtype == kBF16 ? 1u : 0u;
  p.idesc = umma_idesc(f, f, A_MN, B_MN, 2 * BLOCK_M, BLOCK_N, false);   // UMMA M = 256 across the CTA pair
  static bool attr_set = false;
  auto kern = gemm2_kernel<A_MN, B_MN>;
  if (!attr_set) {
    B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_set = true;
  }
  const int num_tiles = ((g.m + 2 * BLOCK_M - 1) / (2 * BLOCK_M)) * ((g.n + BLOCK_N - 1) / BLOCK_N) * (int)batch;
  // B200_GEMM_RESERVE_SMS=<n>: keep n SMs out of every persistent GEMM grid so that concurrently launched collective kernels are resident
  // unconditionally (docs/race_detection.md, "cross-rank progress"); default 0
  static const int reserve = [] { const char* e = getenv("B200_GEMM_RESERVE_SMS"); const int v = e ? atoi(e) : 0; return v < 0 ? 0 : v; }();
  const int usable = sm_count() - reserve;
  const int max_clusters = usable >= 2 ? usable / 2 : 1;
  const int clusters = num_tiles < max_clusters ? num_tiles : max_clusters;
  kern<<<clusters * 2, kThreads, SMEM_BYTES, s>>>(ma, mb, dm, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_last_error(__FILE__, __LINE__, cudaGetErrorString(e)); return 3; }
  return 0;
}

}  // namespace gemm2

int gemm_tcgen05_2cta(const GemmArgs& g, cudaStream_t s) {
  if (g.a_is_km) return g.b_is_nk ? gemm2::launch<true, false>(g, s) : gemm2::launch<true, true>(g, s);
  return g.b_is_nk ? gemm2::launch<false, false>(g, s) : gemm2::launch<false, true>(g, s);
}

}  // namespace b200
