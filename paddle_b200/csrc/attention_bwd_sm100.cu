// Flash-attention backward for sm_100a (head_dim 128, bf16/fp16), tcgen05 + TMA.
//
// One CTA owns a 128-key K/V tile of one (batch, kv head) and walks the query tiles that can see it (and, under GQA, every
// query head of the group).  Per query tile five 128x128x128 tensor-core GEMMs:
//   S   = Q K^T          dP  = dO V^T                      (TMEM, lane = query row)
//   dV += P^T dO         dK += dS^T Q                      (TMEM accumulators, lane = key row, live across the whole loop)
//   dQ^T = K^T dS^T                                        (TMEM, lane = head dim; reduced into fp32 dQ with coalesced atomics)
// P and dS are produced by the 128 softmax threads (thread = query row) from S, dP, the forward's logsumexp and
// delta = rowsum(dO * O), and are written ONCE to shared memory in the 128B-swizzled [key-half][query row] layout that
// serves both as MN-major A operand (P^T, dS^T) and as K-major B operand (dS^T of the dQ GEMM) by choice of descriptor
// strides; the K tile is likewise consumed K-major (S) and MN-major (dQ^T) from one copy.
//
// Parity (behaviour): flash_attn_grad (paddle/phi/kernels/gpu/flash_attn_grad_kernel.cu -> flash-attention library).
// Warps 0-7: softmax / dQ reduction / epilogue (two warpgroups, one 64-column half each), warp 8: TMA producer,
// warp 9: TMEM alloc + MMA issuer.
// TMEM columns: [0,128) S then dQ^T, [128,256) dP, [256,384) dV, [384,512) dK.
#include <cuda.h>
#include <cstdio>

#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_ptx.cuh"
#include "include/b200_tcgen05_host.h"

namespace b200 {
namespace attn_bwd {
using namespace ptx;

constexpr int BM = 128, BN = 128, HD = 128;
constexpr int kThreads = 320;   // warps 0-7: softmax / dQ / epilogue (2 warpgroups), warp 8: TMA producer, warp 9: TMEM alloc + MMA issuer
constexpr uint32_t TILE_BYTES = 128 * 128 * 2;
constexpr uint32_t HALF_BYTES = TILE_BYTES / 2;
constexpr uint32_t SMEM_BYTES = 6 * TILE_BYTES + 1024 + 256;
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t S_COL = 0, DP_COL = 128, DV_COL = 256, DK_COL = 384;


// Operand descriptors for one 128x128 bf16 tile stored as two 64-wide halves [half][row 0..127][128 B swizzled]:
//   K-major use   (rows = M or N index, inner = K):   K step k (16 elems) inside half kb -> +kb*HALF + k*32,  LBO 16, SBO 1024
//   MN-major use  (rows = K index, inner = M or N):   K step k (16 rows)                 -> +k*2048,         LBO HALF (next 64 M/N), SBO 1024
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t tile, int kb, int k) { return make_smem_desc(tile + kb * HALF_BYTES + k * 32, 16, 1024); }
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t tile, int kk) { return make_smem_desc(tile + kk * 2048, HALF_BYTES, 1024); }

struct Params {
  int b, sq, sk, h, hk;
  float scale, scale_log2;
  int causal, causal_off;
  const float* lse;      // [B,H,Sq] natural log
  const float* delta;    // [B,H,Sq]
  float* dq;             // fp32 [B,Sq,H,D] (zero-initialised; reduced with atomics)
  void* dk;              // [B,Sk,Hk,D] with element strides (dkv_sb, dkv_ss, dkv_sh): may be slices of a packed dQKV tensor
  void* dv;
  int64_t dkv_sb, dkv_ss, dkv_sh;
  int64_t dq_sb, dq_ss, dq_sh;   // element strides of the fp32 dQ accumulator [B,Sq,H,D] (may be laid out seq-major)
  uint32_t idesc_kk;     // A K-major, B K-major   (S, dP)
  uint32_t idesc_mm;     // A MN-major, B MN-major (dV, dK)
  uint32_t idesc_mk;     // A MN-major, B K-major  (dQ^T)
  const int4* colmask;   // [b, mask_heads, sk] hidden row ranges per key column (see AttnArgs::colmask); nullptr: none
  int mask_heads;
  int* dq_sem;           // deterministic dQ: turn counter per (batch, head, query tile); nullptr = reduce in arrival order
};

template <typename T, bool MASKED>
__global__ void __launch_bounds__(kThreads, 1)
bwd_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
           const __grid_constant__ CUtensorMap map_do, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sK = base, sV = base + TILE_BYTES, sQ = base + 2 * TILE_BYTES, sDO = base + 3 * TILE_BYTES, sP = base + 4 * TILE_BYTES,
                 sDS = base + 5 * TILE_BYTES;
  const uint32_t bars = base + 6 * TILE_BYTES;
  const uint32_t kv_full = bars, qdo_full = bars + 8, qdo_empty = bars + 16, s_full = bars + 24, s_free = bars + 32, pds_full = bars + 40,
                 dq_full = bars + 48, acc_done = bars + 56;
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(gen + 6 * TILE_BYTES + 8 * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tile = blockIdx.x, kv_head = blockIdx.y, batch = blockIdx.z;
  const int n0 = n_tile * BN;
  const int group = p.h / p.hk;
  const int num_m = (p.sq + BM - 1) / BM;
  int m_first = 0;
  if (p.causal) {                       // first query row that can see key n0: i >= n0 - causal_off
    const int r0 = max(0, n0 - p.causal_off);
    m_first = min(num_m, r0 / BM);
  }
  const int tiles_per_head = num_m - m_first;
  const int total = tiles_per_head * group;    // iteration it -> (query head = kv_head*group + it / tiles_per_head, m tile = m_first + it % tiles_per_head)

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    tma_prefetch_desc(&map_do);
    mbar_init(kv_full, 1); mbar_init(qdo_full, 1); mbar_init(qdo_empty, 1); mbar_init(s_full, 1); mbar_init(s_free, 8);
    mbar_init(pds_full, 8); mbar_init(dq_full, 1); mbar_init(acc_done, 1);
    fence_barrier_init();
    fence_proxy_async();
  } else if (warp == 9) {
    tmem_alloc(smem_u32((const void*)tmem_ptr), TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 8) {
    if (lane == 0 && total > 0) {
      // ================= TMA producer =================
      mbar_expect_tx(kv_full, 2 * TILE_BYTES);
      tma_load_4d(sK, &map_k, kv_full, 0, n0, kv_head, batch);
      tma_load_4d(sK + HALF_BYTES, &map_k, kv_full, 64, n0, kv_head, batch);
      tma_load_4d(sV, &map_v, kv_full, 0, n0, kv_head, batch);
      tma_load_4d(sV + HALF_BYTES, &map_v, kv_full, 64, n0, kv_head, batch);
      for (int it = 0; it < total; ++it) {
        const int head = kv_head * group + it / tiles_per_head;
        const int m0 = (m_first + it % tiles_per_head) * BM;
        mbar_wait(qdo_empty, (it & 1) ^ 1);
        mbar_expect_tx(qdo_full, 2 * TILE_BYTES);
        tma_load_4d(sQ, &map_q, qdo_full, 0, m0, head, batch);
        tma_load_4d(sQ + HALF_BYTES, &map_q, qdo_full, 64, m0, head, batch);
        tma_load_4d(sDO, &map_do, qdo_full, 0, m0, head, batch);
        tma_load_4d(sDO + HALF_BYTES, &map_do, qdo_full, 64, m0, head, batch);
      }
    }
  } else if (warp == 9) {
    if (lane == 0 && total > 0) {
      // ================= MMA issuer =================
      mbar_wait(kv_full, 0);
      for (int it = 0; it < total; ++it) {
        const uint32_t ph = it & 1;
        mbar_wait(qdo_full, ph);
        mbar_wait(s_free, ph ^ 1);        // S / dQ^T columns drained by the softmax warps (previous iteration)
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_f16(tmem_base + S_COL, desc_kmajor(sQ, kb, k), desc_kmajor(sK, kb, k), p.idesc_kk, (kb | k) != 0);    // S = Q K^T
            umma_f16(tmem_base + DP_COL, desc_kmajor(sDO, kb, k), desc_kmajor(sV, kb, k), p.idesc_kk, (kb | k) != 0);  // dP = dO V^T
          }
        umma_commit(s_full);
        mbar_wait(pds_full, ph);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {     // K dimension = 128 query rows, 16 per MMA
          umma_f16(tmem_base + DV_COL, desc_mnmajor(sP, kk), desc_mnmajor(sDO, kk), p.idesc_mm, (it | kk) != 0);   // dV += P^T dO
          umma_f16(tmem_base + DK_COL, desc_mnmajor(sDS, kk), desc_mnmajor(sQ, kk), p.idesc_mm, (it | kk) != 0);   // dK += dS^T Q
        }
        umma_commit(qdo_empty);              // Q / dO tiles may be overwritten by the next loads
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)       // K dimension = 128 keys; A = K tile read MN-major (M = head dim), B = dS read K-major (N = query)
          umma_f16(tmem_base + S_COL, desc_mnmajor(sK, kk), desc_kmajor(sDS, kk >> 2, kk & 3), p.idesc_mk, kk != 0);  // dQ^T = K^T dS^T
        umma_commit(dq_full);
      }
      umma_commit(acc_done);
    }
  } else {
    // ================= softmax / dQ reduction / epilogue: 2 warpgroups, each owns one 64-column half =================
    const int half = warp >> 2;                      // key half for S/dP, query half for dQ^T, head-dim half for dV/dK
    const int rl = (warp & 3) * 32 + lane;           // TMEM lane
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    constexpr float kLog2e = 1.4426950408889634f;
    for (int it = 0; it < total; ++it) {
      const uint32_t ph = it & 1;
      const int head = kv_head * group + it / tiles_per_head;
      const int m0 = (m_first + it % tiles_per_head) * BM;
      const int row = m0 + rl;
      const bool row_ok = row < p.sq;
      const int64_t stat = ((int64_t)batch * p.h + head) * p.sq + row;
      const float lse2 = row_ok ? p.lse[stat] * kLog2e : 0.f;
      const float dl = row_ok ? p.delta[stat] : 0.f;
      const int lim = p.causal ? min(p.sk - 1, row + p.causal_off) : p.sk - 1;   // last visible key of this query row
      const int4* cm = MASKED ? p.colmask + ((int64_t)batch * p.mask_heads + (p.mask_heads > 1 ? head : 0)) * p.sk : nullptr;
      (void)cm;
      mbar_wait(s_full, ph);
      tc_fence_after();
      // previous iteration's dV/dK/dQ MMAs have retired (we waited dq_full below), so the P / dS tiles are free
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t rs[32], rp[32];
        tmem_ld_32x32(tmem_base + lane_off + S_COL + half * 64 + c * 32, rs);
        tmem_ld_32x32(tmem_base + lane_off + DP_COL + half * 64 + c * 32, rp);
#pragma unroll
        for (int q8 = 0; q8 < 4; ++q8) {
          uint32_t up[4], ud[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float pv[2], ds[2];
#pragma unroll
            for (int t2 = 0; t2 < 2; ++t2) {
              const int i = q8 * 8 + 2 * e + t2;
              const int key = n0 + half * 64 + c * 32 + i;
              float x = ex2(fmaf(__uint_as_float(rs[i]), p.scale_log2, -lse2));
              if (!row_ok || key > lim) x = 0.f;
              if constexpr (MASKED) {
                if (key < p.sk) {
                  const int4 m = __ldg(cm + key);
                  if ((row >= m.x && row < m.y) || (row >= m.z && row < m.w)) x = 0.f;
                }
              }
              pv[t2] = x;
              ds[t2] = x * (__uint_as_float(rp[i]) - dl) * p.scale;
            }
            up[e] = pack2<T>(pv[0], pv[1]);
            ud[e] = pack2<T>(ds[0], ds[1]);
          }
          const int col = c * 32 + q8 * 8;              // key index inside this 64-key half
          const uint32_t off = half * HALF_BYTES + rl * 128 + (((col >> 3) ^ (rl & 7)) << 4);
          st_shared_v4(sP + off, up[0], up[1], up[2], up[3]);
          st_shared_v4(sDS + off, ud[0], ud[1], ud[2], ud[3]);
        }
      }
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(pds_full);          // 8 warp arrivals
      // dQ^T tile: TMEM lane = head-dim index (d = rl), columns = query rows; this warpgroup handles query columns [half*64, +64)
      mbar_wait(dq_full, ph);
      tc_fence_after();
      // Transpose through shared memory (the P + dS tiles are free: every MMA of this iteration has retired) into a row-major
      // fp32 [query][d] tile, then let the TMA engine reduce each 512-byte row into dQ (cp.reduce.async.bulk ... add.f32).
      const uint32_t sDQ = sP;   // 64 KB: sP and sDS are adjacent
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + lane_off + S_COL + half * 64 + c * 32, r);
#pragma unroll
        for (int i = 0; i < 32; ++i)
          asm volatile("st.shared.b32 [%0], %1;" ::"r"(sDQ + (uint32_t)(half * 64 + c * 32 + i) * 512u + (uint32_t)rl * 4u), "r"(r[i]) : "memory");
      }
      tc_fence_before();
      fence_proxy_async();
      // Deterministic mode (FLAGS_cudnn_deterministic): the fp32 adds of the bulk reduce are order dependent, so the key tiles take turns on
      // a query tile in ascending order (tile n waits for the counter to reach n; every key tile from 0 on contributes to every query tile
      // it visits, masked or not).  CTAs with a lower blockIdx.x are dispatched first, so the tile waited for is resident or done.
      int* sem = nullptr;
      if (p.dq_sem) {
        sem = p.dq_sem + ((int64_t)batch * p.h + head) * num_m + (m0 / BM);
        if (threadIdx.x == 0) {
          uint64_t t0 = 0;
          uint32_t spins = 0;
          while (true) {
            int v;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(sem) : "memory");
            if (v >= n_tile) break;
            if (++spins == 4096) t0 = globaltimer_ns();
            if (spins > 4096 && (spins & 1023) == 0 && globaltimer_ns() - t0 > 10000000000ull) {
              printf("b200 attention bwd: deterministic dQ turn timeout (block %d,%d,%d)\n", blockIdx.x, blockIdx.y, blockIdx.z);
              __trap();
            }
          }
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");      // both softmax warpgroups: the whole [128][128] fp32 tile is in smem (and it is our turn)
      if (half == 0 && m0 + rl < p.sq) {
        float* dst = p.dq + (int64_t)batch * p.dq_sb + (int64_t)(m0 + rl) * p.dq_ss + (int64_t)head * p.dq_sh;
        bulk_reduce_add_f32<512>(dst, sDQ + (uint32_t)rl * 512u);
      }
      bulk_commit();
      if (sem) {
        bulk_wait<0>();                                    // the adds have been performed, not just read from smem
        __threadfence();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (threadIdx.x == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(sem), "r"(n_tile + 1) : "memory");
      } else {
        bulk_wait_read<0>();                               // the tile in shared memory may be overwritten
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(s_free);            // 8 warp arrivals
    }
    // epilogue: dV, dK rows (lane = key row); this warpgroup writes head-dim columns [half*64, +64)
    if (total > 0) {
      mbar_wait(acc_done, 0);
      tc_fence_after();
    }
    const int key = n0 + rl;
    const int64_t kv_off = (int64_t)batch * p.dkv_sb + (int64_t)key * p.dkv_ss + (int64_t)kv_head * p.dkv_sh + half * 64;
    T* dv_row = reinterpret_cast<T*>(p.dv) + kv_off;
    T* dk_row = reinterpret_cast<T*>(p.dk) + kv_off;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      uint32_t rv[32], rk[32];
      if (total > 0) {
        tmem_ld_32x32(tmem_base + lane_off + DV_COL + half * 64 + c * 32, rv);
        tmem_ld_32x32(tmem_base + lane_off + DK_COL + half * 64 + c * 32, rk);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) { rv[i] = 0u; rk[i] = 0u; }
      }
      if (key < p.sk) {
#pragma unroll
        for (int q8 = 0; q8 < 4; ++q8) {
          uint4 ov, ok;
          ov.x = pack2<T>(__uint_as_float(rv[q8 * 8 + 0]), __uint_as_float(rv[q8 * 8 + 1]));
          ov.y = pack2<T>(__uint_as_float(rv[q8 * 8 + 2]), __uint_as_float(rv[q8 * 8 + 3]));
          ov.z = pack2<T>(__uint_as_float(rv[q8 * 8 + 4]), __uint_as_float(rv[q8 * 8 + 5]));
          ov.w = pack2<T>(__uint_as_float(rv[q8 * 8 + 6]), __uint_as_float(rv[q8 * 8 + 7]));
          ok.x = pack2<T>(__uint_as_float(rk[q8 * 8 + 0]), __uint_as_float(rk[q8 * 8 + 1]));
          ok.y = pack2<T>(__uint_as_float(rk[q8 * 8 + 2]), __uint_as_float(rk[q8 * 8 + 3]));
          ok.z = pack2<T>(__uint_as_float(rk[q8 * 8 + 4]), __uint_as_float(rk[q8 * 8 + 5]));
          ok.w = pack2<T>(__uint_as_float(rk[q8 * 8 + 6]), __uint_as_float(rk[q8 * 8 + 7]));
          *reinterpret_cast<uint4*>(dv_row + c * 32 + q8 * 8) = ov;
          *reinterpret_cast<uint4*>(dk_row + c * 32 + q8 * 8) = ok;
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// delta[b,h,s] = sum_d dO[b,s,h,d] * O[b,s,h,d]   (one warp per row; O and dO share the element strides (sb, ss, sh), d contiguous)
template <typename T>
__global__ void delta_kernel(const T* __restrict__ o, const T* __restrict__ d_o, float* __restrict__ delta, int64_t rows, int sq, int h,
                             int64_t sb, int64_t ss, int64_t sh) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // row = (b*sq + s)*h + head
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int64_t bs = row / h;
  const int head = (int)(row - bs * h);
  const int64_t bb = bs / sq;
  const int sidx = (int)(bs - bb * sq);
  const int64_t off = bb * sb + (int64_t)sidx * ss + (int64_t)head * sh + lane * 4;
  const uint2 a = *reinterpret_cast<const uint2*>(o + off);
  const uint2 b = *reinterpret_cast<const uint2*>(d_o + off);
  const T* pa = reinterpret_cast<const T*>(&a);
  const T* pb = reinterpret_cast<const T*>(&b);
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) acc += to_f(pa[i]) * to_f(pb[i]);
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o2);
  if (lane == 0) delta[(bb * h + head) * sq + sidx] = acc;
}

// 4-D map {d, s, h, b} over a strided [B,S,H,D] view (strides in elements), box {64, 128, 1, 1}, 128B swizzle
static bool make_map4(CUtensorMap* out, const void* ptr, int d, int s, int h, int b, int64_t ss, int64_t sh, int64_t sb, int dtype) {
  cuuint64_t dims[4] = {(cuuint64_t)d, (cuuint64_t)s, (cuuint64_t)h, (cuuint64_t)b};
  cuuint64_t strides[3] = {(cuuint64_t)ss * 2, (cuuint64_t)sh * 2, (cuuint64_t)sb * 2};
  cuuint32_t box[4] = {64, 128, 1, 1};
  return encode_tiled(out, dtype == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, ptr, dims, strides, box,
                      "attention bwd");
}

}  // namespace attn_bwd

int attention_bwd(const AttnBwdArgs& a, cudaStream_t s) {
  using namespace attn_bwd;
  if (!attention_fwd_supported(a.fwd)) return 1;
  const AttnArgs& f = a.fwd;
  CUtensorMap mq, mk, mv, mdo;
  if (!make_map4(&mq, f.q, f.d, f.sq, f.h, f.b, f.q_strides[1], f.q_strides[2], f.q_strides[0], f.dtype)) return 2;
  if (!make_map4(&mk, f.k, f.d, f.sk, f.hk, f.b, f.k_strides[1], f.k_strides[2], f.k_strides[0], f.dtype)) return 2;
  if (!make_map4(&mv, f.v, f.d, f.sk, f.hk, f.b, f.v_strides[1], f.v_strides[2], f.v_strides[0], f.dtype)) return 2;
  if (!make_map4(&mdo, a.d_o, f.d, f.sq, f.h, f.b, a.o_strides[1], a.o_strides[2], a.o_strides[0], f.dtype)) return 2;
  const int64_t rows = (int64_t)f.b * f.sq * f.h;
  const int wpb = 8;
  if (f.dtype == kBF16)
    delta_kernel<__nv_bfloat16><<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, s>>>((const __nv_bfloat16*)f.o, (const __nv_bfloat16*)a.d_o, a.delta, rows, f.sq, f.h,
                                                                                     a.o_strides[0], a.o_strides[1], a.o_strides[2]);
  else
    delta_kernel<__half><<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, s>>>((const __half*)f.o, (const __half*)a.d_o, a.delta, rows, f.sq, f.h, a.o_strides[0], a.o_strides[1], a.o_strides[2]);
  Params p;
  p.b = f.b; p.sq = f.sq; p.sk = f.sk; p.h = f.h; p.hk = f.hk;
  p.scale = f.scale; p.scale_log2 = f.scale * 1.4426950408889634f;
  p.causal = f.causal; p.causal_off = f.sk - f.sq;
  p.colmask = reinterpret_cast<const int4*>(f.colmask);
  p.mask_heads = f.mask_heads > 0 ? f.mask_heads : 1;
  p.dq_sem = a.dq_sem;
  p.lse = f.lse; p.delta = a.delta; p.dq = a.dq; p.dk = a.dk; p.dv = a.dv;
  p.dkv_sb = a.dkv_strides[0]; p.dkv_ss = a.dkv_strides[1]; p.dkv_sh = a.dkv_strides[2];
  p.dq_sb = a.dq_strides[0]; p.dq_ss = a.dq_strides[1]; p.dq_sh = a.dq_strides[2];
  const uint32_t fmt = f.dtype == kBF16 ? 1u : 0u;
  p.idesc_kk = umma_idesc(fmt, fmt, false, false, BM, BN, false);
  p.idesc_mm = umma_idesc(fmt, fmt, true, true, BM, BN, false);
  p.idesc_mk = umma_idesc(fmt, fmt, true, false, BM, BN, false);
  dim3 grid((f.sk + BN - 1) / BN, f.hk, f.b);
  static bool attr_set[4] = {false, false, false, false};
  auto go = [&](auto kern, int slot) {
    if (!attr_set[slot]) { B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)); attr_set[slot] = true; }
    kern<<<grid, kThreads, SMEM_BYTES, s>>>(mq, mk, mv, mdo, p);
  };
  if (f.dtype == kBF16) { if (p.colmask) go(bwd_kernel<__nv_bfloat16, true>, 0); else go(bwd_kernel<__nv_bfloat16, false>, 1); }
  else { if (p.colmask) go(bwd_kernel<__half, true>, 2); else go(bwd_kernel<__half, false>, 3); }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_last_error(__FILE__, __LINE__, cudaGetErrorString(e)); return 3; }
  return 0;
}

}  // namespace b200
