// Flash-attention forward for sm_100a (head_dim 128, bf16/fp16): S = Q K^T and O += P V run on tcgen05 tensor cores with
// the S tiles double-buffered in TMEM, K/V tiles streamed by TMA (4-D maps straight over the strided [B,S,H,D] views of a
// packed QKV tensor, so no q/k/v split copies), online softmax in registers (one thread = one query row = one TMEM lane),
// lazy O rescaling in TMEM.  Hand-written PTX; no CUTLASS, no library attention.
//
// Parity (behaviour): paddle.nn.functional.flash_attention / scaled_dot_product_attention
// (python/paddle/nn/functional/flash_attention.py -> phi flash_attn kernels calling the flash-attention library).
//
// CTA = 128 query rows of one (batch, head).  The key tiles are dealt to TWO independent softmax streams by parity: warpgroup w
// (warps 4w .. 4w+3, one thread = one query row = one TMEM lane, the whole 128-key row of the tile) owns tiles w, w + 2, ... with its own
// S buffer, P buffer, running (max, sum) and its own O accumulator in TMEM; the two partial results are merged once in the epilogue
// (flash-decoding style).  Nothing is exchanged between the warpgroups per tile, so their phases drift apart and the exp2 unit, which
// bounds the softmax (16 / clk / SM = 1024 cycles per tile, the same as the two MMAs), is fed by one stream while the other loads,
// reduces, stores P or waits.  Warp 8: TMA producer; warp 9: TMEM alloc + S = Q K^T issuer; warp 10: O += P V issuer - one thread
// issuing all 16 MMAs of a tile (descriptor arithmetic included) needed ~2900 cycles per tile and was itself the bound (ncu: the issuer
// warp busy 78 % of the time, profiles/ncu_attention_r2.md).
// TMEM columns: [0,128) S stream 0, [128,256) S stream 1, [256,384) O stream 0, [384,512) O stream 1.
#include <cuda.h>
#include <cstdio>

#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_ptx.cuh"
#include "include/b200_tcgen05_host.h"

namespace b200 {
namespace attn {
using namespace ptx;

constexpr int BM = 128, BN = 128, HD = 128;
constexpr int kThreads = 352;   // warps 0-7: softmax (2 warpgroups = 2 streams), warp 8: TMA producer, warp 9: TMEM alloc + QK issuer, warp 10: PV issuer
constexpr uint32_t TILE_BYTES = 128 * 128 * 2;   // 32 KB: every operand tile (Q, K, V, P)
constexpr uint32_t HALF_BYTES = TILE_BYTES / 2;  // one 64-wide K-block of a tile
constexpr uint32_t SMEM_BYTES = 7 * TILE_BYTES + 1024 /*align*/ + 256 /*barriers*/;   // Q, 2x K, 2x V, 2x P (the epilogue exchange reuses the Q tile)
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t O_COL = 256;

struct Params {
  int b, sq, sk, h, hk;
  float scale_log2;
  int causal, causal_off;     // key j is visible to query i iff j <= i + causal_off
  void* o;
  float* lse;
  int64_t o_sb, o_ss, o_sh;   // element strides of the output [B,S,H,D]
  int dtype;
  uint32_t idesc_qk, idesc_pv;
  const int4* colmask;        // [b, mask_heads, sk] row ranges hidden from every key column (nullptr: none)
  int mask_heads;
};

// MASKED: column-wise row-range mask (flashmask / varlen) compiled in; the dense instantiation carries none of its code or registers
template <typename T, bool MASKED>
__global__ void __launch_bounds__(kThreads, 1)
fwd_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
           const __grid_constant__ CUtensorMap map_v, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQ = base;
  auto sP = [&](int s) { return base + (5 + s) * TILE_BYTES; };
  auto sK = [&](int s) { return base + (1 + s) * TILE_BYTES; };
  auto sV = [&](int s) { return base + (3 + s) * TILE_BYTES; };
  const uint32_t bars = base + 7 * TILE_BYTES;
  const uint32_t q_full = bars;
  auto k_full = [&](int s) { return bars + 8u * (1 + s); };
  auto v_full = [&](int s) { return bars + 8u * (3 + s); };
  auto k_empty = [&](int s) { return bars + 8u * (5 + s); };
  auto v_empty = [&](int s) { return bars + 8u * (7 + s); };
  auto s_full = [&](int w) { return bars + 8u * (9 + w); };      // per stream: S tile computed
  auto s_empty = [&](int w) { return bars + 8u * (11 + w); };    // per stream: S tile consumed (4 warp arrivals)
  auto pv_done = [&](int w) { return bars + 8u * (13 + w); };    // per stream: O accumulator holds every P V issued so far
  auto p_full = [&](int w) { return bars + 8u * (15 + w); };     // per stream: P tile written (4 warp arrivals)
  auto p_free = [&](int w) { return bars + 8u * (17 + w); };     // per stream: P tile read by its P V
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(gen + 7 * TILE_BYTES + 8 * 20);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = (int)gridDim.x - 1 - (int)blockIdx.x;   // long (late) rows first under the causal mask
  const int head = blockIdx.y, batch = blockIdx.z;
  const int kv_head = head / (p.h / p.hk);
  const int m0 = m_tile * BM;
  int n_tiles = (p.sk + BN - 1) / BN;
  if (p.causal) {
    const int last_key = min(p.sk - 1, m0 + BM - 1 + p.causal_off);
    n_tiles = last_key < 0 ? 0 : min(n_tiles, last_key / BN + 1);
  }

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(k_full(s), 1); mbar_init(v_full(s), 1); mbar_init(k_empty(s), 1); mbar_init(v_empty(s), 1);
      mbar_init(s_full(s), 1); mbar_init(s_empty(s), 4);
      mbar_init(p_full(s), 4); mbar_init(p_free(s), 1);
      mbar_init(pv_done(s), 1);
    }
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
    if (lane == 0 && n_tiles > 0) {
      // ================= TMA producer =================
      mbar_expect_tx(q_full, TILE_BYTES);
      tma_load_4d(sQ, &map_q, q_full, 0, m0, head, batch);
      tma_load_4d(sQ + HALF_BYTES, &map_q, q_full, 64, m0, head, batch);
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j & 1, n0 = j * BN;
        const uint32_t ph = ((j >> 1) & 1) ^ 1;
        mbar_wait(k_empty(s), ph);
        mbar_expect_tx(k_full(s), TILE_BYTES);
        tma_load_4d(sK(s), &map_k, k_full(s), 0, n0, kv_head, batch);               // box {64 d, 128 keys}: K-major B operand
        tma_load_4d(sK(s) + HALF_BYTES, &map_k, k_full(s), 64, n0, kv_head, batch);
        mbar_wait(v_empty(s), ph);
        mbar_expect_tx(v_full(s), TILE_BYTES);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)                                              // box {64 d, 64 keys}: MN-major B operand
#pragma unroll
          for (int i = 0; i < 2; ++i)
            tma_load_4d(sV(s) + kb * HALF_BYTES + i * 8192, &map_v, v_full(s), i * 64, n0 + kb * 64, kv_head, batch);
      }
    }
  } else if (warp == 9) {
    if (lane == 0 && n_tiles > 0) {
      // ================= S = Q K^T issuer.  Descriptors are built once; a k-step only adds to the 14-bit (address >> 4) field =========
      mbar_wait(q_full, 0);
      const uint64_t qd = make_smem_desc(sQ, 16, 1024), kd0 = make_smem_desc(sK(0), 16, 1024);
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j & 1, ph = (j >> 1) & 1;              // K stage and stream share the parity of j
        mbar_wait(k_full(s), ph);
        mbar_wait(s_empty(s), ph ^ 1);
        tc_fence_after();
        const uint64_t kd = kd0 + (uint64_t)((s * TILE_BYTES) >> 4);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16(tmem_base + s * BN, qd + ((kb * HALF_BYTES + k * 32) >> 4), kd + ((kb * HALF_BYTES + k * 32) >> 4), p.idesc_qk, (kb | k) != 0);
        umma_commit(s_full(s));
        umma_commit(k_empty(s));
      }
    }
  } else if (warp == 10) {
    if (lane == 0 && n_tiles > 0) {
      // ================= O_stream += P V issuer =================
      const uint64_t pd0 = make_smem_desc(sP(0), 16, 1024), vd0 = make_smem_desc(sV(0), 8192, 1024);
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j & 1, ph = (j >> 1) & 1;
        mbar_wait(p_full(s), ph);
        mbar_wait(v_full(s), ph);
        tc_fence_after();
        const uint64_t pd = pd0 + (uint64_t)((s * TILE_BYTES) >> 4), vd = vd0 + (uint64_t)((s * TILE_BYTES) >> 4);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16(tmem_base + O_COL + s * HD, pd + ((kb * HALF_BYTES + k * 32) >> 4), vd + ((kb * HALF_BYTES + k * 2048) >> 4), p.idesc_pv, (j >= 2) || (kb | k) != 0);
        umma_commit(pv_done(s));
        umma_commit(p_free(s));
        umma_commit(v_empty(s));
      }
    }
  } else {
    // ================= softmax + epilogue: warpgroup w is stream w (tiles w, w + 2, ...); thread -> query row = TMEM lane ==========
    const int w = warp >> 2;
    const int rl = (warp & 3) * 32 + lane;           // row inside the tile == TMEM lane
    const int row = m0 + rl;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tS = tmem_base + lane_off + w * BN, tO = tmem_base + lane_off + O_COL + w * HD;
    float m_i = -INFINITY, l_i = 0.f;
    int it = 0;                                      // local iteration of this stream
    for (int j = w; j < n_tiles; j += 2, ++it) {
      const int ph = it & 1;
      mbar_wait(s_full(w), ph);
      tc_fence_after();
      // The whole 128-key row goes to registers at once and the S buffer is handed back immediately: this stream's next Q K^T (issue +
      // MMA + commit is ~1500-2500 cycles of latency) then runs under this tile's softmax instead of after it.
      float sv[128];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(tS + c * 32, r);
#pragma unroll
        for (int i = 0; i < 32; ++i) sv[c * 32 + i] = __uint_as_float(r[i]);   // raw logits; the softmax scale is folded into the exp2 FFMA
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty(w));
      const bool edge = (j * BN + BN > p.sk) || (p.causal && j * BN + BN - 1 > m0 + p.causal_off);
      if (edge) {
        const int lim = (p.causal ? min(p.sk - 1, row + p.causal_off) : p.sk - 1) - j * BN;   // last visible key, tile-relative
#pragma unroll
        for (int i = 0; i < 128; ++i)
          if (i > lim) sv[i] = -INFINITY;
      }
      if constexpr (MASKED) {     // flashmask / varlen: key column j hides the query rows [lt_start, lt_end) and [ut_start, ut_end)
        const int4* cm = p.colmask + ((int64_t)batch * p.mask_heads + (p.mask_heads > 1 ? head : 0)) * p.sk;
#pragma unroll
        for (int i = 0; i < 128; ++i) {
          const int key = j * BN + i;
          if (key < p.sk) {
            const int4 m = __ldg(cm + key);         // same address in every lane: one broadcast transaction
            if ((row >= m.x && row < m.y) || (row >= m.z && row < m.w)) sv[i] = -INFINITY;
          }
        }
      }
      float mxp[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) mxp[i] = sv[i];
#pragma unroll
      for (int i = 8; i < 128; ++i) mxp[i & 7] = fmaxf(mxp[i & 7], sv[i]);
      const float mx = fmaxf(fmaxf(fmaxf(mxp[0], mxp[1]), fmaxf(mxp[2], mxp[3])), fmaxf(fmaxf(mxp[4], mxp[5]), fmaxf(mxp[6], mxp[7]))) * p.scale_log2;   // scale > 0
      float m_new = fmaxf(m_i, mx);
      if (m_new == -INFINITY) m_new = 0.f;          // fully masked so far: keep exp2 finite
      if (it == 0) {
        m_i = m_new;
      } else {
        const bool need = (m_new - m_i) > 8.f;      // lazy rescale: keep a stale max while exp2 stays <= 2^8
        if (__any_sync(0xffffffffu, need)) {         // rare: only then must this stream's previous P V have landed before we touch O
          mbar_wait(pv_done(w), (it - 1) & 1);
          tc_fence_after();
          const float alpha = need ? ex2(m_i - m_new) : 1.f;
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            uint32_t r[32];
            tmem_ld_32x32(tO + c * 32, r);
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
            tmem_st32(tO + c * 32, r);
          }
          tc_fence_before();
          l_i *= alpha;
          if (need) m_i = m_new;
        }
      }
      mbar_wait(p_free(w), ph ^ 1);                 // this stream's previous P V has finished reading the P buffer
      // ---- P = exp2(S * scale - m), row sum, P tile to shared memory (K-major SWIZZLE_128B, two 64-key blocks) ----
      float sump[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) sump[e] = 0.f;
#pragma unroll
      for (int c = 0; c < 16; ++c) {                 // 8 keys = one 16-byte piece
        uint32_t u[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float p0 = ex2(fmaf(sv[c * 8 + 2 * e], p.scale_log2, -m_i));
          const float p1 = ex2(fmaf(sv[c * 8 + 2 * e + 1], p.scale_log2, -m_i));
          sump[2 * e] += p0;
          sump[2 * e + 1] += p1;
          u[e] = pack2<T>(p0, p1);          // one cvt.rn.{bf16x2,f16x2}.f32 per pair
        }
        const uint32_t addr = sP(w) + (c >> 3) * HALF_BYTES + rl * 128 + (((c & 7) ^ (rl & 7)) << 4);
        st_shared_v4(addr, u[0], u[1], u[2], u[3]);
      }
      l_i += ((sump[0] + sump[1]) + (sump[2] + sump[3])) + ((sump[4] + sump[5]) + (sump[6] + sump[7]));
      fence_proxy_async();     // generic-proxy smem writes -> visible to the tensor core (async proxy)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full(w));       // this stream's P V may start
    }
    if (it > 0) {
      mbar_wait(pv_done(w), (it - 1) & 1);
      tc_fence_after();
    }
    // ---- merge the two streams: row r of both O accumulators lives in TMEM lane r, which both warpgroups' warp (r / 32) can read; only
    // (max, sum) cross through shared memory - each stream publishes in its OWN P buffer, which is idle once its last P V completed
    // (the Q / K / V tiles may still be read by the other stream's MMAs) ----
    float* xch_me = reinterpret_cast<float*>(gen + (5 + w) * TILE_BYTES);        // [128][2] floats
    const float* xch_x = reinterpret_cast<const float*>(gen + (5 + (w ^ 1)) * TILE_BYTES);
    xch_me[rl * 2] = it > 0 ? m_i : -INFINITY;
    xch_me[rl * 2 + 1] = it > 0 ? l_i : 0.f;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const float m_x = xch_x[rl * 2], l_x = xch_x[rl * 2 + 1];
    const float m_me = it > 0 ? m_i : -INFINITY, l_me = it > 0 ? l_i : 0.f;
    float m_tot = fmaxf(m_me, m_x);
    if (m_tot == -INFINITY) m_tot = 0.f;
    const float a_me = l_me > 0.f ? ex2(m_me - m_tot) : 0.f, a_x = l_x > 0.f ? ex2(m_x - m_tot) : 0.f;
    const float l_tot = l_me * a_me + l_x * a_x;
    const float inv = l_tot > 0.f ? 1.f / l_tot : 0.f;
    const float c_me = a_me * inv, c_x = a_x * inv;
    const bool any_me = __any_sync(0xffffffffu, c_me != 0.f), any_x = __any_sync(0xffffffffu, c_x != 0.f);   // tcgen05.ld is warp-collective
    // warpgroup w writes output columns [64 w, 64 w + 64) of its rows from BOTH accumulators
    const uint32_t tO_me = tmem_base + lane_off + O_COL + w * HD + w * 64, tO_x = tmem_base + lane_off + O_COL + (w ^ 1) * HD + w * 64;
    T* orow = reinterpret_cast<T*>(p.o) + (int64_t)batch * p.o_sb + (int64_t)row * p.o_ss + (int64_t)head * p.o_sh + w * 64;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      float acc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = 0.f;
      if (any_me) {
        uint32_t r[32];
        tmem_ld_32x32(tO_me + c * 32, r);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = c_me != 0.f ? __uint_as_float(r[i]) * c_me : 0.f;
      }
      if (any_x) {
        uint32_t r[32];
        tmem_ld_32x32(tO_x + c * 32, r);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] += c_x != 0.f ? __uint_as_float(r[i]) * c_x : 0.f;
      }
      if (row < p.sq) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 o;
          o.x = pack2<T>(acc[q * 8 + 0], acc[q * 8 + 1]);
          o.y = pack2<T>(acc[q * 8 + 2], acc[q * 8 + 3]);
          o.z = pack2<T>(acc[q * 8 + 4], acc[q * 8 + 5]);
          o.w = pack2<T>(acc[q * 8 + 6], acc[q * 8 + 7]);
          *reinterpret_cast<uint4*>(orow + c * 32 + q * 8) = o;
        }
      }
    }
    if (w == 0 && row < p.sq && p.lse) p.lse[((int64_t)batch * p.h + head) * p.sq + row] = l_tot > 0.f ? (m_tot + log2f(l_tot)) * 0.69314718055994531f : -INFINITY;
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------- host side
// 4-D map {d, s, h, b} over a strided [B,S,H,D] view (strides in elements), box {64, rows, 1, 1}, 128B swizzle
static bool make_map4(CUtensorMap* out, const void* ptr, int d, int s, int h, int b, int64_t ss, int64_t sh, int64_t sb, uint32_t box_rows, int dtype) {
  cuuint64_t dims[4] = {(cuuint64_t)d, (cuuint64_t)s, (cuuint64_t)h, (cuuint64_t)b};
  cuuint64_t strides[3] = {(cuuint64_t)ss * 2, (cuuint64_t)sh * 2, (cuuint64_t)sb * 2};
  cuuint32_t box[4] = {64, box_rows, 1, 1};
  return encode_tiled(out, dtype == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, ptr, dims, strides, box,
                      "attention");
}

}  // namespace attn

int attention_fwd_supported(const AttnArgs& a) {
  if (a.d != 128 || (a.dtype != kBF16 && a.dtype != kF16)) return 0;
  if (a.h % a.hk) return 0;
  const int64_t* st[3] = {a.q_strides, a.k_strides, a.v_strides};
  for (auto s : st)
    for (int i = 0; i < 3; ++i)
      if (s[i] % 8) return 0;                    // TMA strides: multiples of 16 bytes
  if ((reinterpret_cast<uintptr_t>(a.q) | reinterpret_cast<uintptr_t>(a.k) | reinterpret_cast<uintptr_t>(a.v) | reinterpret_cast<uintptr_t>(a.o)) & 15) return 0;
  if (a.o_strides[0] % 8 || a.o_strides[1] % 8 || a.o_strides[2] % 8) return 0;
  return 1;
}

int attention_fwd(const AttnArgs& a, cudaStream_t s) {
  using namespace attn;
  if (!attention_fwd_supported(a)) return 1;
  CUtensorMap mq, mk, mv;
  // strides arrays are (batch, seq, head)
  if (!make_map4(&mq, a.q, a.d, a.sq, a.h, a.b, a.q_strides[1], a.q_strides[2], a.q_strides[0], BM, a.dtype)) return 2;
  if (!make_map4(&mk, a.k, a.d, a.sk, a.hk, a.b, a.k_strides[1], a.k_strides[2], a.k_strides[0], BN, a.dtype)) return 2;
  if (!make_map4(&mv, a.v, a.d, a.sk, a.hk, a.b, a.v_strides[1], a.v_strides[2], a.v_strides[0], 64, a.dtype)) return 2;
  Params p;
  p.b = a.b; p.sq = a.sq; p.sk = a.sk; p.h = a.h; p.hk = a.hk;
  p.scale_log2 = a.scale * 1.4426950408889634f;
  p.causal = a.causal; p.causal_off = a.sk - a.sq;
  p.o = a.o; p.lse = a.lse;
  p.o_sb = a.o_strides[0]; p.o_ss = a.o_strides[1]; p.o_sh = a.o_strides[2];
  p.dtype = a.dtype;
  const uint32_t f = a.dtype == kBF16 ? 1u : 0u;
  p.idesc_qk = umma_idesc(f, f, false, false, BM, BN, false);
  p.idesc_pv = umma_idesc(f, f, false, true, BM, HD, false);   // B operand MN-major (V: head_dim contiguous)
  p.colmask = reinterpret_cast<const int4*>(a.colmask);
  p.mask_heads = a.mask_heads > 0 ? a.mask_heads : 1;
  dim3 grid((a.sq + BM - 1) / BM, a.h, a.b);
  static bool attr_bf = false, attr_h = false;
  static bool attr_bf_m = false, attr_h_m = false;
  if (a.dtype == kBF16 && !p.colmask) {
    auto kern = fwd_kernel<__nv_bfloat16, false>;
    if (!attr_bf) { B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)); attr_bf = true; }
    kern<<<grid, kThreads, SMEM_BYTES, s>>>(mq, mk, mv, p);
  } else if (a.dtype == kBF16) {
    auto kern = fwd_kernel<__nv_bfloat16, true>;
    if (!attr_bf_m) { B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)); attr_bf_m = true; }
    kern<<<grid, kThreads, SMEM_BYTES, s>>>(mq, mk, mv, p);
  } else if (!p.colmask) {
    auto kern = fwd_kernel<__half, false>;
    if (!attr_h) { B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)); attr_h = true; }
    kern<<<grid, kThreads, SMEM_BYTES, s>>>(mq, mk, mv, p);
  } else {
    auto kern = fwd_kernel<__half, true>;
    if (!attr_h_m) { B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)); attr_h_m = true; }
    kern<<<grid, kThreads, SMEM_BYTES, s>>>(mq, mk, mv, p);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_last_error(__FILE__, __LINE__, cudaGetErrorString(e)); return 3; }
  return 0;
}

}  // namespace b200
