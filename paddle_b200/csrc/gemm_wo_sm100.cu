// Weight-only quantised GEMM for sm_100a: out[M,N] = x[M,K] (bf16 / fp16) @ dequant(Wq[N,K] int8 | int4) * scale[N] (+ bias), M <= 64.
//
// The int8 / int4 weights never exist as 16-bit values in HBM or in shared memory: TMA streams raw [128 channels x 128 B] boxes into a
// deep ring, sixteen dequantise warps expand them IN REGISTERS with packed 16-bit magic-number arithmetic and store them straight into
// TMEM (tcgen05.st), and tcgen05.mma reads its A operand from there.  The problem is computed transposed (D^T[N, M] = W[N, K] x^T) so
// that the weight tile is the 128-row A operand at full UMMA height even when M is a handful of decode tokens, the per-channel scale is
// a per-thread scalar in the epilogue (TMEM lane = output channel), and the token tile (UMMA N = 16 / 64) only costs what the batch
// needs.  Narrow layers are split along K over a thread-block CLUSTER whose CTAs reduce their partial tiles through DSMEM - no
// workspace, no atomics, no second kernel.  What each design step bought (k = 5120, n = 15360, m = 1, B200, profiles/
// bench_weight_only_r2.json and ncu_weight_only_r2.md): 64-byte boxes + one issuer + smem operand 43 us; four issuers 30 us; weight
// producer no longer throttled by the activation ring 23 us (cuBLAS bf16 on the 2x larger weight: 25 us).
//
// Parity: paddle/phi/kernels/gpu/weight_only_linear_kernel.cu:27, python/paddle/nn/quant/quantized_linear.py:183.
#include <cuda.h>
#include <cstdio>

#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_ptx.cuh"
#include "include/b200_tcgen05_host.h"

namespace b200 {
namespace wo {
using namespace ptx;

constexpr int BLOCK_N = 128;     // output channels per CTA = UMMA M (TMEM lanes)
constexpr int BLOCK_K = 64;
__host__ __device__ constexpr int wo_threads(int G) { return 32 * (4 + 4 * G + (G > 3 ? G - 3 : 0)); }   // producer, 3 issuers, 4G dequantise, issuers 3 ..
__host__ __device__ constexpr uint32_t pow2_at_least(uint32_t v) { uint32_t r = 32; while (r < v) r *= 2; return r; }


struct Params {
  int m, n, k;                 // tokens, output channels, reduction
  int kb_per_split;            // 64-wide k-blocks handled by one blockIdx.y
  const float* scale;          // [n] per-channel dequantisation factors
  const void* bias;            // [n] in the activation dtype or nullptr
  void* out;                   // [m, n] activation dtype (splits == 1)
  int splits;                  // blockIdx.y extent = cluster size: the CTAs of one output tile
  int bf16;                    // activation dtype: 1 bf16, 0 fp16
  uint32_t idesc;
};

// PTX prmt in its default mode: selector nibble bit 3 replicates the sign bit of the selected byte (the __byte_perm intrinsic only documents 3 bits)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ __half2 u32_as_half2(uint32_t v) { return *reinterpret_cast<__half2*>(&v); }
__device__ __forceinline__ uint32_t half2_as_u32(__half2 v) { return *reinterpret_cast<uint32_t*>(&v); }
__device__ __forceinline__ __nv_bfloat162 u32_as_bf162(uint32_t v) { return *reinterpret_cast<__nv_bfloat162*>(&v); }
__device__ __forceinline__ uint32_t bf162_as_u32(__nv_bfloat162 v) { return *reinterpret_cast<uint32_t*>(&v); }

// NTOK: token tile (UMMA N).  INT4: two weights per byte (low nibble = even k).
//
// Data path of one 64-wide k-block:  TMA raw box (128 channels x 128 B, shared by 2 int8 / 4 int4 k-blocks) -> one thread per channel
// row reads its 64 (32) bytes, expands them to 64 bf16 / fp16 in registers and stores them with tcgen05.st into the TMEM rows the tensor
// core reads its A operand from (tcgen05.mma with A in TMEM) -> D^T[128 channels, NTOK tokens] += A x_tile^T.  The dequantised weights
// never touch shared memory: the first version wrote them to a swizzled smem tile and the MMA read them back, and that round trip
// (16 KB written + 16 KB read per k-block on top of the raw bytes) saturated the 128 B/clk shared-memory pipe at ~600 cycles per k-block.
//
// Warp roles for G ring slots: warp 0 TMA producer; warps 1-3 and 4+4G .. issuers 0 .. G-1 (warp 1 also owns the TMEM allocation);
// warps 4 .. 4+4G-1 dequantise, four per group = one per TMEM lane quadrant (a warp may only touch lanes 32 (warp % 4) ..).  Group g
// converts k-blocks g, g + G, ... into TMEM slot g and issuer g multiplies them: the MMAs are tiny (NTOK columns), a k-block costs what
// its ISSUE sequence costs (~800 cycles for one thread), so every slot has its own issuer and the chains of G k-blocks overlap.
template <int NTOK, int G, int WST, int XPER, bool INT4, bool BF16>
__global__ void __launch_bounds__(wo_threads(G), 1)
wo_gemm_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x, const Params p) {
  constexpr int KB_PER_W = INT4 ? 4 : 2;                        // k-blocks covered by one raw box
  constexpr uint32_t W_BYTES = BLOCK_N * 128;                   // 16 KB raw box
  constexpr uint32_t X_BYTES = NTOK * BLOCK_K * 2;
  constexpr int ACC_PER = NTOK <= 16 ? 2 : 1;                   // independent TMEM accumulators per issuer (summed in the epilogue)
  constexpr int NACC = G * ACC_PER;
  constexpr uint32_t A_COLS = BLOCK_K / 2;                      // one slot: 128 lanes x 32 columns, two 16-bit k values per column
  constexpr uint32_t A_COL0 = NACC * NTOK;                      // accumulators first, then the G operand slots
  constexpr uint32_t TMEM_COLS = pow2_at_least(A_COL0 + G * A_COLS);
  static_assert(TMEM_COLS <= 512, "weight-only gemm: TMEM budget");
  static_assert(NTOK * 512 <= WST * W_BYTES, "weight-only gemm: the split-K partial tile is staged in the raw weight ring");
  // Activation tiles: XPER private stages per issuer (k-block i -> stage (i % G) * XPER + (i / G) % XPER), so every x_full barrier has ONE
  // waiter that sees its phases in order.  (A ring shared by all issuers lets one issuer run a whole phase ahead of another and read
  // the parity of the previous phase as "done".)
  constexpr int XST = G * XPER;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t wring = base;                                  // [WST] raw weight boxes
  const uint32_t xring = wring + WST * W_BYTES;                 // [XST] activation tiles
  const uint32_t bars = xring + XST * X_BYTES;
  auto w_full = [&](int s) { return bars + 8u * s; };
  auto w_empty = [&](int s) { return bars + 8u * (WST + s); };
  auto x_full = [&](int s) { return bars + 8u * (2 * WST + s); };
  auto x_empty = [&](int s) { return bars + 8u * (2 * WST + XST + s); };
  auto a_ready = [&](int s) { return bars + 8u * (2 * WST + 2 * XST + s); };
  auto a_empty = [&](int s) { return bars + 8u * (2 * WST + 2 * XST + G + s); };
  const uint32_t tfull = bars + 8u * (2 * WST + 2 * XST + 2 * G);
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(gen + WST * W_BYTES + XST * X_BYTES + 8 * (2 * WST + 2 * XST + 2 * G + 1));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BLOCK_N;
  const int tok0 = blockIdx.z * NTOK;
  const int num_kb_total = (p.k + BLOCK_K - 1) / BLOCK_K;
  const int kb0 = blockIdx.y * p.kb_per_split;
  const int num_kb = max(0, min(p.kb_per_split, num_kb_total - kb0));

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_x);
    for (int s = 0; s < WST; ++s) { mbar_init(w_full(s), 1); mbar_init(w_empty(s), KB_PER_W * 4); }
    for (int s = 0; s < XST; ++s) { mbar_init(x_full(s), 1); mbar_init(x_empty(s), 1); }
    for (int s = 0; s < G; ++s) { mbar_init(a_ready(s), 4); mbar_init(a_empty(s), 1); }
    mbar_init(tfull, G);
    fence_barrier_init();
    fence_proxy_async();
  } else if (warp == 1) {
    tmem_alloc(smem_u32((const void*)tmem_ptr), TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const bool is_dq = warp >= 4 && warp < 4 + 4 * G;
  const int ew = warp & 3;                                  // TMEM lane quadrant this warp may access (hardware: warp id % 4)

  if (warp == 0) {
    if (lane == 0) {
      // ================= TMA producer: raw quantised weights, one box per KB_PER_W k-blocks, throttled only by the box ring.  (The
      // activation tiles are loaded by the issuers: on this thread their small ring capped the weight bytes in flight.) =================
      const int num_box = (num_kb + KB_PER_W - 1) / KB_PER_W;
      for (int j = 0; j < num_box; ++j) {                   // kb0 is a multiple of KB_PER_W (launcher), so boxes start on 128-byte columns
        const int ws = j % WST;
        mbar_wait(w_empty(ws), ((j / WST) & 1) ^ 1);
        mbar_expect_tx(w_full(ws), W_BYTES);
        tma_load_2d(wring + ws * W_BYTES, &map_w, w_full(ws), (kb0 + j * KB_PER_W) * (INT4 ? BLOCK_K / 2 : BLOCK_K), n0);
      }
    }
  } else if (!is_dq) {
    if (lane == 0) {
      // ================= MMA issuers: D^T[128 channels, NTOK tokens] += A(TMEM slot g)[128, 64] x_tile[NTOK, 64]^T =================
      const int g = warp < 4 ? warp - 1 : warp - (4 + 4 * G) + 3;
      if (g < G) {
        const uint64_t bdesc0 = make_smem_desc(xring, 16, 1024);
        const uint32_t tacc = tmem_base + (uint32_t)(g * ACC_PER * NTOK), ta = tmem_base + A_COL0 + (uint32_t)g * A_COLS;
        int aph = 0;
        // issuer g also streams its own activation tiles: the tile of local iteration jj goes to private stage jj % XPER, XPER - 1 ahead
        auto load_x = [&](int jj) {
          const int i2 = g + jj * G;
          if (i2 >= num_kb) return;
          const int st = g * XPER + jj % XPER;
          mbar_wait(x_empty(st), ((jj / XPER) & 1) ^ 1);     // the MMAs of iteration jj - XPER (committed XPER - 1 iterations ago) are done
          mbar_expect_tx(x_full(st), X_BYTES);
          tma_load_3d(xring + st * X_BYTES, &map_x, x_full(st), (kb0 + i2) * BLOCK_K, tok0, 0);
        };
        for (int jj = 0; jj < XPER - 1; ++jj) load_x(jj);
        for (int i = g, j = 0; i < num_kb; i += G, ++j) {
          load_x(j + XPER - 1);
          const int s = g * XPER + j % XPER;
          mbar_wait(x_full(s), (j / XPER) & 1);              // the activation tile of this k-block has landed
          mbar_wait(a_ready(g), aph);                        // dequantise group g has stored the weight rows (tcgen05.st, waited, fenced)
          aph ^= 1;
          tc_fence_after();
          const uint64_t bd = bdesc0 + (uint64_t)((s * X_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k)
            umma_f16_ts(tacc + (uint32_t)((k % ACC_PER) * NTOK), ta + 8u * k, bd + 2 * k, p.idesc, (i != g || k >= ACC_PER) ? 1u : 0u);
          umma_commit(x_empty(s));
          umma_commit(a_empty(g));
        }
        umma_commit(tfull);
      }
    }
  } else {
    // ================= dequantise warps (warps 4-7 also run the epilogue): thread = one channel row of the box =================
    const int grp = (warp - 4) >> 2;
    const int r = ew * 32 + lane;                            // channel row inside the tile = TMEM lane
    const uint32_t ta = tmem_base + ((uint32_t)(ew * 32) << 16) + A_COL0 + (uint32_t)grp * A_COLS;
    for (int i = grp; i < num_kb; i += G) {
      const int j = i / KB_PER_W, ws = j % WST, sub = i % KB_PER_W;
      mbar_wait(w_full(ws), (j / WST) & 1);
      const uint32_t rowp = wring + ws * W_BYTES + r * 128;  // 128 rows x 128 B, SWIZZLE_128B: 16-byte piece c of row r sits at piece c ^ (r & 7)
      // 64 dequantised values, two per register, k ascending, in the activation dtype (tcgen05 kind::f16 rejects mixed f16 x bf16
      // operands).  The conversion rate is what bounds this kernel once the loads are deep enough, so it is done with packed 16-bit
      // arithmetic and magic numbers instead of int -> fp32 -> 16-bit:
      //   fp16: 0x6400 | u = 1024 + u exactly (10-bit mantissa holds a whole byte); one HSUB2 / HFMA2 removes the offset.
      //   bf16: only 7 mantissa bits: 0x4300 | (b & 0x7F) = 128 + low7 and 0x4300 | (b & 0x80) = 128 + 128 sign, whose difference is the
      //         two's-complement byte; int4 nibbles (value + 8 < 128) fit directly.
      uint32_t o[32];
      if constexpr (!INT4) {
        uint4 v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[q].x), "=r"(v[q].y), "=r"(v[q].z), "=r"(v[q].w) : "r"(rowp + (((sub * 4 + q) ^ (r & 7)) << 4)));
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t w4[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if constexpr (BF16) {
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                const uint32_t t = __byte_perm(w4[e], 0x43434343u, hh ? 0x5342 : 0x5140);      // [0x43 b1 0x43 b0]
                o[q * 8 + e * 2 + hh] = bf162_as_u32(__hsub2(u32_as_bf162(t & 0xFF7FFF7Fu), u32_as_bf162(t & 0xFF80FF80u)));
              }
            } else {
              const uint32_t u = w4[e] ^ 0x80808080u;        // byte + 128 in 0..255
              const __half2 bias8 = u32_as_half2(0x64806480u);   // 1024 + 128
              o[q * 8 + e * 2] = half2_as_u32(__hsub2(u32_as_half2(__byte_perm(u, 0x64646464u, 0x5140)), bias8));
              o[q * 8 + e * 2 + 1] = half2_as_u32(__hsub2(u32_as_half2(__byte_perm(u, 0x64646464u, 0x5342)), bias8));
            }
          }
        }
      } else {
        uint4 v[2];
#pragma unroll
        for (int q = 0; q < 2; ++q)
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[q].x), "=r"(v[q].y), "=r"(v[q].z), "=r"(v[q].w) : "r"(rowp + (((sub * 2 + q) ^ (r & 7)) << 4)));
        // byte c = (k = 2c low nibble, k = 2c + 1 high nibble), nibble ^ 8 = value + 8
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const uint32_t w4[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if constexpr (BF16) {
              // low / high nibbles as separate byte vectors; PRMT picks byte c of each and zero-fills the upper bytes (selector | 8
              // replicates the sign bit of a byte < 16): [0 hi 0 lo] | 0x43004300 = (128 + lo, 128 + hi), minus 136
              const uint32_t lo = (w4[e] ^ 0x88888888u) & 0x0F0F0F0Fu, hi = ((w4[e] >> 4) ^ 0x88888888u) & 0x0F0F0F0Fu;
              const __nv_bfloat162 off = u32_as_bf162(0x43084308u);   // 136
#pragma unroll
              for (int b = 0; b < 4; ++b) {
                const uint32_t t = prmt(lo, hi, 0x8080 + b * 0x0001 + (4 + b) * 0x0100) | 0x43004300u;
                o[q * 16 + e * 4 + b] = bf162_as_u32(__hsub2(u32_as_bf162(t), off));
              }
            } else {
              // [0x64 byte 0x64 byte] & 0x64F0640F = (1024 + lo, 1024 + 16 hi); HFMA2 with (1, 1/16) and (-1032, -72) leaves (lo - 8, hi - 8)
              const __half2 mul4 = u32_as_half2(0x2C003C00u), add4 = u32_as_half2(0xD480E408u);
              const uint32_t u = w4[e] ^ 0x88888888u;
#pragma unroll
              for (int b = 0; b < 4; ++b) {
                const uint32_t t = __byte_perm(u, 0x64646464u, 0x4040 + b * 0x0101) & 0x64F0640Fu;
                o[q * 16 + e * 4 + b] = half2_as_u32(__hfma2(u32_as_half2(t), mul4, add4));
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(w_empty(ws));               // the raw bytes are in registers: the box slot may be refilled
      mbar_wait(a_empty(grp), ((i / G) & 1) ^ 1);            // the MMAs that read this slot's previous contents have completed
      tc_fence_after();
      tmem_st32(ta, o);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready(grp));
    }
    // ---- epilogue (warps 4-7: one per TMEM lane quadrant): TMEM lane = output channel, column = token ----
    if (warp < 8) {
      if (num_kb > 0) {
        mbar_wait(tfull, 0);
        tc_fence_after();
      }
      const int chl = ew * 32 + lane, ch = n0 + chl;
      const bool ch_ok = ch < p.n;
      const float sc = ch_ok ? p.scale[ch] : 0.f;
      float bv = 0.f;
      if (ch_ok && p.bias && p.splits == 1) bv = BF16 ? __bfloat162float(((const __nv_bfloat16*)p.bias)[ch]) : __half2float(((const __half*)p.bias)[ch]);
      const int nacc = min(G, num_kb) * ACC_PER;           // accumulators that received at least one MMA (issuer g has work iff num_kb > g)
#pragma unroll 1
      for (int c = 0; c < NTOK / 16; ++c) {
        uint32_t acc[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = 0u;
        for (int a = 0; a < nacc; ++a) {
          uint32_t r2[16];
          tmem_ld16(tmem_base + ((uint32_t)(ew * 32) << 16) + a * NTOK + c * 16, r2);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[j] = __float_as_uint(__uint_as_float(acc[j]) + __uint_as_float(r2[j]));
        }
        if (p.splits > 1) {
          // split-K inside a cluster: park the partial tile [token][channel] in this CTA's shared memory (the raw weight ring is idle
          // now: every box was consumed before the last MMA could be issued); the cluster reduces it below through DSMEM
#pragma unroll
          for (int j = 0; j < 16; ++j)
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(wring + (uint32_t)(((c * 16 + j) * BLOCK_N + chl) * 4)), "r"(acc[j]) : "memory");
          continue;
        }
        if (!ch_ok) continue;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int tok = tok0 + c * 16 + j;
          if (tok >= p.m) break;
          const float y = __uint_as_float(acc[j]) * sc + bv;
          if constexpr (BF16) ((__nv_bfloat16*)p.out)[(int64_t)tok * p.n + ch] = __float2bfloat16_rn(y);
          else ((__half*)p.out)[(int64_t)tok * p.n + ch] = __float2half_rn(y);
        }
      }
      tc_fence_before();
    }
  }
  if (p.splits > 1) {
    // ---- cluster reduction: the p.splits CTAs of a cluster hold the partial tiles of ONE output tile; CTA r sums 32-channel chunks
    // r, r + splits, ... over all ranks (ld.shared::cluster) and writes the scaled result.  No workspace, no atomics, no second kernel.
    cluster_sync();
    if (warp >= 4 && warp < 8) {
      const uint32_t rank = cluster_ctarank();
      const int tok_n = min(NTOK, p.m - tok0);
      for (int c = (int)rank * 4 + (warp - 4); c < tok_n * 4; c += p.splits * 4) {
        const int tok = c >> 2, chl = (c & 3) * 32 + lane, ch = n0 + chl;
        float acc = 0.f;
        const uint32_t local = wring + (uint32_t)((tok * BLOCK_N + chl) * 4);
        for (int q = 0; q < p.splits; ++q) {
          float v;
          asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(mapa(local, q)) : "memory");
          acc += v;
        }
        if (ch < p.n) {
          float y = acc * p.scale[ch];
          if (p.bias) y += BF16 ? __bfloat162float(((const __nv_bfloat16*)p.bias)[ch]) : __half2float(((const __half*)p.bias)[ch]);
          if constexpr (BF16) ((__nv_bfloat16*)p.out)[(int64_t)(tok0 + tok) * p.n + ch] = __float2bfloat16_rn(y);
          else ((__half*)p.out)[(int64_t)(tok0 + tok) * p.n + ch] = __float2half_rn(y);
        }
      }
    }
    cluster_sync();                                        // nobody leaves while a peer may still read its partial tile
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// raw weights as bytes: [n rows, row_bytes], box {128 bytes, 128 rows}, SWIZZLE_128B
static bool make_w_map(CUtensorMap* out, const void* w, int n, int row_bytes) {
  cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)n};
  cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
  cuuint32_t box[2] = {128u, (cuuint32_t)BLOCK_N};
  return encode_tiled(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, w, dims, strides, box, "weight-only gemm");
}

template <int NTOK, int G, int WST, int XPER, bool INT4, bool BF16>
static int launch(const WoGemmArgs& g, const CUtensorMap& mw, cudaStream_t s) {
  constexpr int XST = G * XPER;
  constexpr uint32_t SMEM = WST * BLOCK_N * 128 + XST * NTOK * BLOCK_K * 2 + 1024 + 512;
  static_assert(SMEM <= 232448, "weight-only gemm: shared memory budget");
  static_assert(8 * (2 * WST + 2 * XST + 2 * G + 1) + 8 <= 512, "weight-only gemm: barrier area");
  constexpr int kMaxSplits = 8;                 // portable cluster size
  CUtensorMap mx;
  if (!gemm::make_map(&mx, g.x, g.k, g.m, 1, g.k, 0, BLOCK_K, NTOK, g.bf16 ? kBF16 : kF16)) return 2;
  auto kern = wo_gemm_kernel<NTOK, G, WST, XPER, INT4, BF16>;
  static bool attr_set = false;
  static int wave_ctas[kMaxSplits + 1];         // CTAs the device holds at once when they come in clusters of `splits`
  if (!attr_set) {
    B200_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    for (int c = 1; c <= kMaxSplits; ++c) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(1, c, 1); cfg.blockDim = dim3(wo_threads(G)); cfg.dynamicSmemBytes = SMEM;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 1; at[0].val.clusterDim.y = c; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      int n_clusters = 0;
      if (cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg) != cudaSuccess) { cudaGetLastError(); n_clusters = 0; }
      wave_ctas[c] = n_clusters * c;
    }
    if (wave_ctas[1] <= 0) wave_ctas[1] = sm_count();
    attr_set = true;
  }
  Params p;
  p.m = g.m; p.n = g.n; p.k = g.k;
  const int num_kb = (g.k + BLOCK_K - 1) / BLOCK_K;
  const int n_tiles = (g.n + BLOCK_N - 1) / BLOCK_N, t_tiles = (g.m + NTOK - 1) / NTOK;
  // Split-K (a cluster of `splits` CTAs per output tile) when the output tiles alone leave SMs idle or the last wave ragged.  Cost in
  // k-block units: waves x (k-blocks per CTA + fixed prologue / epilogue) + the cluster reduction.
  const int ctas = n_tiles * t_tiles;
  int splits = 1, kb_per = (num_kb + 3) / 4 * 4;
  long best = -1;
  for (int c = 1; c <= kMaxSplits; ++c) {
    if (wave_ctas[c] <= 0) continue;
    const int per = ((num_kb + c - 1) / c + 3) / 4 * 4;           // raw boxes span up to 4 k-blocks: split boundaries stay on box boundaries
    if (c > 1 && (c - 1) * per >= num_kb) continue;               // every rank of the cluster gets work
    const long waves = ((long)ctas * c + wave_ctas[c] - 1) / wave_ctas[c];
    const long cost = waves * (per + 24) + (c > 1 ? 6 : 0);
    if (best < 0 || cost < best) { best = cost; splits = c; kb_per = per; }
  }
  p.splits = splits;
  p.kb_per_split = kb_per;
  p.scale = g.scale; p.bias = g.bias; p.out = g.out; p.bf16 = g.bf16;
  // UMMA M = 128 channels, N = tokens; A (dequantised weights, TMEM) in the activation dtype: mixed f16 x bf16 traps
  const uint32_t f = g.bf16 ? 1u : 0u;
  p.idesc = umma_idesc(f, f, false, false, BLOCK_N, NTOK, false);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(n_tiles, splits, t_tiles); cfg.blockDim = dim3(wo_threads(G)); cfg.dynamicSmemBytes = SMEM; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 1; at[0].val.clusterDim.y = splits; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, mw, mx, p);
  if (e != cudaSuccess) { cudaGetLastError(); set_last_error(__FILE__, __LINE__, cudaGetErrorString(e)); return 3; }
  return 0;
}

template <bool INT4, bool BF16>
static int dispatch_tok(const WoGemmArgs& g, const CUtensorMap& mw, cudaStream_t s) {
  if (g.m <= 16) return launch<16, 4, 10, 4, INT4, BF16>(g, mw, s);      // decode: 160 KB of raw weights in flight
  return launch<64, 4, 8, 3, INT4, BF16>(g, mw, s);
}

}  // namespace wo

int gemm_weight_only(const WoGemmArgs& g, cudaStream_t s) {
  using namespace wo;
  if (g.k % 64 || g.n % 8 || g.m <= 0 || g.m > 64) return 1;      // larger batches: dequantise once + the bf16 GEMM (nn/quant.py)
  if ((reinterpret_cast<uintptr_t>(g.x) | reinterpret_cast<uintptr_t>(g.w) | reinterpret_cast<uintptr_t>(g.out)) & 15) return 1;
  CUtensorMap mw;
  const int row_bytes = g.int4 ? g.k / 2 : g.k;
  if (!make_w_map(&mw, g.w, g.n, row_bytes)) return 2;
  if (g.int4) return g.bf16 ? dispatch_tok<true, true>(g, mw, s) : dispatch_tok<true, false>(g, mw, s);
  return g.bf16 ? dispatch_tok<false, true>(g, mw, s) : dispatch_tok<false, false>(g, mw, s);
}

}  // namespace b200
