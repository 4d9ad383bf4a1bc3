// Collectives over NVLink/NVSwitch peer memory: the kernels issue ld/st.global directly on IPC-mapped peer pointers
// (symmetric heap, csrc/runtime/symm_heap.cpp).  No NCCL on these paths.
//
// Parity (role): ProcessGroupNCCL::AllReduce/ReduceScatter/AllGather (paddle/fluid/distributed/collective/
// process_group_nccl.cc) as used by DataParallel's EagerReducer, GroupSharded stage2/3 and the mp layers.
//
// Protocol: every rank owns a signal pad (first bytes of its heap slab): pad[slot][src_rank] (uint32).
//   start barrier  : rank r stores `epoch` into pad[0][r] of every peer (st.release.sys); all CTAs spin on their local
//                    pad[0][*] >= epoch (ld.acquire.sys)  -> peers' input data is visible.
//   end barrier    : the last CTA of the grid stores `epoch` into pad[1][r] of every peer and waits for pad[1][*]
//                    -> when the kernel retires, every peer has finished reading/writing this rank's buffer.
// Reductions accumulate in fp32 in a fixed rank order (deterministic).
#include <cstdio>

#include "../include/b200_common.cuh"
#include "../include/b200_comm.h"
#include "../include/b200_signal_pad.cuh"

namespace b200 {
namespace comm {

constexpr int kMaxRanks = 8;
constexpr int kThreads = 512;
constexpr uint64_t kBarrierTimeoutNs = 10000000000ull;   // 10 s: a dead peer or a protocol bug traps instead of hanging the GPU

struct Peers {
  char* base[kMaxRanks];
};

// the signal pad of every rank is the first bytes of its heap slab
__device__ __forceinline__ uint32_t* const* pads(const Peers& P) { return reinterpret_cast<uint32_t* const*>(P.base); }
__device__ __forceinline__ void signal_all(const Peers& P, int rank, int world, int slot, uint32_t epoch) {
  pad::signal_all(pads(P), rank, world, slot, epoch);
}
__device__ __forceinline__ void wait_all(const Peers& P, int rank, int world, int slot, uint32_t epoch) {
  pad::wait_all(pads(P), rank, world, slot, epoch, kBarrierTimeoutNs, B200_PAD_TIMEOUT("p2p"));
}
using pad::last_cta;

// ---------------------------------------------------------------------------------------------- two-shot all-reduce
// buffer of n elements at `off` in every rank's heap. Rank r owns elements [r*chunk, (r+1)*chunk): it reads that range
// from every peer, sums, and writes the result back into every peer's buffer.
// U vectors per thread and iteration (U * world 16-byte peer loads in flight per thread); see the launcher for the measured choice.
template <typename T, int U>
__global__ void __launch_bounds__(kThreads) allreduce_kernel(Peers P, int64_t off, int64_t n, int rank, int world,
                                                             uint32_t epoch, uint32_t* counter) {
  constexpr int N = Vec16<T>::N;
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);
  const int64_t nvec = n / N;
  const int64_t per = (nvec + world - 1) / world;
  const int64_t v0 = per * rank, v1 = min(nvec, v0 + per);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t vb = v0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; vb < v1; vb += stride * U) {
    Vec16<T> in[U][kMaxRanks];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = vb + u * stride;
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)
        if (r < world && v < v1) in[u][r] = ld16(reinterpret_cast<const T*>(P.base[r] + off) + v * N);   // all peer loads in flight
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = vb + u * stride;
      if (v >= v1) continue;
      float acc[N];
#pragma unroll
      for (int j = 0; j < N; ++j) acc[j] = 0.f;
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)
        if (r < world) {
#pragma unroll
          for (int j = 0; j < N; ++j) acc[j] += to_f(in[u][r].v[j]);
        }
      Vec16<T> o;
#pragma unroll
      for (int j = 0; j < N; ++j) o.v[j] = from_f<T>(acc[j]);
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)
        if (r < world) st16(reinterpret_cast<T*>(P.base[r] + off) + v * N, o);
    }
  }
  // scalar tail (n % N) handled by the last rank
  if (rank == world - 1 && blockIdx.x == 0) {
    for (int64_t i = nvec * N + threadIdx.x; i < n; i += blockDim.x) {
      float a = 0.f;
      for (int r = 0; r < world; ++r) a += to_f(reinterpret_cast<const T*>(P.base[r] + off)[i]);
      for (int r = 0; r < world; ++r) reinterpret_cast<T*>(P.base[r] + off)[i] = from_f<T>(a);
    }
  }
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// ---------------------------------------------------------------------------------------------- reduce-scatter
// input: n elements at `off` in every heap; rank r's output = sum over peers of elements [r*n/world, (r+1)*n/world)
template <typename T, int U>
__global__ void __launch_bounds__(kThreads) reduce_scatter_kernel(Peers P, int64_t off, T* __restrict__ out, int64_t n, int rank,
                                                                  int world, uint32_t epoch, uint32_t* counter) {
  constexpr int N = Vec16<T>::N;
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);
  const int64_t chunk = n / world;          // caller guarantees divisibility and chunk % N == 0
  const int64_t nvec = chunk / N;
  const int64_t base = chunk * rank;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t vb = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; vb < nvec; vb += stride * U) {
    Vec16<T> in[U][kMaxRanks];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = vb + u * stride;
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)
        if (r < world && v < nvec) in[u][r] = ld16(reinterpret_cast<const T*>(P.base[r] + off) + base + v * N);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = vb + u * stride;
      if (v >= nvec) continue;
      float acc[N];
#pragma unroll
      for (int j = 0; j < N; ++j) acc[j] = 0.f;
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)
        if (r < world) {
#pragma unroll
          for (int j = 0; j < N; ++j) acc[j] += to_f(in[u][r].v[j]);
        }
      Vec16<T> o;
#pragma unroll
      for (int j = 0; j < N; ++j) o.v[j] = from_f<T>(acc[j]);
      st16_stream(out + v * N, o);
    }
  }
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// ---------------------------------------------------------------------------------------------- reduce of pushed slots
// Tail of the fused GEMM -> reduce-scatter: every rank's GEMM epilogue has stored its partial rows for rank r into slot
// [src] of r's staging area (world slots of n elements at `off`).  Here rank r waits until all pushes have landed and
// sums its slots from LOCAL HBM (the NVLink traffic already happened, tile by tile, under the GEMM main loop).
template <typename T>
__global__ void __launch_bounds__(kThreads) reduce_slots_kernel(Peers P, int64_t off, T* __restrict__ out, int64_t n, int rank,
                                                                int world, uint32_t epoch, uint32_t* counter) {
  constexpr int N = Vec16<T>::N;
  if (blockIdx.x == 0) {
    __threadfence_system();
    signal_all(P, rank, world, 0, epoch);   // stream order: my GEMM (and its pushes) completed before this kernel started
  }
  wait_all(P, rank, world, 0, epoch);
  const T* base = reinterpret_cast<const T*>(P.base[rank] + off);
  const int64_t nvec = n / N;
  for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) {
    Vec16<T> in[kMaxRanks];
#pragma unroll
    for (int r = 0; r < kMaxRanks; ++r)
      if (r < world) in[r] = ld16(base + (int64_t)r * n + v * N);
    float acc[N];
#pragma unroll
    for (int j = 0; j < N; ++j) acc[j] = 0.f;
#pragma unroll
    for (int r = 0; r < kMaxRanks; ++r)
      if (r < world) {
#pragma unroll
        for (int j = 0; j < N; ++j) acc[j] += to_f(in[r].v[j]);
      }
    Vec16<T> o;
#pragma unroll
    for (int j = 0; j < N; ++j) o.v[j] = from_f<T>(acc[j]);
    st16_stream(out + v * N, o);
  }
  if (last_cta(counter)) {                  // peers may push the next GEMM into my slots only after I have read them
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// ---------------------------------------------------------------------------------------------- all-gather (pull)
// every rank has its shard at [rank*chunk, (rank+1)*chunk) of the buffer at `off`; pull the other shards from their owners.
__global__ void __launch_bounds__(kThreads) allgather_kernel(Peers P, int64_t off, int64_t chunk_bytes, int rank, int world,
                                                             uint32_t epoch, uint32_t* counter) {
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);
  const int64_t nvec = chunk_bytes / 16;
  for (int pr = 1; pr < world; ++pr) {
    const int src = (rank + pr) % world;  // stagger peers so the switch sees a permutation, not a hotspot
    const uint4* s = reinterpret_cast<const uint4*>(P.base[src] + off + chunk_bytes * src);
    uint4* d = reinterpret_cast<uint4*>(P.base[rank] + off + chunk_bytes * src);
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) d[v] = s[v];
  }
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// ---------------------------------------------------------------------------------------------- all-to-all (push)
// send buffer at off_send: world chunks of chunk_bytes (chunk d goes to rank d); recv buffer at off_recv: chunk s comes from rank s.
__global__ void __launch_bounds__(kThreads) alltoall_kernel(Peers P, int64_t off_send, int64_t off_recv, int64_t chunk_bytes, int rank,
                                                            int world, uint32_t epoch, uint32_t* counter) {
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);  // receivers' previous consumers are done (stream order on each rank + end barrier)
  const int64_t nvec = chunk_bytes / 16;
  for (int pr = 0; pr < world; ++pr) {
    const int dst = (rank + pr) % world;
    const uint4* s = reinterpret_cast<const uint4*>(P.base[rank] + off_send + chunk_bytes * dst);
    uint4* d = reinterpret_cast<uint4*>(P.base[dst] + off_recv + chunk_bytes * rank);
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) d[v] = s[v];
  }
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// ---------------------------------------------------------------------------------------------- MoE dispatch / combine
// Variable-size all-to-all with an optional row gather, fused into one push kernel (MoE expert dispatch: the routed copy
// x[tok] is never materialised; combine: gather == nullptr).  Parity (role): global_scatter / global_gather
// (paddle/fluid/operators/collective/global_scatter_op.cu.cc) which issue ncclSend/ncclRecv per (rank, expert).
//   src            local rows [*, row_bytes]
//   gather[i]      source row of sorted slot i (nullptr: slot i = row i)
//   meta_off       byte offset of a symmetric int64 [world] array: THIS rank stored its send counts there before the launch
//                  (send count to rank r = number of sorted slots destined to r; slots are grouped by destination rank)
//   recv_off       byte offset of the symmetric receive buffer; rank r's buffer is filled in source-rank order, so the rows
//                  this rank sends to r start at row sum_{s < me} count[s][r]  (read from the peers' meta arrays)
__global__ void __launch_bounds__(kThreads) a2av_kernel(Peers P, const char* __restrict__ src, const int64_t* __restrict__ gather,
                                                        int64_t meta_off, int64_t recv_off, int64_t row_bytes, int rank, int world,
                                                        uint32_t epoch, uint32_t* counter) {
  __shared__ int64_t seg_start[kMaxRanks + 1];   // first sorted slot going to rank r
  __shared__ int64_t dst_row0[kMaxRanks];        // first row of rank r's receive buffer reserved for this rank
  if (blockIdx.x == 0) {
    __threadfence_system();
    signal_all(P, rank, world, 0, epoch);        // my meta array is in place; my previous receive buffer has been consumed (stream order)
  }
  wait_all(P, rank, world, 0, epoch);
  if (threadIdx.x == 0) {
    const int64_t* mine = reinterpret_cast<const int64_t*>(P.base[rank] + meta_off);
    int64_t acc = 0;
    for (int r = 0; r < world; ++r) { seg_start[r] = acc; acc += mine[r]; }
    seg_start[world] = acc;
    for (int r = 0; r < world; ++r) {
      int64_t before = 0;
      for (int sr = 0; sr < rank; ++sr) before += reinterpret_cast<const volatile int64_t*>(P.base[sr] + meta_off)[r];
      dst_row0[r] = before;
    }
  }
  __syncthreads();
  const int64_t total = seg_start[world];
  const int vec_per_row = (int)(row_bytes / 16);
  const int warps = (gridDim.x * blockDim.x) >> 5;
  const int lane = threadIdx.x & 31;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < total; i += warps) {   // one warp per row
    int r = 0;
    while (i >= seg_start[r + 1]) ++r;
    const int64_t srow = gather ? gather[i] : i;
    const uint4* sp = reinterpret_cast<const uint4*>(src + srow * row_bytes);
    uint4* dp = reinterpret_cast<uint4*>(P.base[r] + recv_off + (dst_row0[r] + (i - seg_start[r])) * row_bytes);
    for (int v = lane; v < vec_per_row; v += 32) dp[v] = sp[v];
  }
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// ---------------------------------------------------------------------------------------------- gather-pull (sharded parameters)
// dst (ordinary local memory, [world, chunk_bytes]) <- every rank's `chunk_bytes` at byte offset src_off of ITS heap.  GroupSharded
// stage 3 keeps each rank's parameter shards in the symmetric heap; a layer's full weights are pulled straight into a fresh
// allocation that the layer's kernels then read (no staging window, no copy-out).
__global__ void __launch_bounds__(kThreads) gather_pull_kernel(Peers P, int64_t src_off, char* __restrict__ dst, int64_t chunk_bytes,
                                                               int rank, int world, uint32_t epoch, uint32_t* counter) {
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);
  const int64_t nvec = chunk_bytes / 16;
  const int64_t total = nvec * world;
  constexpr int U = 4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; base < total; base += stride * U) {
    uint4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = base + u * stride;
      if (i < total) {
        const int r = (int)(i / nvec);
        const int64_t j = i - (int64_t)r * nvec;
        v[u] = reinterpret_cast<const uint4*>(P.base[r] + src_off)[j];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = base + u * stride;
      if (i < total) reinterpret_cast<uint4*>(dst)[i] = v[u];
    }
  }
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

void p2p_gather_pull(const int64_t* bases, int64_t src_off, void* dst, int64_t chunk_bytes, int rank, int world, uint32_t epoch,
                     uint32_t* counter, cudaStream_t s) {
  if (world > kMaxRanks || chunk_bytes % 16 || src_off % 16 || (reinterpret_cast<uintptr_t>(dst) & 15)) {
    set_last_error(__FILE__, __LINE__, "p2p_gather_pull: bad world / alignment");
    return;
  }
  Peers P;
  for (int r = 0; r < kMaxRanks; ++r) P.base[r] = r < world ? reinterpret_cast<char*>(bases[r]) : nullptr;
  int64_t blocks = (chunk_bytes / 16 * world + kThreads * 4 - 1) / (kThreads * 4);
  const int grid = (int)(blocks < 1 ? 1 : (blocks > 96 ? 96 : blocks));
  gather_pull_kernel<<<grid, kThreads, 0, s>>>(P, src_off, static_cast<char*>(dst), chunk_bytes, rank, world, epoch, counter);
  B200_CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------- mailbox signal / wait
// Point-to-point "mailbox" used by the pipeline engine (distributed/fleet/pipeline.py): the producer copies a tensor into a slot
// of the consumer's heap with the copy engine (cudaMemcpyAsync on the IPC-mapped pointer: no SM work), then this one-thread kernel
// publishes the slot with a release store; the consumer's stream runs wait_flag_kernel before the first kernel that reads the
// slot.  The waiting thread accounts the time it spun into stats[0] (ns) / stats[1] (waits) = exposed pipeline wait on the device.
__global__ void signal_flag_kernel(uint32_t* remote_flag, uint32_t value) {
  __threadfence_system();
  ptx::st_release_sys_u32(remote_flag, value);
}

__global__ void wait_flag_kernel(const uint32_t* flag, uint32_t value, unsigned long long* stats, unsigned long long timeout_ns) {
  const uint64_t t0 = ptx::globaltimer_ns();
  while ((int32_t)(ptx::ld_acquire_sys_u32(flag) - value) < 0) {
    if (ptx::globaltimer_ns() - t0 > timeout_ns) {
      printf("b200 p2p mailbox: timeout waiting for flag value %u (have %u)\n", value, ptx::ld_acquire_sys_u32(flag));
      __trap();
    }
    __nanosleep(200);
  }
  if (stats) {
    atomicAdd(stats, (unsigned long long)(ptx::globaltimer_ns() - t0));
    atomicAdd(stats + 1, 1ull);
  }
}

void p2p_signal_flag(void* remote_flag, uint32_t value, cudaStream_t s) {
  signal_flag_kernel<<<1, 1, 0, s>>>(static_cast<uint32_t*>(remote_flag), value);
  B200_CUDA_CHECK(cudaGetLastError());
}

void p2p_wait_flag(const void* flag, uint32_t value, void* stats, double timeout_s, cudaStream_t s) {
  wait_flag_kernel<<<1, 1, 0, s>>>(static_cast<const uint32_t*>(flag), value, static_cast<unsigned long long*>(stats),
                                   (unsigned long long)(timeout_s * 1e9));
  B200_CUDA_CHECK(cudaGetLastError());
}

static Peers make_peers(const int64_t* bases, int world) {
  Peers P;
  for (int r = 0; r < kMaxRanks; ++r) P.base[r] = r < world ? reinterpret_cast<char*>(bases[r]) : nullptr;
  return P;
}

static int comm_grid(int64_t work_vecs) {
  // NVLink saturates with a fraction of the SMs; keep the rest free for overlapped compute
  int64_t blocks = (work_vecs + kThreads - 1) / kThreads;
  const int cap = 64;
  return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

void p2p_allreduce(const int64_t* bases, int64_t off, int64_t n, int dtype, int rank, int world, uint32_t epoch, uint32_t* counter,
                   cudaStream_t s) {
  if (world > kMaxRanks) { set_last_error(__FILE__, __LINE__, "p2p collectives support up to 8 ranks (one NVSwitch domain)"); return; }
  Peers P = make_peers(bases, world);
  B200_DISPATCH_DTYPE(dtype, T, {
    constexpr int N = Vec16<T>::N;
    // measured on 2 x B200 (6.5 GB slab): more peer loads in flight per thread (U = 4) was SLOWER (53.6 vs 29.3 ms) - the loop is bound by
    // the posted remote stores, not by load latency - so every world size keeps one vector per thread and iteration
    allreduce_kernel<T, 1><<<comm_grid(n / N / world + 1), kThreads, 0, s>>>(P, off, n, rank, world, epoch, counter);
  });
  B200_CUDA_CHECK(cudaGetLastError());
}

void p2p_reduce_scatter(const int64_t* bases, int64_t off, void* out, int64_t n, int dtype, int rank, int world, uint32_t epoch,
                        uint32_t* counter, cudaStream_t s) {
  if (world > kMaxRanks) { set_last_error(__FILE__, __LINE__, "p2p collectives support up to 8 ranks"); return; }
  Peers P = make_peers(bases, world);
  B200_DISPATCH_DTYPE(dtype, T, {
    constexpr int N = Vec16<T>::N;
    if (n % world || (n / world) % N) { set_last_error(__FILE__, __LINE__, "p2p_reduce_scatter: n/world must be a multiple of the 16B vector"); return; }
    const int grid = comm_grid(n / world / N);
    if (world <= 2) reduce_scatter_kernel<T, 4><<<grid, kThreads, 0, s>>>(P, off, (T*)out, n, rank, world, epoch, counter);
    else if (world <= 4) reduce_scatter_kernel<T, 2><<<grid, kThreads, 0, s>>>(P, off, (T*)out, n, rank, world, epoch, counter);
    else reduce_scatter_kernel<T, 1><<<grid, kThreads, 0, s>>>(P, off, (T*)out, n, rank, world, epoch, counter);
  });
  B200_CUDA_CHECK(cudaGetLastError());
}

void p2p_reduce_slots(const int64_t* bases, int64_t off, void* out, int64_t n, int dtype, int rank, int world, uint32_t epoch,
                      uint32_t* counter, cudaStream_t s) {
  if (world > kMaxRanks) { set_last_error(__FILE__, __LINE__, "p2p collectives support up to 8 ranks"); return; }
  Peers P = make_peers(bases, world);
  B200_DISPATCH_DTYPE(dtype, T, {
    constexpr int N = Vec16<T>::N;
    if (n % N) { set_last_error(__FILE__, __LINE__, "p2p_reduce_slots: slot size must be a multiple of the 16B vector"); return; }
    // purely local HBM traffic (the NVLink part happened in the GEMM epilogue): use the whole machine, not the comm-sized grid
    int64_t blocks = (n / N + kThreads * 4 - 1) / (kThreads * 4);
    const int cap = sm_count() * 4;
    const int grid = (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
    reduce_slots_kernel<T><<<grid, kThreads, 0, s>>>(P, off, (T*)out, n, rank, world, epoch, counter);
  });
  B200_CUDA_CHECK(cudaGetLastError());
}

void p2p_allgather(const int64_t* bases, int64_t off, int64_t chunk_bytes, int rank, int world, uint32_t epoch, uint32_t* counter,
                   cudaStream_t s) {
  if (world > kMaxRanks || chunk_bytes % 16) { set_last_error(__FILE__, __LINE__, "p2p_allgather: bad world/chunk"); return; }
  Peers P = make_peers(bases, world);
  allgather_kernel<<<comm_grid(chunk_bytes / 16), kThreads, 0, s>>>(P, off, chunk_bytes, rank, world, epoch, counter);
  B200_CUDA_CHECK(cudaGetLastError());
}

void p2p_alltoall(const int64_t* bases, int64_t off_send, int64_t off_recv, int64_t chunk_bytes, int rank, int world, uint32_t epoch,
                  uint32_t* counter, cudaStream_t s) {
  if (world > kMaxRanks || chunk_bytes % 16) { set_last_error(__FILE__, __LINE__, "p2p_alltoall: bad world/chunk"); return; }
  Peers P = make_peers(bases, world);
  alltoall_kernel<<<comm_grid(chunk_bytes / 16), kThreads, 0, s>>>(P, off_send, off_recv, chunk_bytes, rank, world, epoch, counter);
  B200_CUDA_CHECK(cudaGetLastError());
}

void p2p_a2av(const int64_t* bases, const void* src, const int64_t* gather, int64_t meta_off, int64_t recv_off, int64_t row_bytes,
              int64_t rows_hint, int rank, int world, uint32_t epoch, uint32_t* counter, cudaStream_t s) {
  if (world > kMaxRanks || row_bytes % 16) { set_last_error(__FILE__, __LINE__, "p2p_a2av: bad world / row size"); return; }
  Peers P = make_peers(bases, world);
  a2av_kernel<<<comm_grid(rows_hint * 32), kThreads, 0, s>>>(P, (const char*)src, gather, meta_off, recv_off, row_bytes, rank, world, epoch, counter);
  B200_CUDA_CHECK(cudaGetLastError());
}

}  // namespace comm
}  // namespace b200
