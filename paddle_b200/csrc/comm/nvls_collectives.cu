// NVLS (NVLink SHARP) collectives: the reduction / broadcast happens INSIDE the NVSwitch through a multicast address.
//
//   all-reduce      rank r owns slice r of the buffer: `multimem.ld_reduce` on the multicast address returns the sum over every GPU's copy
//                   (one request, the switch reads all replicas and adds), `multimem.st` writes the result to every replica (one store,
//                   replicated by the switch).  Per GPU: n/world loads + n/world stores on the wire, against (world-1)/world * n * 2 for
//                   the peer-memory two-shot in p2p_collectives.cu.
//   reduce-scatter  the ld_reduce half, result to ordinary local memory.
//   all-gather      the multimem.st half: every rank broadcasts its chunk into slot `rank` of every replica.
//
// Memory plumbing (multicast object, binding, handle exchange) is torch.distributed._symmetric_memory's; the kernels get the multicast
// pointer, the local replica pointer and every rank's signal pad.  Cross-rank barriers are the epoch protocol of the p2p collectives
// (include/b200_signal_pad.cuh) on two slots at the END of the signal pads (the front belongs to torch's own barrier channels).
//
// Status: compiled for sm_100a (SASS holds the multimem instructions); NOT yet run on hardware - opt-in behind FLAGS_b200_nvls.
// Parity (role): NCCL's NVLS algorithm under ProcessGroupNCCL::AllReduce (paddle/fluid/distributed/collective/process_group_nccl.cc).
#include <cstdio>

#include "../include/b200_common.cuh"
#include "../include/b200_comm.h"
#include "../include/b200_signal_pad.cuh"

namespace b200 {
namespace comm {

namespace {
constexpr int kMaxRanks = 8;
constexpr int kThreads = 512;
constexpr uint64_t kBarrierTimeoutNs = 10000000000ull;   // 10 s: a dead peer or a protocol bug traps instead of hanging the GPU

struct NvlsPeers {
  uint32_t* pad[kMaxRanks];      // our two barrier rows inside every rank's signal pad: pad[r][slot * kMaxRanks + src]
  char* mc;                      // multicast address of the symmetric buffer
  char* local;                   // this rank's replica
};

__device__ __forceinline__ void signal_all(const NvlsPeers& P, int rank, int world, int slot, uint32_t epoch) {
  pad::signal_all(P.pad, rank, world, slot, epoch);
}
__device__ __forceinline__ void wait_all(const NvlsPeers& P, int rank, int world, int slot, uint32_t epoch) {
  pad::wait_all(P.pad, rank, world, slot, epoch, kBarrierTimeoutNs, B200_PAD_TIMEOUT("nvls"));
}
using pad::last_cta;

// 16 bytes reduced across every replica by the switch (fp32 accumulation for the 16-bit types)
template <typename T> struct Mm;
template <> struct Mm<float> {
  static __device__ __forceinline__ uint4 ld_reduce(const void* mc) {
    uint4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
    return v;
  }
};
template <> struct Mm<__nv_bfloat16> {
  static __device__ __forceinline__ uint4 ld_reduce(const void* mc) {
    uint4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
    return v;
  }
};
template <> struct Mm<__half> {
  static __device__ __forceinline__ uint4 ld_reduce(const void* mc) {
    uint4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.f16x2 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
    return v;
  }
};
// 16 bytes written to every replica with one store
__device__ __forceinline__ void mm_st(void* mc, const uint4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// mode 0: all-reduce in place (every replica ends with the sum); mode 1: reduce-scatter (slice `rank` of the sum -> out)
template <typename T, int MODE>
__global__ void __launch_bounds__(kThreads) nvls_reduce_kernel(NvlsPeers P, int64_t off, T* __restrict__ out, int64_t n, int rank, int world, uint32_t epoch,
                                                               uint32_t* counter) {
  constexpr int N = 16 / sizeof(T);
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);                      // every rank's input is in its replica
  const int64_t nvec = n / N;
  const int64_t per = (nvec + world - 1) / world;
  const int64_t v0 = per * rank, v1 = min(nvec, v0 + per);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v = v0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < v1; v += stride) {
    char* a = P.mc + off + v * 16;
    const uint4 s = Mm<T>::ld_reduce(a);
    if (MODE == 0) mm_st(a, s);
    else reinterpret_cast<uint4*>(out)[v - v0] = s;
  }
  if (last_cta(counter)) {                                  // this rank is done reading (and, for the all-reduce, writing) every replica
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

// slot `rank` (chunk_bytes, multiple of 16) of every replica <- src
__global__ void __launch_bounds__(kThreads) nvls_allgather_kernel(NvlsPeers P, int64_t off, const char* __restrict__ src, int64_t chunk_bytes, int rank, int world,
                                                                  uint32_t epoch, uint32_t* counter) {
  if (blockIdx.x == 0) signal_all(P, rank, world, 0, epoch);
  wait_all(P, rank, world, 0, epoch);                      // nobody is still reading the buffer from the previous use
  const int64_t nvec = chunk_bytes / 16;
  char* dst = P.mc + off + (int64_t)rank * chunk_bytes;
  for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x)
    mm_st(dst + v * 16, reinterpret_cast<const uint4*>(src)[v]);
  if (last_cta(counter)) {
    signal_all(P, rank, world, 1, epoch);
    wait_all(P, rank, world, 1, epoch);
  }
}

NvlsPeers make_peers(const int64_t* pads, int64_t pad_off, int64_t mc, int64_t local, int world) {
  NvlsPeers P{};
  for (int r = 0; r < world; ++r) P.pad[r] = reinterpret_cast<uint32_t*>(pads[r] + pad_off);
  P.mc = reinterpret_cast<char*>(mc);
  P.local = reinterpret_cast<char*>(local);
  return P;
}

int grid_for(int64_t nvec_per_rank) {
  const int64_t want = (nvec_per_rank + kThreads - 1) / kThreads;
  return (int)std::max<int64_t>(1, std::min<int64_t>(want, 64));        // the switch, not the SMs, does the arithmetic: 64 CTAs keep the links busy
}
}  // namespace

// dtype: 0 fp32, 1 bf16, 2 fp16.  n must be a multiple of 16 bytes worth of elements; `off` a multiple of 16.
void nvls_allreduce(const int64_t* pads, int64_t pad_off, int64_t mc, int64_t local, int64_t off, int64_t n, int dtype, int rank, int world, uint32_t epoch,
                    uint32_t* counter, cudaStream_t s) {
  const NvlsPeers P = make_peers(pads, pad_off, mc, local, world);
  const int64_t nvec = n / (dtype == 0 ? 4 : 8);
  const int g = grid_for((nvec + world - 1) / world);
  if (dtype == 0) nvls_reduce_kernel<float, 0><<<g, kThreads, 0, s>>>(P, off, nullptr, n, rank, world, epoch, counter);
  else if (dtype == 1) nvls_reduce_kernel<__nv_bfloat16, 0><<<g, kThreads, 0, s>>>(P, off, nullptr, n, rank, world, epoch, counter);
  else nvls_reduce_kernel<__half, 0><<<g, kThreads, 0, s>>>(P, off, nullptr, n, rank, world, epoch, counter);
}

void nvls_reduce_scatter(const int64_t* pads, int64_t pad_off, int64_t mc, int64_t local, int64_t off, void* out, int64_t n, int dtype, int rank, int world,
                         uint32_t epoch, uint32_t* counter, cudaStream_t s) {
  const NvlsPeers P = make_peers(pads, pad_off, mc, local, world);
  const int64_t nvec = n / (dtype == 0 ? 4 : 8);
  const int g = grid_for((nvec + world - 1) / world);
  if (dtype == 0) nvls_reduce_kernel<float, 1><<<g, kThreads, 0, s>>>(P, off, (float*)out, n, rank, world, epoch, counter);
  else if (dtype == 1) nvls_reduce_kernel<__nv_bfloat16, 1><<<g, kThreads, 0, s>>>(P, off, (__nv_bfloat16*)out, n, rank, world, epoch, counter);
  else nvls_reduce_kernel<__half, 1><<<g, kThreads, 0, s>>>(P, off, (__half*)out, n, rank, world, epoch, counter);
}

void nvls_allgather(const int64_t* pads, int64_t pad_off, int64_t mc, int64_t local, int64_t off, const void* src, int64_t chunk_bytes, int rank, int world,
                    uint32_t epoch, uint32_t* counter, cudaStream_t s) {
  const NvlsPeers P = make_peers(pads, pad_off, mc, local, world);
  nvls_allgather_kernel<<<grid_for(chunk_bytes / 16), kThreads, 0, s>>>(P, off, (const char*)src, chunk_bytes, rank, world, epoch, counter);
}

}  // namespace comm
}  // namespace b200
