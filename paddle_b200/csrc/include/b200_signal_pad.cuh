// Cross-rank barriers on signal pads, shared by the peer-memory (p2p) and NVLink SHARP (nvls) collectives.
//
// Every rank owns a pad row of uint32 flags, pad[slot * kPadRanks + src], in memory its peers can write.  Rank src publishes an epoch
// in slot `slot` of rank r's row with a release store (signal_all); r waits until its own row holds that epoch from every peer
// (wait_all).  Epochs only grow, so a wait is a spin on ">= epoch", bounded by the protocol's timeout: a dead peer or a protocol bug
// traps instead of hanging the GPU.
#pragma once
#include <cstdint>
#include <cstdio>

#include "b200_ptx.cuh"

// Timeout message of wait_all.  `label` (a string literal) names the protocol, so that a trap says which one stalled; the message
// receives the rank, the peer waited for, the slot, the epoch and the value seen.
#define B200_PAD_TIMEOUT(label) "b200 " label ": barrier timeout rank %d waiting for %d slot %d epoch %u (have %u)\n"

namespace b200 {
namespace pad {

constexpr int kPadRanks = 8;

// Thread `src` < world of the CTA publishes `epoch` in slot `slot` of peer src's row (the entry of this rank).
__device__ __forceinline__ void signal_all(uint32_t* const* pads, int rank, int world, int slot, uint32_t epoch) {
  if ((int)threadIdx.x < world && (int)threadIdx.x != rank) ptx::st_release_sys_u32(pads[threadIdx.x] + slot * kPadRanks + rank, epoch);
}

// All threads of the CTA return once every peer has published `epoch` in slot `slot` of this rank's row.  A peer still missing after
// `timeout_ns` makes the waiting thread print `timeout_fmt` (built with B200_PAD_TIMEOUT) and trap.
__device__ __forceinline__ void wait_all(uint32_t* const* pads, int rank, int world, int slot, uint32_t epoch, uint64_t timeout_ns,
                                         const char* timeout_fmt) {
  if ((int)threadIdx.x < world && (int)threadIdx.x != rank) {
    const uint32_t* f = pads[rank] + slot * kPadRanks + threadIdx.x;
    // ptx::spin_sys_ge, written out: the timeout message shows the flag value seen at that moment
    const uint64_t t0 = ptx::globaltimer_ns();
    while ((int32_t)(ptx::ld_acquire_sys_u32(f) - epoch) < 0) {
      if (ptx::globaltimer_ns() - t0 > timeout_ns) {
        printf(timeout_fmt, rank, (int)threadIdx.x, slot, epoch, ptx::ld_acquire_sys_u32(f));
        __trap();
      }
    }
  }
  __syncthreads();
}

// Grid-wide completion: returns true in the last CTA to arrive.
__device__ __forceinline__ bool last_cta(uint32_t* counter) {
  __shared__ bool is_last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t prev = atomicAdd(counter, 1u);
    is_last = (prev == gridDim.x - 1);
    if (is_last) *counter = 0;  // reset for the next launch (stream-ordered)
  }
  __syncthreads();
  return is_last;
}

}  // namespace pad
}  // namespace b200
