// Data-parallel exchange over NVLink peer memory (SURVEY.md 8e): buffer layout, arguments and protocol.  Host side:
// pinn_dp.cu.  Callers: the reduction (pinn_reduce.cu) and the sampler (pinn_sample.cuh).
// Every rank owns one exchange buffer that all peers of the box can write (cudaIpc / peer access).  A 64-bit value travels
// as a word pair: two 8-byte words {32 data bits, 32-bit step number}.  8-byte stores are single-copy atomic, so a reader
// that sees this exchange's step number in both words has the value - no fence, no separate flag, one NVLink one-way
// latency.  Rank r writes slot r of every peer's buffer; the values are added in rank order, so every
// rank computes bit-identical sums.  Two slot sets alternate by step parity: a peer can be at most one exchange ahead.
//   rows [2 parities][DP_MAX_WORLD][NPART] word pairs (dp_row) | ctl DP_CTL_SLOTS x u64 (dp_ctl, DpCtl)
//   cnt  [2 parities][DP_MAX_WORLD] word pairs: the sampler's two set sizes (dp_cnt)
#pragma once
#include "pinn_common.cuh"

namespace pinn {

constexpr int DP_MAX_WORLD = 8;
// How long a rank polls for a peer's contribution before it declares the run failed (SM cycles, ~30 s): long enough for any
// host-side skew between the ranks' launches (one rank writing a checkpoint, drawing a batch on the CPU ...), short
// enough that a dead peer does not hang the GPU.
constexpr long long DP_TIMEOUT_CYCLES = 60000000000ll;

struct DpArgs {
  int world = 0;  // <= 1: no exchange
  int rank = 0;
  unsigned char* peer[DP_MAX_WORLD] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // exchange buffers, [rank] = own
  long long timeout_cycles = DP_TIMEOUT_CYCLES;  // pinn_dp_set_timeout
};

// Control slots: reduction exchanges completed on this rank, blocks of the current one done, failed (a peer did not
// deliver in time: set in every rank's buffer, and stays set), sampler set-size exchanges completed.
enum DpCtl { DP_EXCHANGES, DP_BLOCKS_DONE, DP_FAILED, DP_COUNT_EXCHANGES };
constexpr int DP_CTL_SLOTS = 8;
constexpr size_t DP_ROWS_BYTES = 2ull * DP_MAX_WORLD * NPART * 16;
constexpr size_t DP_CTL_BYTES = DP_CTL_SLOTS * 8;
constexpr size_t DP_BUFFER_BYTES = DP_ROWS_BYTES + DP_CTL_BYTES + 2ull * DP_MAX_WORLD * 16;

// the word pair of entry `entry` of rank `rank` in exchange `step` / of rank `rank`'s set sizes in set-size exchange `step`
__host__ __device__ inline unsigned int* dp_row(unsigned char* buf, unsigned int step, int rank, int entry) {
  return reinterpret_cast<unsigned int*>(buf) + (((size_t)(step & 1u) * DP_MAX_WORLD + rank) * NPART + entry) * 4;
}
__host__ __device__ inline unsigned int* dp_cnt(unsigned char* buf, unsigned int step, int rank) {
  return reinterpret_cast<unsigned int*>(buf + DP_ROWS_BYTES + DP_CTL_BYTES) + ((size_t)(step & 1u) * DP_MAX_WORLD + rank) * 4;
}
__host__ __device__ inline unsigned long long* dp_ctl(unsigned char* buf) {
  return reinterpret_cast<unsigned long long*>(buf + DP_ROWS_BYTES);
}

// system-scope accesses (peer memory over NVLink)
__device__ __forceinline__ void st_relaxed_sys_v2(unsigned int* p, unsigned int a, unsigned int b) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ uint2 ld_relaxed_sys_v2(const unsigned int* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// this rank's control slots: has an earlier exchange of the run failed; the step number of the next exchange of a kind
// (DP_EXCHANGES or DP_COUNT_EXCHANGES); exchange `step` of a kind is complete
__device__ __forceinline__ bool dp_has_failed(const DpArgs& dp) {
  return ld_acquire_sys(dp_ctl(dp.peer[dp.rank]) + DP_FAILED) != 0ull;
}
__device__ __forceinline__ unsigned long long dp_next_step(const DpArgs& dp, DpCtl kind) {
  return ld_acquire_sys(dp_ctl(dp.peer[dp.rank]) + kind) + 1;
}
__device__ __forceinline__ void dp_complete(const DpArgs& dp, DpCtl kind, unsigned long long step) {
  st_release_sys(dp_ctl(dp.peer[dp.rank]) + kind, step);
}
// Run by one thread of each of the `blocks` exchanging blocks of a reduction, after its block has received: the last one
// completes exchange `step` (the next launch is stream-ordered behind it).
__device__ __forceinline__ void dp_block_done(const DpArgs& dp, unsigned long long step, int blocks) {
  unsigned long long* ctl = dp_ctl(dp.peer[dp.rank]);
  __threadfence();
  if (atomicAdd(&ctl[DP_BLOCKS_DONE], 1ull) == (unsigned long long)blocks - 1) {
    ctl[DP_BLOCKS_DONE] = 0ull;
    dp_complete(dp, DP_EXCHANGES, step);
  }
}

// Stores v as the word pair of exchange `step` at dst (a slot of a peer's buffer).
__device__ __forceinline__ void dp_send(unsigned int* dst, unsigned long long v, unsigned int step) {
  st_relaxed_sys_v2(dst, (unsigned int)v, step);
  st_relaxed_sys_v2(dst + 2, (unsigned int)(v >> 32), step);
}
// Polls the word pair at src (a slot of this rank's buffer) until both words carry `step`: true, with the value in v.
// False at once while `stop` is set.  A peer that has not delivered within dp.timeout_cycles fails the run: DP_FAILED is
// set in every rank's buffer (the peers stop updating their replicas as well) and so is `stop`; false.
template <typename Flag>
__device__ __forceinline__ bool dp_recv(const DpArgs& dp, const unsigned int* src, unsigned int step, Flag& stop,
                                        unsigned long long& v) {
  const long long t0 = clock64();
  while (!stop) {
    const uint2 lo = ld_relaxed_sys_v2(src), hi = ld_relaxed_sys_v2(src + 2);
    if (lo.y == step && hi.y == step) {
      v = ((unsigned long long)hi.x << 32) | lo.x;
      return true;
    }
    if (clock64() - t0 > dp.timeout_cycles) {
      for (int q = 0; q < dp.world; q++) st_release_sys(dp_ctl(dp.peer[q]) + DP_FAILED, 1ull);
      stop = 1;
      return false;
    }
  }
  return false;
}

}  // namespace pinn
