// Collocation sampler + clamp + boundary sets (train.py:26-39; poc/main.py:124-156, 390-393) as device code shared by
// sample_kernel (pinn_train.cu) and by the sampler blocks that ride in the reduction kernel of the previous step
// (pinn_reduce.cu: the batch of step t+1 is drawn while step t is reduced).
#pragma once
#include "pinn_device.cuh"
#include "pinn_train.h"

namespace pinn {

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11): counter (c0..c3), key (k0,k1) -> 4 x 32 random bits
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-08f; }  // [0,1), 24 bits

// weights {1/n, 1/|set1|, 1/|set2|} of the reference's means (empty set -> inf -> NaN loss, as in the reference),
// and the batch counter moves on.  Run by one warp of the block of sample_kernel that finishes last.  Data-parallel runs
// (dp.world > 1) first add the set sizes of all ranks: lane r sends this rank's two counts (32 bits each) to peer r and
// receives peer r's (pinn_dp.cuh), lane 0 adds them in rank order.
__device__ __forceinline__ void sample_finish(const SampleParams& s) {
  __shared__ unsigned long long c[DP_MAX_WORLD][2];
  const DpArgs& dp = s.dp;
  const int lane = threadIdx.x;
  const long long n = s.n;
  double* w = s.weights;
  unsigned long long c1 = atomicAdd(&s.counts[0], 0ull), c2 = atomicAdd(&s.counts[1], 0ull);  // L2 values of the other blocks' atomics
  long long ntot = n;
  if (dp.world > 1) {
    const unsigned long long step64 = dp_next_step(dp, DP_COUNT_EXCHANGES);
    const unsigned int step = (unsigned int)step64;
    if (lane < dp.world) {
      const int r = lane;
      if (r == dp.rank) {
        c[r][0] = c1; c[r][1] = c2;
      } else {
        dp_send(dp_cnt(dp.peer[r], step, dp.rank), (c2 << 32) | (unsigned int)c1, step);
        // an earlier exchange of this run already failed (a peer never delivered): do not wait again
        bool failed = dp_has_failed(dp);
        unsigned long long v = 0;
        const bool ok = dp_recv(dp, dp_cnt(dp.peer[dp.rank], step, r), step, failed, v);
        c[r][0] = ok ? (unsigned int)v : 0ull; c[r][1] = ok ? v >> 32 : 0ull;
      }
    }
    __syncwarp();
    if (lane == 0) {
      c1 = 0; c2 = 0;
      for (int r = 0; r < dp.world; r++) { c1 += c[r][0]; c2 += c[r][1]; }
      ntot = n * dp.world;
      dp_complete(dp, DP_COUNT_EXCHANGES, step64);
    }
  }
  if (lane == 0) {
    w[0] = 1.0 / (double)ntot;
    w[1] = 1.0 / (double)c1;
    w[2] = 1.0 / (double)c2;
    *s.batch_counter += 1ull;
    *s.ticket = 0ull;
    if (s.reset_counts) { s.counts[0] = 0ull; s.counts[1] = 0ull; }
  }
}

// One thread per point.  Point i of batch b uses counter (i_lo, i_hi, b_lo, b_hi) and key = seed; its four words give
// x, y, z, R.  Clamp and sets follow the reference literally: both tests use the radii of the UN-clamped point
// (train.py:32-35), the clamp writes the VALUE `cutoff` into x, and the sets are taken after it (train.py:36-39).
// Work of block `block` of `nblocks` sampler blocks (any block size that is a multiple of 32, at most 1024 threads).
__device__ __forceinline__ void sample_block(const SampleParams& s, int block, int nblocks) {
  const unsigned long long batch = *s.batch_counter;
  unsigned c1 = 0, c2 = 0;
  for (long long i = (long long)block * blockDim.x + threadIdx.x; i < s.n; i += (long long)nblocks * blockDim.x) {
    uint32_t r[4];
    const unsigned long long gi = (unsigned long long)(i + s.index_offset);  // index of the point in the global batch
    philox4x32_10((uint32_t)gi, (uint32_t)(gi >> 32), (uint32_t)batch, (uint32_t)(batch >> 32),
                  (uint32_t)s.seed, (uint32_t)(s.seed >> 32), r);
    float x = fmaf(s.xR - s.xL, u01(r[0]), s.xL);
    const float y = fmaf(s.yR - s.yL, u01(r[1]), s.yL);
    const float z = fmaf(s.zR - s.zL, u01(r[2]), s.zL);
    const float R = fmaf(s.RR - s.RL, u01(r[3]), s.RL);
    const float yz = fmaf(y, y, z * z);
    const float c2cut = s.cutoff * s.cutoff;
    const bool near1 = fmaf(x - R, x - R, yz) < c2cut, near2 = fmaf(x + R, x + R, yz) < c2cut;
    if (near1 || near2) x = s.cutoff;
    const float b2 = s.bcutoff * s.bcutoff;
    const unsigned m1 = fmaf(x - R, x - R, yz) >= b2, m2 = fmaf(x + R, x + R, yz) >= b2;
    s.x[i] = x; s.y[i] = y; s.z[i] = z; s.R[i] = R;
    s.mask[i] = (uint8_t)(m1 | (m2 << 1));
    c1 += m1; c2 += m2;
  }
  c1 = __reduce_add_sync(0xffffffffu, c1);
  c2 = __reduce_add_sync(0xffffffffu, c2);
  __shared__ unsigned sh1[32], sh2[32];
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { sh1[w] = c1; sh2[w] = c2; }
  __syncthreads();
  __shared__ int last_block;
  if (threadIdx.x == 0) {
    unsigned t1 = 0, t2 = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) { t1 += sh1[k]; t2 += sh2[k]; }
    atomicAdd(&s.counts[0], (unsigned long long)t1);  // integer atomics: order-independent result
    atomicAdd(&s.counts[1], (unsigned long long)t2);
    __threadfence();
    last_block = atomicAdd(s.ticket, 1ull) == (unsigned long long)nblocks - 1;
  }
  __syncthreads();
  if (last_block && threadIdx.x < 32) sample_finish(s);  // every other block has added its counts and read the batch index
}

}  // namespace pinn
