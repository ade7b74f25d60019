// Residual-adaptive collocation (RAD; Wu, Zhu, Tan, Kartha & Lu, CMAME 403, 2023): the batch of a step is drawn from a
// pool of uniform candidates with probability proportional to w_i = |res_i|^k * N / sum_j |res_j|^k + c, by systematic
// resampling over the inclusive prefix sum of w.  Four launches on top of the pool draw and the pool's residual:
//   rad_sum_kernel     q_i = |res_i|^k, one float64 sum per block of RAD_TILE points
//   rad_scan_kernel    Q (the block sums folded in one fixed order), w_i and its prefix sum inside the block; the block
//                      finishing last folds the block totals into the block offsets (sequentially) and draws u0
//   rad_offset_kernel  cdf = block offset + in-block prefix
//   rad_select_kernel  output j takes the first i with cdf[i] > (j + u0) / n * cdf[N-1]; gather, set sizes, loss weights
//                      (importance mode: also omega_j = T / (N w_i), from w_i formed again exactly as the scan formed it)
// Every sum has a fixed association order and there are no floating-point atomics, so cdf and the selection are the same
// bits on every run.  Each partial prefix is a sequential fold, cdf[i+1] = fl(.. + w_i+1) with w >= 0 across every block
// and thread boundary too, so cdf never decreases and a binary search finds the first index the rule names.
#include "pinn_device.cuh"
#include "pinn_sample.cuh"
#include "pinn_train.h"

namespace pinn {

constexpr int RAD_THREADS = 256, RAD_PER_THREAD = 16, RAD_TILE = RAD_THREADS * RAD_PER_THREAD;

long long adaptive_scratch_doubles(long long pool) {
  const long long blocks = (pool + RAD_TILE - 1) / RAD_TILE;
  return 3 * blocks + 3;  // block sums of q, block totals of w, block offsets + total, u0, Q
}

__device__ __forceinline__ double rad_q(float r, double k) {
  return isfinite(r) ? pow(fabs((double)r), k) : 0.0;
}

// sum over the block in a fixed order: each thread's value, a butterfly inside every warp, the warps in order
__device__ __forceinline__ double rad_block_sum(double v) {
  __shared__ double wsum[RAD_THREADS / 32];
  __shared__ double total;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = wsum[0];
    for (int w = 1; w < RAD_THREADS / 32; w++) s += wsum[w];
    total = s;
  }
  __syncthreads();
  return total;
}

__global__ void __launch_bounds__(RAD_THREADS) rad_sum_kernel(const AdaptiveParams a) {
  pdl_wait();
  const long long i0 = (long long)blockIdx.x * RAD_TILE + (long long)threadIdx.x * RAD_PER_THREAD;
  double s = 0.0;
  for (int e = 0; e < RAD_PER_THREAD; e++)
    if (i0 + e < a.pool) s += rad_q(a.res[i0 + e], a.k);
  s = rad_block_sum(s);
  if (threadIdx.x == 0) a.part[blockIdx.x] = s;
  if (blockIdx.x == 0 && threadIdx.x == 0) {  // the selection's set sizes and block ticket start from zero
    a.out.counts[0] = 0ull; a.out.counts[1] = 0ull; *a.out.ticket = 0ull;
  }
}

// off[0] = 0, off[t + 1] = off[t] + v[t] for t < RAD_THREADS: one thread, a sequential fold (two arrays, so that the loads
// run ahead of the dependent adds)
__device__ __forceinline__ void rad_fold(const double* v, double* off, double start) {
  double s = start;
  off[0] = s;
#pragma unroll 16
  for (int t = 0; t < RAD_THREADS; t++) {
    s += v[t];
    off[t + 1] = s;
  }
}

__global__ void __launch_bounds__(RAD_THREADS) rad_scan_kernel(const AdaptiveParams a) {
  __shared__ double tot[RAD_THREADS], off[RAD_THREADS + 1];
  __shared__ int last_block;
  pdl_wait();
  const int nb = gridDim.x;
  const double* qsum = a.part;
  double* wtot = a.part + nb;
  double* boff = a.part + 2 * nb;
  double qs = 0.0;
  for (int b = threadIdx.x; b < nb; b += RAD_THREADS) qs += qsum[b];
  const double Q = rad_block_sum(qs);  // every block folds the same values in the same order: the same Q
  const bool uniform = !(Q > 0.0 && isfinite(Q));
  const double N = (double)a.pool;
  const long long i0 = (long long)blockIdx.x * RAD_TILE + (long long)threadIdx.x * RAD_PER_THREAD;
  double run[RAD_PER_THREAD];
  double acc = 0.0;
#pragma unroll
  for (int e = 0; e < RAD_PER_THREAD; e++) {
    double w = 0.0;
    if (i0 + e < a.pool) w = uniform ? 1.0 : rad_q(a.res[i0 + e], a.k) * N / Q + a.c;
    acc += w;  // 0 + w_0 = w_0 exactly
    run[e] = acc;
  }
  tot[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) rad_fold(tot, off, 0.0);  // sequential: a thread's first prefix is never below the last one before it
  __syncthreads();
  const double o = off[threadIdx.x];
#pragma unroll
  for (int e = 0; e < RAD_PER_THREAD; e++)
    if (i0 + e < a.pool) a.cdf[i0 + e] = o + run[e];
  if (threadIdx.x == 0) {
    wtot[blockIdx.x] = off[RAD_THREADS];
    __threadfence();
    last_block = atomicAdd(a.out.ticket, 1ull) == (unsigned long long)nb - 1;
  }
  __syncthreads();
  if (!last_block) return;
  // the block offsets, a sequential fold of the block totals, RAD_THREADS at a time through shared memory
  __threadfence();
  double s = 0.0;
  for (int b0 = 0; b0 < nb; b0 += RAD_THREADS) {
    const int b = b0 + threadIdx.x;
    tot[threadIdx.x] = b < nb ? *(volatile const double*)&wtot[b] : 0.0;
    __syncthreads();
    if (threadIdx.x == 0) {
      rad_fold(tot, off, s);
      s = off[RAD_THREADS];
    }
    __syncthreads();
    if (b < nb) boff[b] = off[threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    boff[nb] = s;  // the total; the padding of the last group adds exact zeros
    // u0: word 0 of Philox4x32-10 at counter {N, batch of the pool}, the point just past the pool in its own stream
    const unsigned long long batch = *a.pool_batch - 1ull;  // the pool's draw moved the counter on
    const unsigned long long gi = (unsigned long long)a.pool;
    uint32_t r[4];
    philox4x32_10((uint32_t)gi, (uint32_t)(gi >> 32), (uint32_t)batch, (uint32_t)(batch >> 32), (uint32_t)a.out.seed,
                  (uint32_t)(a.out.seed >> 32), r);
    boff[nb + 1] = (double)r[0] * 2.3283064365386963e-10;  // 2^-32
    boff[nb + 2] = Q;  // the importance weights form w_i again from it
    *a.out.ticket = 0ull;
  }
}

__global__ void __launch_bounds__(RAD_THREADS) rad_offset_kernel(const AdaptiveParams a) {
  pdl_wait();
  if (blockIdx.x == 0) return;  // block 0's in-block prefix is already the cdf
  const double o = a.part[2 * gridDim.x + blockIdx.x];
  const long long i0 = (long long)blockIdx.x * RAD_TILE;
  for (int e = threadIdx.x; e < RAD_TILE; e += RAD_THREADS)
    if (i0 + e < a.pool) a.cdf[i0 + e] = o + a.cdf[i0 + e];
}

__global__ void __launch_bounds__(RAD_THREADS) rad_select_kernel(const AdaptiveParams a, int scan_blocks) {
  pdl_wait();
  const SampleParams& s = a.out;
  const long long N = a.pool;
  const double total = a.cdf[N - 1];
  const double u0 = a.part[3 * (long long)scan_blocks + 1];
  unsigned c1 = 0, c2 = 0;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < s.n; j += (long long)gridDim.x * blockDim.x) {
    const double t = ((double)j + u0) / (double)s.n * total;
    long long lo = 0, hi = N;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (a.cdf[mid] > t) hi = mid; else lo = mid + 1;
    }
    const long long i = lo < N ? lo : N - 1;  // t rounded up to the total: the last candidate
    s.x[j] = a.px[i]; s.y[j] = a.py[i]; s.z[j] = a.pz[i]; s.R[j] = a.pR[i];
    const uint8_t m = a.pmask[i];
    s.mask[j] = m;
    if (a.idx) a.idx[j] = i;
    if (a.point_w) {
      const double Q = a.part[3 * (long long)scan_blocks + 2];
      const double Nd = (double)N;
      const double w = (Q > 0.0 && isfinite(Q)) ? rad_q(a.res[i], a.k) * Nd / Q + a.c : 1.0;  // rad_scan_kernel's w_i
      a.point_w[j] = (float)(total / (Nd * w));
    }
    c1 += m & 1u; c2 += (m >> 1) & 1u;
  }
  c1 = __reduce_add_sync(0xffffffffu, c1);
  c2 = __reduce_add_sync(0xffffffffu, c2);
  __shared__ unsigned sh1[RAD_THREADS / 32], sh2[RAD_THREADS / 32];
  __shared__ int last_block;
  if ((threadIdx.x & 31) == 0) { sh1[threadIdx.x >> 5] = c1; sh2[threadIdx.x >> 5] = c2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t1 = 0, t2 = 0;
    for (int w = 0; w < RAD_THREADS / 32; w++) { t1 += sh1[w]; t2 += sh2[w]; }
    atomicAdd(&s.counts[0], (unsigned long long)t1);  // integer atomics: order-independent result
    atomicAdd(&s.counts[1], (unsigned long long)t2);
    __threadfence();
    last_block = atomicAdd(s.ticket, 1ull) == (unsigned long long)gridDim.x - 1;
  }
  __syncthreads();
  if (last_block && threadIdx.x < 32) {
    sample_finish(s);  // the loss weights exactly as the uniform sampler forms them
    if (a.point_w && threadIdx.x == 0) {
      // importance batch: each weighted batch sum estimates the pool's sum times n / N, so the means take the pool's sizes
      const double nd = (double)s.n, Nd = (double)N;
      s.weights[1] = Nd / (nd * (double)a.pool_counts[0]);  // an empty set of the pool: inf, a NaN loss, as uniform
      s.weights[2] = Nd / (nd * (double)a.pool_counts[1]);
      a.pool_counts[0] = 0ull; a.pool_counts[1] = 0ull;
    }
  }
}

cudaError_t launch_adaptive_select(const AdaptiveParams& a, cudaStream_t st) {
  const unsigned nb = (unsigned)((a.pool + RAD_TILE - 1) / RAD_TILE);
  cudaError_t e = launch_pdl(rad_sum_kernel, dim3(nb), dim3(RAD_THREADS), 0, st, a);
  if (e == cudaSuccess) e = launch_pdl(rad_scan_kernel, dim3(nb), dim3(RAD_THREADS), 0, st, a);
  if (e == cudaSuccess) e = launch_pdl(rad_offset_kernel, dim3(nb), dim3(RAD_THREADS), 0, st, a);
  long long sel = (a.out.n + RAD_THREADS - 1) / RAD_THREADS;
  if (sel > 148 * 4) sel = 148 * 4;
  if (e == cudaSuccess) e = launch_pdl(rad_select_kernel, dim3((unsigned)sel), dim3(RAD_THREADS), 0, st, a, (int)nb);
  return e;
}

}  // namespace pinn
