// Small kernels around the fused step kernel (pinn_step_tc.cu): boundary-set counting, and the reduction of the per-CTA
// partial rows - which is also the data-parallel exchange over NVLink peer memory, the optimizer step and the sampler
// of the device-resident trainer (SURVEY.md 8e, 8f-1, 8f-2; poc/main.py:341-355, 403-417; train.py:55-72).
#include "pinn_device.cuh"
#include "pinn_sample.cuh"
#include "pinn_train.h"

namespace pinn {


// counts of the two boundary sets -> weights {1/n, 1/cnt1, 1/cnt2} (only when the caller passes no weights)
__global__ void count_sets_kernel(const StepParams p, unsigned long long* counts) {
  unsigned c1 = 0, c2 = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += (long long)gridDim.x * blockDim.x) {
    if (p.mask) {
      const unsigned mk = p.mask[i];
      c1 += mk & 1u; c2 += (mk >> 1) & 1u;
    } else {
      const Geom g = load_geom(p, i);
      c1 += (g.ir1 * p.bcut <= 1.0f); c2 += (g.ir2 * p.bcut <= 1.0f);
    }
  }
  c1 = __reduce_add_sync(0xffffffffu, c1);
  c2 = __reduce_add_sync(0xffffffffu, c2);
  if ((threadIdx.x & 31) == 0) { atomicAdd(&counts[0], c1); atomicAdd(&counts[1], c2); }
}
__global__ void weights_from_counts_kernel(const unsigned long long* counts, long long n, double* w) {
  w[0] = 1.0 / (double)n;
  w[1] = 1.0 / (double)counts[0];  // empty set -> inf -> NaN loss, like the reference's mean over an empty selection
  w[2] = 1.0 / (double)counts[1];
}

// ---------------------------------------------------------------------------------------------
// add the partial rows (fixed order, double) -> dtheta, sums
// block = 1024 threads = 32 entries x 32 row-slices (every thread has at most 5 independent loads in flight: one
// round trip to L2 instead of a chain of 19); RED_BLOCKS blocks of 32 entries cover a row
//
// With dp.world > 1 the kernel is also the data-parallel all-reduce (pinn_dp.cuh): thread (r, e) of block b sends the
// block's reduced entry e to peer r and receives peer r's; the `world` values are added in rank order.  No NCCL launch,
// no extra kernel.
// ---------------------------------------------------------------------------------------------
constexpr int RED_BLOCKS = NPART / 32;
constexpr int RED_SLICES = 32;
static_assert(RED_SLICES >= DP_MAX_WORLD, "one row-slice of threads per data-parallel peer");
struct RedWeights {  // loss weights by value (the *_host entry) instead of through device memory
  double w[3];
  int use;
};
// Optimizer step fused behind the reduction (the device-resident trainer): every block updates the 32 parameters whose
// gradient it has just completed; the block that finishes last does the once-per-step bookkeeping.
struct AdamFuse {
  int on;
  AdamParams a;
  unsigned long long* ticket;  // device, zero between launches
};
// The batch of the NEXT step drawn by extra blocks of this launch (blocks RED_BLOCKS .. gridDim.x-1), into the trainer's
// other batch buffer: the sampler overlaps the reduction / optimizer step instead of standing between two kernels.
struct SampleFuse {
  int on;
  SampleParams s;
};
constexpr int PRESAMPLE_BLOCKS = 96;
__global__ void __launch_bounds__(RED_SLICES * 32) reduce_partials_kernel(const double* __restrict__ partials, int nrows,
                                                              const double* __restrict__ weights, const RedWeights wi,
                                                              uint32_t grad_mask,
                                                              double* __restrict__ dtheta, double* __restrict__ sums,
                                                              const float* __restrict__ E_out, long long n, const DpArgs dp,
                                                              const AdamFuse ad, const SampleFuse sf, const int E_f64,
                                                              const int dtheta_in_out) {
  if (blockIdx.x >= RED_BLOCKS) {
    // sampler blocks: they touch nothing the step kernel in front reads or writes (other batch buffer), so they do not
    // wait for it; the reduction blocks below do, which also keeps this grid from completing early
    if (sf.on) sample_block(sf.s, blockIdx.x - RED_BLOCKS, gridDim.x - RED_BLOCKS);
    return;
  }
  __shared__ double sh[RED_SLICES][33];
  __shared__ double tot[32];
  __shared__ double l3[3];
  __shared__ int flag_s;
  const int e = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + e;
  // launched as a programmatic dependent of the step kernel (which signals launch_dependents when its tile loop is
  // done): this grid is set up while the step kernel folds its accumulators; the partial rows are complete and
  // visible once the wait returns
  pdl_wait();
  double s = 0.0;
#pragma unroll 5
  for (int r = sl; r < nrows; r += RED_SLICES) s += partials[(size_t)r * NPART + idx];
  sh[sl][e] = s;
  __syncthreads();
  unsigned int step = 0;
  // A peer that never delivers poisons the run (DP_FAILED stays set): this and every later launch then skips the polling
  // (no 30 s stall per step) AND the fused optimizer step, so the parameters stay what they were before the failed
  // exchange; pinn_dp_status / pinn_trainer_read report PINN_ETIMEDOUT.
  __shared__ volatile int dp_failed_s;
  if (threadIdx.x == 0) dp_failed_s = 0;
  if (dp.world > 1) {
    if (threadIdx.x == 0) dp_failed_s = dp_has_failed(dp);
    const unsigned long long step64 = dp_next_step(dp, DP_EXCHANGES);
    step = (unsigned int)step64;
    if (sl == 0) {
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < RED_SLICES; i++) t += sh[i][e];
      tot[e] = t;
    }
    __syncthreads();
    double v = 0.0;
    if (sl < dp.world) {
      const int r = sl;
      if (r == dp.rank) {
        v = tot[e];
      } else {
        dp_send(dp_row(dp.peer[r], step, dp.rank, idx), (unsigned long long)__double_as_longlong(tot[e]), step);
        unsigned long long bits = 0;
        if (dp_recv(dp, dp_row(dp.peer[dp.rank], step, r, idx), step, dp_failed_s, bits))
          v = __longlong_as_double((long long)bits);
      }
    }
    __syncthreads();  // every thread is done with sh / tot of the local pass
    sh[sl][e] = v;    // slices >= world contribute 0; the fixed-order sum below is the sum over ranks
    __syncthreads();
    if (threadIdx.x == 0) dp_block_done(dp, step64, RED_BLOCKS);
  }
  if (sl == 0) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < RED_SLICES; i++) t += sh[i][e];
    tot[e] = t;
    if (idx < NTHETA) {
      // tensor index of this scalar -> honour grad_mask
      int ti, off;
      theta_locate(idx, ti, off);
      // the caller's layout: nn.Linear (out,in) = canonical, or train.py's (in,out) for the 2-D tensors
      const int dst = dtheta_in_out ? off + in_out_index(ti, idx - off) : idx;
      dtheta[dst] = ((grad_mask >> ti) & 1u) ? t : 0.0;
    }
  }
  __syncthreads();
  const double w0 = wi.use ? wi.w[0] : weights[0], w1 = wi.use ? wi.w[1] : weights[1], w2 = wi.use ? wi.w[2] : weights[2];
  constexpr int SB = S_RES2 / 32, b = S_RES2 - SB * 32;   // the block / lane that own the loss sums
  if (blockIdx.x == SB && threadIdx.x == 0) {
    const double r2 = tot[b], p1 = tot[b + 1], p2 = tot[b + 2], sE = tot[b + 3];
    const double Lpde = w0 * r2, Lbc = w1 * p1 + w2 * p2;
    sums[0] = Lpde + Lbc; sums[1] = Lpde; sums[2] = Lbc; sums[3] = sE;
    sums[4] = r2; sums[5] = p1; sums[6] = p2;
    sums[7] = (E_out && n > 0) ? (E_f64 ? reinterpret_cast<const double*>(E_out)[n - 1] : (double)E_out[n - 1]) : 0.0;
  }
  if (!ad.on) return;

  // ---- fused optimizer step.  Every block needs Ltot for the best-model rule: the blocks that do not own the loss
  //      sums add those three entries themselves, in exactly the order used above (row slices, then slices in order,
  //      then ranks in order), so that all blocks - and all ranks - decide on identical bits ----
  if (blockIdx.x == SB) {
    if (threadIdx.x < 3) l3[threadIdx.x] = tot[b + threadIdx.x];
  } else {
    if (threadIdx.x < 96) {
      const int j = threadIdx.x >> 5, sj = threadIdx.x & 31;
      double ps = 0.0;
#pragma unroll 5
      for (int r = sj; r < nrows; r += RED_SLICES) ps += partials[(size_t)r * NPART + S_RES2 + j];
      sh[sj][j] = ps;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
      const int j = threadIdx.x;
      double local = 0.0;
#pragma unroll
      for (int i = 0; i < RED_SLICES; i++) local += sh[i][j];
      double g = local;
      if (dp.world > 1) {
        g = 0.0;
        for (int r = 0; r < dp.world; r++) {
          double v = local;
          if (r != dp.rank) {  // the peer's block SB sent this entry to our buffer; only received here
            unsigned long long bits = 0;
            const bool ok = dp_recv(dp, dp_row(dp.peer[dp.rank], step, r, S_RES2 + j), step, dp_failed_s, bits);
            v = ok ? __longlong_as_double((long long)bits) : 0.0;
          }
          g += v;
        }
      }
      l3[j] = g;
    }
  }
  __syncthreads();
  const AdamParams& a = ad.a;
  const unsigned long long tstep = *a.step;  // read before any block can finish the step (the last block advances it)
  const double Lpde = w0 * l3[0], Lbc = w1 * l3[1] + w2 * l3[2];
  const double Ltot = Lpde + Lbc;
  // (dp_failed_s was last written before the barrier above.)  After a failed exchange the sums are incomplete: no update,
  // no best-model take; the step still counts, its history row holds whatever arrived.
  const bool dp_failed = dp_failed_s != 0;
  const bool take_best = !dp_failed && adam_take_best(a, tstep, Ltot);
  if (sl == 0 && idx < NTHETA && !dp_failed) adam_update_entry(a, adam_coef(a, tstep), idx, tot[e], take_best);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    flag_s = atomicAdd(ad.ticket, 1ull) == (unsigned long long)RED_BLOCKS - 1;
    if (flag_s) {  // every block has updated its parameters and read the step / best loss; the loss sums are visible
      __threadfence();
      const double sv[8] = {ld_acquire_gpu(&sums[0]), ld_acquire_gpu(&sums[1]), ld_acquire_gpu(&sums[2]), ld_acquire_gpu(&sums[3]),
                            0.0, 0.0, 0.0, ld_acquire_gpu(&sums[7])};
      adam_bookkeeping(a, tstep, sv, take_best);
      *ad.ticket = 0ull;
    }
  }
}

}  // namespace pinn

// =================================================================================================
// host-side launchers used by pinn_capi.cu
// =================================================================================================
namespace pinn {

cudaError_t launch_count(const StepParams& p, unsigned long long* counts, double* weights, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(counts, 0, 2 * sizeof(unsigned long long), st);
  if (e != cudaSuccess) return e;
  count_sets_kernel<<<296, 256, 0, st>>>(p, counts);
  weights_from_counts_kernel<<<1, 1, 0, st>>>(counts, p.n, weights);
  return cudaGetLastError();
}

cudaError_t launch_reduce(const double* partials, int nrows, const double* weights, const double* weights_inline,
                          uint32_t grad_mask, double* dtheta, double* sums, const float* E_out, long long n, const DpArgs& dp,
                          cudaStream_t st, const AdamParams* adam, unsigned long long* adam_ticket,
                          const SampleParams* presample, int E_f64, int dtheta_in_out) {
  AdamFuse ad{};
  if (adam) { ad.on = 1; ad.a = *adam; ad.ticket = adam_ticket; }
  SampleFuse sf{};
  if (presample) { sf.on = 1; sf.s = *presample; }
  RedWeights wi{};
  if (weights_inline) { wi.w[0] = weights_inline[0]; wi.w[1] = weights_inline[1]; wi.w[2] = weights_inline[2]; wi.use = 1; }
  return launch_pdl(reduce_partials_kernel, dim3(RED_BLOCKS + (presample ? PRESAMPLE_BLOCKS : 0)), dim3(RED_SLICES * 32), 0, st,
                    partials, nrows, weights, wi, grad_mask, dtheta, sums, E_out, n, dp, ad, sf, E_f64, dtheta_in_out);
}

// Boundary index sets -> mask bytes.  The reference hands LossFunctions the two sets as index tensors
// (torch.where(r >= BCcutoff), poc/main.py:392-393; train.py:38-39); the step kernel wants one byte per point.  One
// launch for both sets: bits are OR-ed into the aligned 32-bit word that holds the byte (a point may be in both sets).
__global__ void __launch_bounds__(256) mask_from_index_sets_kernel(const long long* __restrict__ idx1, long long n1,
                                                                 const long long* __restrict__ idx2, long long n2,
                                                                 unsigned int* __restrict__ mask_words, long long n) {
  const long long tot = n1 + n2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    const bool second = i >= n1;
    const long long row = second ? idx2[i - n1] : idx1[i];
    if (row < 0 || row >= n) continue;  // (the reference would raise an IndexError; out-of-range rows are ignored here)
    atomicOr(&mask_words[row >> 2], (second ? 2u : 1u) << (8u * (unsigned)(row & 3)));
  }
}
cudaError_t launch_mask_from_index_sets(const long long* idx1, long long n1, const long long* idx2, long long n2, uint8_t* mask,
                                        long long n, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(mask, 0, (size_t)((n + 3) / 4) * 4, st);
  if (e != cudaSuccess) return e;
  const long long tot = n1 + n2;
  if (tot <= 0) return cudaSuccess;
  long long blocks = (tot + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  mask_from_index_sets_kernel<<<(unsigned)blocks, 256, 0, st>>>(idx1, n1, idx2, n2, reinterpret_cast<unsigned int*>(mask), n);
  return cudaGetLastError();
}

}  // namespace pinn
