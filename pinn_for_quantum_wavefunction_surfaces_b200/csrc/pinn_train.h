// Launch parameters of the training-loop kernels (pinn_train.cu), shared with pinn_capi.cu.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/pinn_b200.h"
#include "pinn_dp.cuh"
#include "pinn_launch.h"
#include <cmath>

namespace pinn {

struct SampleParams {
  long long n;
  unsigned long long seed;
  unsigned long long* batch_counter;  // device: index of the batch being drawn (advanced by the sampler itself)
  float xL, xR, yL, yR, zL, zR, RL, RR;
  float cutoff, bcutoff;
  float *x, *y, *z, *R;
  uint8_t* mask;
  unsigned long long* counts;  // device, 2: sizes of the two boundary sets
  long long index_offset;      // data-parallel shard: this rank draws points [index_offset, index_offset + n) of the batch
  // the block that finishes last turns the set sizes into the loss weights (and moves the batch counter on):
  double* weights;             // device, 3: {1/n, 1/|set1|, 1/|set2|} (global sizes when dp.world > 1)
  unsigned long long* ticket;  // device, zero between launches: blocks done
  int reset_counts;            // 1: counts are zeroed again after use (the trainer; no memset in front of the next launch)
  DpArgs dp;
};

struct AdamParams {
  double *theta, *m, *v;        // device float64 [1521]
  const double* grad;           // dLtot/dtheta
  const double* sums;           // the 8 loss sums of the step
  float* theta32;               // refreshed float32 copy the next step kernel reads
  unsigned long long* step;     // device: optimizer steps done
  double *best_loss, *best_theta;
  long long* best_step;
  double* hist;                 // [hist_cap][4] {Ltot, Lpde, Lbc, E} or NULL
  long long hist_cap, n;
  double lr, beta1, beta2, eps, best_after;
  uint32_t grad_mask;
  int best_mode, hist_mean_E;
  unsigned long long step_base;  // optimizer steps done when this run (re)started: history rows and train.py's
                                 // "take the first loss" rule count from here (pinn_trainer_load_state)
};

// One kernel.  zero_counts: put a memset of the two counters in front (callers that own `counts`; the trainer keeps them
// zero itself, reset_counts = 1).  dp.world > 1: the set sizes are summed over the ranks (same exchange buffers as the
// gradient sum) and the weights become {1/(world*n), 1/|set1|, 1/|set2|} of the GLOBAL batch.
cudaError_t launch_sample(const SampleParams& s, bool zero_counts, cudaStream_t st);
cudaError_t launch_adam(const AdamParams& a, cudaStream_t st);

// Residual-adaptive selection (pinn_adaptive.cu): n points out of a pool of N drawn by launch_sample, with the pool's
// residuals.  Four launches; out.counts and out.ticket need not be zero.
struct AdaptiveParams {
  long long pool;                                 // N
  double k, c;                                    // w_i = |res_i|^k * N / sum_j |res_j|^k + c
  const float *px, *py, *pz, *pR, *res;           // device [N]: the pool and its residuals
  const uint8_t* pmask;
  double* cdf;                                    // device [N]: inclusive prefix sum of w
  double* part;                                   // device [adaptive_scratch_doubles(N)]
  const unsigned long long* pool_batch;           // device: the batch counter as the pool's draw left it (one past the pool)
  long long* idx;                                 // device [n] pool index of every output point, or NULL
  // importance weights (pinn_sample_adaptive_importance), or NULL: point_w[j] = float(T / (N w_i)) of the candidate i
  // output j takes, and out.weights = {1/n, N/(n |set1 of the pool|), N/(n |set2 of the pool|)} from pool_counts (the
  // pool's set sizes as its draw counted them: its sampler must not reset them; the selection zeroes them after use)
  float* point_w;
  unsigned long long* pool_counts;
  SampleParams out;                               // the batch: n, seed, x..mask, counts, weights, ticket, batch_counter
                                                  // (moved on by sample_finish: point it at a scratch word), reset_counts
};
long long adaptive_scratch_doubles(long long pool);
cudaError_t launch_adaptive_select(const AdaptiveParams& a, cudaStream_t st);

// The update of one parameter (torch.optim.Adam: lerp first moment, bias corrections, eps outside the square root; no
// weight decay, no amsgrad), shared by adam_kernel and by the optimizer step fused into the reduction kernel.
// t = optimizer steps done before this one.
struct AdamCoef {
  double step_size, bc2_sqrt;
};
__host__ __device__ inline AdamCoef adam_coef(const AdamParams& a, unsigned long long t) {
  const double tt = (double)(t + 1ull);
  const double bc1 = 1.0 - pow(a.beta1, tt), bc2 = 1.0 - pow(a.beta2, tt);
  return {a.lr / bc1, sqrt(bc2)};
}
__host__ __device__ inline int tensor_of_entry(int i) {
  const int offs[17] = {O_W1, O_B1, O_W2, O_B2, O_WO, O_BO, O_WE1, O_BE1, O_WE2, O_BE2, O_WE, O_BE,
                        O_WGL, O_BGL, O_WG, O_BG, NTHETA};
  int ti = 0;
  for (int k = 1; k < 16; k++) ti += (i >= offs[k]);
  return ti;
}
// entry i with gradient g; take_best as decided from the loss of this step (see adam_kernel)
__device__ inline void adam_update_entry(const AdamParams& a, const AdamCoef& c, int i, double g, bool take_best) {
  double th = a.theta[i];
  if (take_best && a.best_mode == 0) a.best_theta[i] = th;  // train.py keeps the parameters the loss was evaluated at
  if ((a.grad_mask >> tensor_of_entry(i)) & 1u) {            // frozen tensors have no gradient: the optimizer skips them
    double m = a.m[i], v = a.v[i];
    m = m + (g - m) * (1.0 - a.beta1);
    v = v * a.beta2 + ((1.0 - a.beta2) * g) * g;
    const double denom = sqrt(v) / c.bc2_sqrt + a.eps;
    th = th - c.step_size * (m / denom);
    a.m[i] = m; a.v[i] = v; a.theta[i] = th;
  }
  if (take_best && a.best_mode == 1) a.best_theta[i] = th;  // poc saves the model after optimizer.step()
  a.theta32[i] = (float)th;
}
__device__ inline bool adam_take_best(const AdamParams& a, unsigned long long t, double Ltot) {
  if (a.best_mode == 0) return (t == a.step_base) || (Ltot < *a.best_loss);       // train.py:58
  return ((double)t > a.best_after) && (Ltot < *a.best_loss);                     // poc/main.py:414 (Llim starts at 10)
}
// once per step, after every entry was updated: history row, best-loss record, step counter
__device__ inline void adam_bookkeeping(const AdamParams& a, unsigned long long t, const double* sums, bool take_best) {
  const double Ltot = sums[0];
  if (a.hist && (long long)(t - a.step_base) < a.hist_cap) {
    double* h = a.hist + 4 * (t - a.step_base);
    h[0] = Ltot; h[1] = sums[1]; h[2] = sums[2];
    h[3] = a.hist_mean_E ? sums[3] / (double)a.n : sums[7];  // train.py prints mean(e); poc keeps E[-1]
  }
  if (take_best) { *a.best_loss = Ltot; *a.best_step = (long long)t; }
  *a.step = t + 1ull;
}

// L-BFGS machine (pinn_lbfgs.cu).  slots: evaluations one call may take.  cond: the WHILE node to clear when the call
// ends (trainer graphs), or NULL.
size_t lbfgs_state_bytes(int history_size);
int lbfgs_slots(const pinn_lbfgs_config& c);
cudaError_t launch_lbfgs_begin(unsigned char* state, const pinn_lbfgs_config& c, const double* theta, float* theta32,
                               cudaStream_t st);
cudaError_t launch_lbfgs_advance(unsigned char* state, const double* sums, const double* grad, double* theta, float* theta32,
                                 double* trace, long long trace_rows, const cudaGraphConditionalHandle* cond, cudaStream_t st);
// sets cond to "the call in `state` has not finished" (the node in front of the trainer's WHILE node)
cudaError_t launch_lbfgs_cond(const unsigned char* state, cudaGraphConditionalHandle cond, cudaStream_t st);

cudaError_t measure_fp32_peak(int sm_count, cudaStream_t st, double* fma_per_s, double* ms_best, double* sm_mhz);
cudaError_t launch_enet_curve(const float* theta, const double* R, int n, double* E, double* dE, double* d2E, double* gate,
                              cudaStream_t st);

}  // namespace pinn
