// Launch parameters and host-side launchers shared by the kernel files (pinn_step_tc.cu, pinn_reduce.cu, pinn_train.cu) and pinn_capi.cu.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "pinn_common.cuh"

namespace pinn {

// Dense-grid mode of the inference kernel (SURVEY.md 8f-3; poc/main.py:438-517, 639-676): point p of the n = nx*ny*nz
// grid is (i,j,k) = meshgrid 'ij' order of three linspaces, R is one value, and instead of per-point stores the kernel
// accumulates the quadrature sums  S = sum_p w_p * {psi H psi, psi^2, lcao H lcao, lcao^2, (dV/dR) psi^2}.
// Second generator, sph = 1 (pinn_spheroidal_reduce): a sweep over nR values of R with the prolate-spheroidal node set
// (s_i, nu_j) at every R.  Each R owns tiles_per_R super-tiles of 128 slots (slot l = i * nnu + j; the slots behind
// ns * nnu repeat the last node with weight 0), so every super-tile has ONE R, and every warp of role 0 writes one row
// {4 sums, -, E(R)} of its 32 points: [tiles][4 groups][8] in partials.  No tile's row depends on the other R of the sweep.
struct GridDesc {
  int on;
  int sph;
  int nx, ny, nz;
  double x0, dx, y0, dy, z0, dz;  // linspace start / step
  double R;
  const double *wx, *wy, *wz;     // 1-D quadrature weights (Simpson), device
  double* partials;               // [gridDim.x][8] (sph: [nR * tiles_per_R * 4][8])
  int ns, nnu, tiles_per_R;       // sph: node counts, super-tiles per R
  const double *Rs, *s, *ws, *nu, *wnu;  // sph: device, [nR], [ns], [ns], [nnu], [nnu]
};

struct StepParams {
  const void *x, *y, *z, *R;
  const uint8_t* mask;
  // Per-point loss weights (device float32 [n], pinn_loss_fwd_bwd_weighted), read only by the WEIGHTED training instances.
  // The member sits in what were 8 unused bytes: without them every member behind moves up by 8 bytes, and ptxas
  // schedules the training kernel <2,true,false> differently (5866 instead of 5874 SASS instructions): measured 0.2 %
  // slower, 0.11085 vs 0.11062 ms per 2^18-point step (tools/ab_time.py, 5 interleaved rounds, B200 at 1000 W).
  const float* point_w;
  const float* theta;     // the raw parameter vector; every CTA builds its own operand images in shared memory
  const double* weights;  // {w_pde, w_bc1, w_bc2}
  double* partials;       // [gridDim.x][NPART]
  float* E_out;
  float *psi, *lap, *hpsi, *res;  // fields mode outputs (nullable)
  long long n;
  int in_f64;
  float bcut;
  VariantCoef vc;
  int base_grads, gate_grads;  // reverse sweeps wanted (fine-tune mode clears both)
  GridDesc grid;
  // HOST pointers, read by the launchers only: when set, theta (1521 float; the *_host entry) and / or the three loss
  // weights travel inside the kernel parameters instead of through a preceding host-to-device copy
  const float* theta_inline;
  const double* weights_inline;
  int w_by_value;         // set by the launcher: the loss weights are in the parameter block behind this struct
  // the caller's 16 parameter tensors instead of a packed vector (pinn_loss_fwd_bwd_tensors): device pointers in
  // canonical (state_dict) order, float32 or float64, nn.Linear (out,in) or train.py (in,out) layout; every CTA gathers
  // them while it builds its operand images - no packing kernel, no packed copy in front of the launch
  const void* theta_tensors[16];
  int theta_from_tensors, tensors_f64, tensors_in_out;
  int E_f64;              // E_out points at float64 (the reference's dtype) instead of float32
};

// Launch as a programmatic dependent of the kernel in front of it in the stream: the grid may be set up (and, where
// resources allow, its CTAs made resident) while that kernel drains.  Every kernel launched this way executes
// griddepcontrol.wait (pdl_wait) before its first global-memory access, which returns once the kernel in front has
// completed and its writes are visible - stream semantics are unchanged, only launch latency is hidden.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// the fused step kernel (pinn_step_tc.cu): super-tiles of 128 points, one persistent CTA per SM.  A training launch with
// p.point_w set runs the WEIGHTED instance (device-resident batches only: no theta_inline, no grid)
cudaError_t launch_step_tc(int nev, bool train, const StepParams& p, int grid, cudaStream_t st);
cudaError_t launch_grid_finish(const double* partials, int nrows, double* out, cudaStream_t st);
// The forward-only loss reduction (pinn_loss_eval): the LOSS instance of the step kernel over n points, one row of 8
// doubles per CTA into p.grid.partials (p.grid.on = 0), then one finishing block -> the 8 sums of pinn_loss_fwd_bwd.
// weights: device {w_pde, w_bc1, w_bc2} or NULL (the counted sets).  val: NULL, or the trainer's validation record.
struct LossValidation {
  int on;
  const unsigned long long* step;  // device: optimizer steps done (column 0 of the row)
  unsigned long long* count;       // device: evaluations recorded; row `count` is written when count < cap
  double* rows;                    // [cap][4] {steps done, Ltot, Lpde, Lbc}
  long long cap;
  double* best_loss;               // +inf when the record starts
  long long* best_step;
  double* best_theta;              // float64 [NTHETA] <- theta of the evaluation taken
  const double* theta;
};
cudaError_t launch_loss_tc(int nev, const StepParams& p, int grid, cudaStream_t st);
cudaError_t launch_loss_finish(const double* partials, int nrows, long long n, const double* weights, double* sums,
                               const LossValidation* val, cudaStream_t st);
// sums the rows_per_R rows of every R in a fixed order -> out [nR][8]; a row with R <= 0 (or NaN) is all NaN
cudaError_t launch_sph_finish(const double* partials, int nR, int rows_per_R, const double* Rs, double* out, cudaStream_t st);
cudaError_t launch_count(const StepParams& p, unsigned long long* counts, double* weights, cudaStream_t st);
// weights: device pointer, or NULL with weights_inline (host, 3 double) carried in the kernel parameters
// dp: the data-parallel exchange fused into the reduction (pinn_dp.cuh)
// adam (optional): the optimizer step of the device-resident trainer fused behind the reduction (pinn_train.h)
// presample (optional): extra blocks of the same launch draw the trainer's next batch (pinn_sample.cuh)
struct DpArgs;
struct AdamParams;
struct SampleParams;
// E_f64: E_out holds float64; dtheta_in_out: the 2-D tensors of dtheta are written in train.py's (in,out) layout
cudaError_t launch_reduce(const double* partials, int nrows, const double* weights, const double* weights_inline,
                          uint32_t grad_mask, double* dtheta, double* sums, const float* E_out, long long n, const DpArgs& dp,
                          cudaStream_t st, const AdamParams* adam = nullptr, unsigned long long* adam_ticket = nullptr,
                          const SampleParams* presample = nullptr, int E_f64 = 0, int dtheta_in_out = 0);
// boundary index sets (int64 row indices, device) -> per-point mask bytes (bit 0: set 1, bit 1: set 2); mask 4-byte aligned
cudaError_t launch_mask_from_index_sets(const long long* idx1, long long n1, const long long* idx2, long long n2, uint8_t* mask,
                                        long long n, cudaStream_t st);

}  // namespace pinn
