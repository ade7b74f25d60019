/*
 * pinn_b200.h - C ABI of the B200-native PINN residual-and-gradient hot path.
 *
 * The reference (slitvinov/PINN_for_quantum_wavefunction_surfaces) has no FFI: its
 * hot path is Python (poc/main.py:341-355 NN_ion.LossFunctions, poc/main.py:321 +
 * 118 parametricPsi + hamiltonian, and the inline block train.py:41-57).  This
 * header is the boundary a binding would use instead (ctypes stub: INTEGRATION.md).
 * Plain pointers and sizes only; no torch types.
 *
 * Conventions
 *  - every entry returns 0 on success, a positive cudaError_t value for CUDA
 *    failures and a negative PINN_E* code for argument errors; the message is
 *    available from pinn_last_error().  Nothing throws across this boundary.
 *  - all device buffers are owned by the caller; the library only owns small
 *    workspaces (per-CTA partial sums, set counters): ONE PER STREAM that calls in,
 *    allocated on the first call on that stream.  No allocation happens on later
 *    calls, so every *device* entry point is CUDA-graph capturable once one plain
 *    call has been made on the capturing stream.  pinn_spheroidal_reduce also keeps
 *    room for the largest sweep it has run on the stream: a capture of it needs one
 *    plain call at least as large (nR * ceil(ns*nnu/128)) first.  Likewise a training
 *    call with more points than any earlier call on its stream grows the row workspace
 *    (past 148 x 256 x 128 = 4.8e6 points a training launch gets one row per 256
 *    super-tiles per SM): capture only after a plain call at least as large.
 *  - every call takes the stream explicitly (as a void* holding a cudaStream_t) and
 *    selects the handle's device itself, so it may be called from any host thread
 *    (torch runs autograd.Function.backward on its own thread).  Calls on ONE stream
 *    are ordered by the stream; calls on DIFFERENT streams of one handle (torch's
 *    current stream, a pinn_trainer's own stream, the *_host entry's private stream)
 *    may overlap on the device - they share no scratch memory.  Exception: with the
 *    data-parallel exchange enabled (pinn_dp_*) the handle carries one sequence of
 *    exchange steps; a call on another stream than the previous exchanging call
 *    first waits on the host for that stream to drain.
 *  - theta is the packed parameter vector, 1521 scalars in NN_ion.state_dict() order
 *    with nn.Linear (out,in) layout (poc/main.py:233-245; SURVEY.md Appendix B):
 *      W1(16,2) b1(16) W2(16,16) b2(16) wo(16) bo | WE1(32) bE1(32) WE2(32,32) bE2(32)
 *      wE(32) bE | WgL(10) bgL(10) wg(10) bg
 *    train.py's tuple (train.py:108-109) is the same set in (in,out) layout with the
 *    gate before the E-net; the host wrapper permutes/transposes.
 */
#ifndef PINN_B200_H
#define PINN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PINN_THETA_SIZE 1521
#define PINN_NUM_TENSORS 16
#define PINN_SUMS_SIZE 8

/* variant: which formulation of the model/residual (SURVEY.md Appendix A/D) */
#define PINN_VARIANT_POC 0     /* poc/main.py: two MLP evaluations summed; res = -1/2 lap psi + V psi - E psi */
#define PINN_VARIANT_TRAINPY 1 /* train.py: one evaluation doubled; res = lap psi + (e + 1/r1 + 1/r2) psi */

/* dtype of the coordinate arrays x,y,z,R */
#define PINN_F32 0
#define PINN_F64 1

#define PINN_EINVAL (-1)  /* bad argument */
#define PINN_ENOTSUP (-2) /* device is not sm_100 or kernel image missing */
#define PINN_ETIMEDOUT (-3) /* data-parallel exchange: a peer never delivered */

typedef struct pinn_handle pinn_handle;

/* Library / layout introspection. */
int pinn_version(void);
int pinn_theta_size(void);
/* Offsets (in scalars) of the 16 tensors inside theta; out must hold 17 ints (last = 1521). */
void pinn_theta_offsets(int* out);

/* Create a handle bound to CUDA device `device`; allocates the *_host entry's stream, its workspace and its
 * page-locked result buffer.  Fails with PINN_ENOTSUP on anything but an sm_100 device (there is no fallback). */
int pinn_create(int device, pinn_handle** out);
int pinn_destroy(pinn_handle* h);
/* Message of the last failure on this handle (or of the last pinn_create failure when h==NULL). */
const char* pinn_last_error(pinn_handle* h);
/* Number of kernels this handle has launched so far (bench.py reports it as gpu_launches). */
int64_t pinn_launch_count(pinn_handle* h);

/* The library carries ONE implementation of the fused step kernel, PINN_ENGINE_TCGEN05 (skinny mat-vecs as M=128 TF32
 * tcgen05.mma with activations in tensor memory, 3xTF32).  pinn_set_engine returns 0 for PINN_ENGINE_TCGEN05,
 * PINN_ENOTSUP for PINN_ENGINE_FFMA (the round-1 engine of DESIGN.md section 3, no longer part of the library) and
 * PINN_EINVAL for any other value; pinn_get_engine returns PINN_ENGINE_TCGEN05. */
#define PINN_ENGINE_FFMA 0
#define PINN_ENGINE_TCGEN05 1
int pinn_set_engine(pinn_handle* h, int engine);
int pinn_get_engine(pinn_handle* h);

/* Measurement helper (bench.py's roofline denominator): the FP32 FFMA rate of this device right now, from a
 * register-resident loop of independent FFMA chains (best of 8 timings of 10 x ~0.55 ms each, CUDA events).
 * fma_per_s: fused multiply-adds per second (x2 = FLOP/s); ms: duration of one timed kernel; sm_mhz: the SM clock the
 * loop ran at (block 0 times itself with clock64 and %globaltimer).  Synchronous. */
int pinn_measure_fp32_peak(pinn_handle* h, double* fma_per_s, double* ms, double* sm_mhz);
/* Effective SM clock of the last training evaluation enqueued on `stream`: CTA 0 of the step kernel times itself (SM
 * cycles and nanoseconds from its entry to the end of its tile loop).  sm_mhz above is the same measurement for the FFMA
 * loop.  Synchronises the stream. */
int pinn_step_kernel_clock(pinn_handle* h, void* stream, double* cycles, double* ns);

/* Host-side wall-clock split of the last pinn_loss_fwd_bwd_host call on this handle, microseconds:
 * {enqueue (argument checks, parameter conversion, launches), wait for the device, copy-out, total}. */
int pinn_host_timing(pinn_handle* h, double* out4);

/* Optional timing of the fused step kernel alone (bench.py's roofline figure): between begin and collect
 * every pinn_loss_fwd_bwd brackets its step-kernel launch with CUDA events on the caller's stream;
 * collect synchronises them and returns the summed duration and the number of launches. */
int pinn_profile_begin(pinn_handle* h);
int pinn_profile_collect(pinn_handle* h, double* total_ms, int* launches);

/*
 * Training evaluation: replaces NN_ion.LossFunctions + Ltot.backward()
 * (poc/main.py:341-355, 403) and train.py:41-57 + 71.
 *
 *   Ltot = w[0] * sum_p res_p^2 + w[1] * sum_{p in set1} psi_p^2 + w[2] * sum_{p in set2} psi_p^2
 *
 * with the reference's means obtained for w = {1/n, 1/|set1|, 1/|set2|}; under
 * data-parallel sharding the caller passes the GLOBAL n and counts so that shard
 * results simply add.
 *
 *  x,y,z,R   device, n scalars each, dtype in_dtype (coordinates of the collocation points)
 *  mask      device, n bytes, bit0 = point in boundary set 1 (r1 >= BCcutoff), bit1 = set 2;
 *            NULL: the kernel derives the sets from r1,r2 >= bcutoff (fp32 compare)
 *  theta     device, 1521 float
 *  weights   device, 3 double {w_pde, w_bc1, w_bc2}; NULL: 1/n and 1/count are used
 *            (a small extra kernel counts the sets first)
 *  grad_mask bit i set = gradient of tensor i (state_dict order) is wanted; tensors
 *            whose bit is clear get zeros.  0x0FC0 is the reference's fine-tune mode
 *            (freezeBase + freezeDecayUnit, poc/main.py:305-319): base-MLP and gate
 *            reverse sweeps are skipped.
 *  sums      device out, 8 double: {Ltot, Lpde, Lbc, sum E, sum res^2, sum psi^2 set1,
 *            sum psi^2 set2, E of the last point}
 *  dtheta    device out, 1521 double: dLtot/dtheta
 *  E_out     device out or NULL, n float: E(R_p) (poc returns it, main.py:355; train.py prints its mean)
 */
int pinn_loss_fwd_bwd(pinn_handle* h, int variant, int64_t n,
                      const void* x, const void* y, const void* z, const void* R, int in_dtype,
                      const uint8_t* mask, const float* theta, const double* weights,
                      uint32_t grad_mask, float bcutoff,
                      double* sums, double* dtheta, float* E_out, void* stream);

/*
 * pinn_loss_fwd_bwd with a per-point loss weight: point_w (device, n float32, finite and >= 0) multiplies every per-point
 * term of the sums and of their gradient,
 *   Lpde = w_pde sum_p om_p res_p^2,   Lbc = w_bc1 sum_p om_p m1_p psi_p^2 + w_bc2 sum_p om_p m2_p psi_p^2,
 *   sums[3] = sum_p om_p E_p,
 * while the set sizes counted for weights = NULL stay counts of points.  om = 1 gives pinn_loss_fwd_bwd's bits.  Its use:
 * an importance-weighted adaptive batch (pinn_sample_adaptive_importance), whose weighted sums estimate the pool's
 * unweighted ones without bias.  Device-resident inputs only (the *_host entry has no weighted form).  PINN_EINVAL, with
 * nothing launched, for a NULL point_w and everything pinn_loss_fwd_bwd refuses.
 */
int pinn_loss_fwd_bwd_weighted(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z,
                               const void* R, int in_dtype, const uint8_t* mask, const float* theta, const double* weights,
                               const float* point_w, uint32_t grad_mask, float bcutoff, double* sums, double* dtheta,
                               float* E_out, void* stream);

/*
 * Inference: replaces the pair parametricPsi + hamiltonian (poc/main.py:321, 118;
 * call sites 451-454) and the residual of train.py:54.  Any output may be NULL.
 *  psi, lap (laplacian of psi), hpsi (-1/2 lap psi + V psi, Hartree form), res
 *  (the variant's PDE residual), E: device, n float each.
 */
int pinn_fields(pinn_handle* h, int variant, int64_t n,
                const void* x, const void* y, const void* z, const void* R, int in_dtype,
                const float* theta,
                float* psi, float* lap, float* hpsi, float* res, float* E, void* stream);

/*
 * The loss without its gradient: the 8 sums of pinn_loss_fwd_bwd at theta over n points, from a forward-only instance of
 * the step kernel that stores nothing per point.
 *  - res, psi and E of every point are the float32 bits pinn_fields writes for it; the set bits come from the mask byte
 *    (bit 0: set 1, bit 1: set 2) or, with mask NULL, from the training rule r >= bcutoff (ir * bcutoff <= 1).
 *  - Every sum is accumulated in DOUBLE: per lane over the CTA's super-tiles, then a fixed shuffle tree, a fixed group
 *    order and the CTA rows in index order.  Repeat calls give the same bits, and the sums do not drift with n the way
 *    the float32 accumulators of the training kernel do.
 *  - weights: device, 3 double {w_pde, w_bc1, w_bc2}, or NULL for {1/n, 1/|set1|, 1/|set2|} of the counted sets (no
 *    separate counting launch).  An empty set gives a NaN Lbc, as in the training path.
 *  - sums (device, 8 double) = {Ltot, Lpde, Lbc, sum E, sum res^2, sum psi^2 over set 1, sum psi^2 over set 2, E of the
 *    last point}; sums[3] is the float64 sum of the float32 E.
 * Two launches (the step kernel, one finishing block); the per-CTA rows live in the stream's workspace, so the call can
 * be captured in a CUDA graph once it has run on the stream outside a capture.  PINN_EINVAL, with nothing launched, for
 * n <= 0, a NULL pointer other than mask and weights, a bad in_dtype or an unknown variant.
 */
int pinn_loss_eval(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z, const void* R,
                   int in_dtype, const uint8_t* mask, const float* theta, const double* weights, float bcutoff,
                   double* sums, void* stream);

/*
 * pinn_loss_fwd_bwd for a caller that holds the model as its 16 PARAMETER TENSORS (an nn.Module / train.py's tuple) -
 * the call behind the torch.autograd.Function that replaces NN_ion.LossFunctions (poc/main.py:341-355) and the inline
 * block train.py:41-57.  Nothing is packed or converted in front of the launch:
 *  params        16 device pointers, one per tensor, in the order and layout named by param_layout:
 *                PINN_VARIANT_POC     = NN_ion.state_dict() order, nn.Linear (out,in) weights (poc/main.py:233-245)
 *                PINN_VARIANT_TRAINPY = train.py's tuple order (gate before E-net), (in,out) weights (train.py:88-109)
 *                every CTA of the step kernel gathers them (and converts float64 -> float32) while it builds its
 *                operand images
 *  param_dtype   PINN_F32 / PINN_F64 (all 16 alike)
 *  weights_host  HOST, 3 double {w_pde, w_bc1, w_bc2}: carried inside the kernel parameters; NULL = counted on the device
 *  dtheta        device, 1521 double, the tensors in canonical ORDER (pinn_theta_offsets) but each in the caller's
 *                LAYOUT ((in,out) for PINN_VARIANT_TRAINPY), so that per-tensor views need no transpose
 *  E_out         device, n values of E_dtype (PINN_F32 / PINN_F64) or NULL
 * Everything else as in pinn_loss_fwd_bwd.
 */
int pinn_loss_fwd_bwd_tensors(pinn_handle* h, int variant, int64_t n,
                              const void* x, const void* y, const void* z, const void* R, int in_dtype,
                              const uint8_t* mask, const void* const* params, int param_dtype, int param_layout,
                              const double* weights_host, uint32_t grad_mask, float bcutoff,
                              double* sums, double* dtheta, void* E_out, int E_dtype, void* stream);

/*
 * The reference passes the two boundary sets as index tensors (torch.where(r >= BCcutoff), poc/main.py:392-393;
 * train.py:38-39); the kernels want one byte per point.  idx1 / idx2: device int64 row indices (n1 / n2 of them);
 * mask: device, 4-byte aligned, room for n rounded up to a multiple of 4 bytes; bit 0 = set 1, bit 1 = set 2.
 * One memset + one kernel on `stream`.
 */
int pinn_mask_from_index_sets(pinn_handle* h, int64_t n, const int64_t* idx1, int64_t n1, const int64_t* idx2, int64_t n2,
                              uint8_t* mask, void* stream);

/*
 * Same as pinn_loss_fwd_bwd but with HOST buffers (the call a CPU-resident caller such
 * as the unmodified reference training loop makes), synchronous.  Page-locked inputs
 * (cudaHostAlloc / cudaHostRegister / torch pin_memory) are read by the step kernel IN PLACE
 * over PCIe, one super-tile ahead of the computation - nothing is copied first; theta and
 * the loss weights travel inside the kernel parameters; the 8 sums and 1521 gradients are
 * written by the reduction kernel into mapped page-locked memory and handed back after one
 * stream synchronisation.  Pageable inputs are staged instead: host->device copies in up
 * to 4 chunks on a copy stream that overlap the kernels (when weights_host is given).
 * theta_host is 1521 double (the reference keeps parameters in float64); weights_host is
 * 3 double or NULL (NULL: the boundary sets are counted on the device first).
 */
int pinn_loss_fwd_bwd_host(pinn_handle* h, int variant, int64_t n,
                           const void* x, const void* y, const void* z, const void* R, int in_dtype,
                           const uint8_t* mask, const double* theta_host, const double* weights_host,
                           uint32_t grad_mask, float bcutoff,
                           double* sums_host, double* dtheta_host, float* E_out_host);

/*
 * Data-parallel exchange (SURVEY.md 8e: collocation points shard across the GPUs of one box, the 8 sums + 1521
 * gradients are summed across ranks once per step; the reference has no multi-GPU code, this replaces the
 * ncclAllReduce a port would add).  The sum is FUSED into the reduction kernel of pinn_loss_fwd_bwd[_host]: each rank
 * stores its reduced row into every peer's exchange buffer through NVLink peer memory as 8-byte {data, step number}
 * words (no fence, no separate flag), polls its own buffer for the peers' rows and adds them in rank order
 * (bit-identical on all ranks).
 * No extra launch, no host synchronisation, CUDA-graph capturable (the step number lives on the device).
 * With the exchange enabled the caller passes the GLOBAL loss weights {1/n, 1/|set1|, 1/|set2|} and every rank must
 * make the same sequence of training-evaluation calls.
 *
 *   one process per GPU:  pinn_dp_init(h, rank, world, my_handle)  ->  all-gather the 64-byte handles (any host
 *                         transport, e.g. torch.distributed)       ->  pinn_dp_connect(h, all_handles)
 *   one process, several handles/devices:  pinn_dp_init(h_r, r, world, NULL) for all r, then
 *                         pinn_dp_connect_local(h_r, handles) for all r
 * The device-resident trainer (pinn_trainer_*) created on a handle with the exchange enabled runs data-parallel without
 * any host involvement: rank r draws points [r n, (r+1) n) of the global batch (Philox counter = global point index, so
 * the union over the ranks is the batch one GPU would draw for world*n points), the sampler's set sizes are summed
 * over the ranks with the same protocol, and every rank's Adam sees the same global gradient (identical replicas).
 * Connect the exchange BEFORE creating the trainer (the peers' addresses are captured in its CUDA graphs).
 * pinn_dp_connect* enable the exchange; pinn_dp_enable switches it off/on; pinn_dp_status returns PINN_ETIMEDOUT if a
 * peer failed to deliver within ~30 s (the kernel then gives up instead of hanging; every rank stops updating its replica) and the number of completed
 * exchanges; pinn_dp_shutdown (collective by convention: call it on every rank after a barrier) frees the buffer.
 */
#define PINN_DP_HANDLE_BYTES 64
#define PINN_DP_MAX_WORLD 8
int pinn_dp_init(pinn_handle* h, int rank, int world, void* ipc_handle_out);
int pinn_dp_connect(pinn_handle* h, const void* all_handles);
int pinn_dp_connect_local(pinn_handle* h, pinn_handle* const* peers);
int pinn_dp_enable(pinn_handle* h, int on);
int pinn_dp_status(pinn_handle* h, int64_t* exchanges);
/* How long a rank polls for its peers before it declares the exchange failed (default ~30 s; call after pinn_dp_init and
 * before creating trainers / capturing graphs on the handle, which copy the value). */
int pinn_dp_set_timeout(pinn_handle* h, double seconds);
int pinn_dp_shutdown(pinn_handle* h);

/* =====================================================================================================
 * Rows next to the hot path (SURVEY.md 8f): device-side sampler, fused Adam, a device-resident trainer,
 * the E(R)/gate curve and dense-grid quadrature.  Same conventions as above.
 * ===================================================================================================== */

/*
 * Collocation sampler + clamp + boundary sets: replaces train.py:26-39 and sampling()/radial()/torch.where of
 * poc/main.py:124-156, 390-393 for runs that do not need the host's torch RNG stream.
 * Point i of batch `batch` is Philox4x32-10(counter = {i_lo, i_hi, batch_lo, batch_hi}, key = seed); word k of the
 * output, u = (word >> 8) * 2^-24 in [0,1), gives x, y, z, R = lo + (hi - lo) * u with box = {xL,xR,yL,yR,zL,zR,RL,RR}.
 * Then, literally as the reference: x = cutoff where r1 < cutoff or r2 < cutoff (radii of the unclamped point), sets
 * r1 >= bcutoff / r2 >= bcutoff after the clamp (bit0 / bit1 of mask).  counts: device, 2 x uint64 set sizes;
 * weights: device, 3 double {1/n, 1/count1, 1/count2}.  All outputs float32 / device.
 */
int pinn_sample(pinn_handle* h, int64_t n, uint64_t seed, uint64_t batch, const float box[8], float cutoff, float bcutoff,
                float* x, float* y, float* z, float* R, uint8_t* mask, uint64_t* counts, double* weights, void* stream);

/*
 * Residual-adaptive collocation (RAD, Wu et al., CMAME 403, 2023): the n points of a batch drawn from `pool` uniform
 * candidates with probability proportional to the PDE residual.
 *  1. The pool is pinn_sample(pool, seed, batch, box, cutoff, bcutoff) bit for bit (pool_x .. pool_mask); pool_res is
 *     its residual at theta (device float32 [1521]), the bits pinn_fields writes to `res`.
 *  2. Weights, in float64: q_i = |res_i|^k (0 where res_i is not finite), Q = sum q_i; w_i = q_i * pool / Q + c when
 *     Q > 0 and finite, else w_i = 1 (uniform).  pool_cdf (device float64 [pool]) = inclusive prefix sum of w, with a
 *     fixed association order (block sums, then a sequential fold of the block totals): the same bits on every call, and
 *     never decreasing.
 *  3. Systematic resampling: u0 = word 0 of Philox4x32-10(counter = {pool_lo, pool_hi, batch_lo, batch_hi}, key = seed)
 *     * 2^-32, the point just past the pool in its own stream.  Output j takes the first i with
 *     pool_cdf[i] > ((double)j + u0) / (double)n * pool_cdf[pool-1] (evaluated exactly as written; no such i: pool-1).
 *     Candidate i is therefore taken floor(n P_i) or ceil(n P_i) times, P_i = w_i / sum w.
 *  4. x, y, z, R, mask = the pool's at the selected indices; idx (device int64 [n], may be NULL) = those indices;
 *     counts (device 2 x uint64) = set sizes of the batch; weights (device 3 double) = {1/n, 1/count1, 1/count2} as
 *     pinn_sample forms them.
 * Eight launches: the batch index, the pool's set-size reset, the pool's sampler, the pool's residual (inference
 * instance of the step kernel), four selection kernels.  All buffers are the caller's, so the call can be captured in a
 * CUDA graph once it has run on the stream outside a capture.  PINN_EINVAL, with nothing launched, for n <= 0,
 * pool < n, k or c negative or not finite, a NULL pointer other than idx, or an unknown variant.
 */
int pinn_sample_adaptive(pinn_handle* h, int variant, const float* theta, int64_t n, int64_t pool, uint64_t seed, uint64_t batch,
                         const float box[8], float cutoff, float bcutoff, float k, float c, float* pool_x, float* pool_y,
                         float* pool_z, float* pool_R, uint8_t* pool_mask, float* pool_res, double* pool_cdf, float* x,
                         float* y, float* z, float* R, uint8_t* mask, int64_t* idx, uint64_t* counts, double* weights,
                         void* stream);

/*
 * pinn_sample_adaptive with importance weights.  The batch (x, y, z, R, mask, idx, counts) is the same bits; in addition
 *  - point_w (device, n float32): om_j = float32(T / (N w_i)) = 1 / (N P_i) of the candidate i that output j took, with
 *    w_i formed again in float64 exactly as step 2 formed it (the same Q) and T = pool_cdf[N-1].  om <= (1 + c) / c; in
 *    the uniform fallback om = 1.
 *  - weights = {1/n, N / (n |set1 of the pool|), N / (n |set2 of the pool|)} (an empty set of the pool: inf, a NaN Lbc).
 * Candidate i is taken c_i times with E_u0[c_i] = n P_i, so the expectation over u0 of pinn_loss_fwd_bwd_weighted on this
 * batch with these weights - its loss and its gradient - is the pool's uniform loss {1/N, 1/|set1|, 1/|set2|}.
 * Importance mode needs c > 0 (Lbc weights psi^2, not res^2, so a candidate of zero residual must keep a positive
 * probability): PINN_EINVAL for c <= 0 or a NULL point_w, and everything pinn_sample_adaptive refuses; nothing launched.
 */
int pinn_sample_adaptive_importance(pinn_handle* h, int variant, const float* theta, int64_t n, int64_t pool, uint64_t seed,
                                    uint64_t batch, const float box[8], float cutoff, float bcutoff, float k, float c,
                                    float* pool_x, float* pool_y, float* pool_z, float* pool_R, uint8_t* pool_mask,
                                    float* pool_res, double* pool_cdf, float* x, float* y, float* z, float* R, uint8_t* mask,
                                    int64_t* idx, uint64_t* counts, double* weights, float* point_w, void* stream);

/*
 * One optimizer step of torch.optim.Adam (no weight decay, no amsgrad) over the 1521 float64 parameters, fused with
 * the reference loops' bookkeeping (train.py:58-72; poc/main.py:403-417).  All pointers are device memory.
 *  theta, m, v   in/out float64 [1521];  grad: dLtot/dtheta;  sums: the 8 sums of pinn_loss_fwd_bwd
 *  theta32       out float32 [1521]: the copy the next pinn_loss_fwd_bwd reads
 *  step          in/out uint64: optimizer steps done (= tt of this step); incremented
 *  best_mode 0   train.py: if tt == 0 or Ltot < best_loss, keep Ltot and the PRE-step parameters
 *  best_mode 1   poc: if tt > best_after and Ltot < best_loss (initialise to 10), keep Ltot and the POST-step parameters
 *  hist          NULL or [hist_cap][4] doubles: row tt = {Ltot, Lpde, Lbc, E}, E = mean over the batch
 *                (history_mean_E, train.py:64) or E of the last point (poc/main.py:411)
 *  grad_mask     tensors whose bit is clear are frozen: no update, state untouched
 */
int pinn_adam_step(pinn_handle* h, double* theta, double* m, double* v, const double* grad, const double* sums, float* theta32,
                   uint64_t* step, double* best_loss, double* best_theta, int64_t* best_step, double* hist, int64_t hist_cap,
                   int64_t n, double lr, double beta1, double beta2, double eps, uint32_t grad_mask, int best_mode,
                   int64_t best_after, int history_mean_E, void* stream);

/* Device-resident training loop, no host synchronisation until pinn_trainer_read.  Mirrors train() of train.py:21-72 and
 * poc/main.py:359-430.  A step is two launches chained as programmatic dependents: the fused loss/gradient kernel, and
 * one kernel that reduces the per-CTA rows (and exchanges them with the data-parallel peers), applies the float64 Adam
 * step with the reference loops' bookkeeping, and - in extra blocks - draws the batch of the next step into the
 * trainer's second batch buffer.  pinn_trainer_run(use_graph = 1) replays captured CUDA graphs of the same launches. */
typedef struct pinn_train_config {
  int variant;               /* PINN_VARIANT_* */
  int best_mode;             /* 0 train.py, 1 poc (see pinn_adam_step) */
  int history_mean_E;        /* history column 3: 1 mean E (train.py), 0 E of the last point (poc) */
  int sc_sampling;           /* resample every sc_sampling steps (train.py:79; params['sc_sampling']) */
  int64_t n;                 /* points per step */
  int64_t freeze_after;      /* no resampling for tt >= freeze_after (poc: 0.9*epochs; train.py: never -> INT64_MAX) */
  int64_t best_after;        /* poc: 0.5*epochs */
  int64_t history_capacity;  /* rows of the device history */
  uint64_t seed;
  float xL, xR, yL, yR, zL, zR, RL, RR, cutoff, bcutoff;
  uint32_t grad_mask;
  double lr, beta1, beta2, eps;
} pinn_train_config;
typedef struct pinn_trainer pinn_trainer;
int pinn_trainer_create(pinn_handle* h, const pinn_train_config* cfg, const double* theta0_host, pinn_trainer** out);
int pinn_trainer_destroy(pinn_trainer* t);
/* Resume: parameters, Adam moments (NULL = zeros), optimizer steps already done (Adam's bias correction, the resampling
 * schedule and best_after keep counting from `step`).  The best-model record restarts (best_theta = theta, best loss back
 * to its initial limit, best_step = -1), the history restarts at row 0, and for best_mode 0 the first step after the
 * resume is taken unconditionally like the first step of a fresh run (train.py:58). */
int pinn_trainer_load_state(pinn_trainer* t, const double* theta, const double* m, const double* v, int64_t step);
int pinn_trainer_set_batch(pinn_trainer* t, const float* x, const float* y, const float* z, const float* R, const uint8_t* mask,
                           const double* weights_host);
int pinn_trainer_run(pinn_trainer* t, int64_t steps, int resample, int use_graph);
int pinn_trainer_read(pinn_trainer* t, double* theta, double* m, double* v, double* best_theta, double* scalars, double* history,
                      int64_t history_rows);
int pinn_trainer_batch(pinn_trainer* t, float** x, float** y, float** z, float** R, uint8_t** mask);
/* Residual-adaptive batches (pinn_sample_adaptive) for this trainer: every step that resamples draws its batch from
 * pool_factor * n candidates, at the float32 parameters the previous step's Adam update left, with the trainer's seed and
 * batch index (one index per draw).  The draw is enqueued in front of that step's step kernel: 6 launches more per
 * resampling step (8 in all), and no batch is drawn inside the reduction kernel while adaptive sampling is on.
 * use_graph = 1 replays the whole adaptive step as one graph of its own (same bits as plain launches).  The history and
 * the best-model record are evaluated on the adaptive batches, so Ltot is not comparable with a uniform run's (the
 * held-out loss of pinn_trainer_set_validation is).
 * pool_factor = 0 (the default) turns it off and frees the pool; the buffers of pool_factor * n points are allocated
 * here, never in pinn_trainer_run.  PINN_EINVAL for pool_factor < 0, or k or c negative or not finite; PINN_ENOTSUP while
 * the data-parallel exchange is on (pinn_trainer_run also refuses an adaptive trainer then). */
int pinn_trainer_set_adaptive(pinn_trainer* t, int pool_factor, float k, float c);
/* Importance weights for the adaptive batches of this trainer (on = 1; off = 0, the default): each adaptive draw is
 * pinn_sample_adaptive_importance, and every step on such a batch - the drawing step and the steps up to the next draw -
 * is pinn_loss_fwd_bwd_weighted with its omega and the pool-based loss weights.  The history and best-model record are
 * then an unbiased estimate of the pool's uniform loss.  use_graph replays the same launches.  pinn_trainer_set_adaptive
 * turns it off again.  PINN_EINVAL when adaptive sampling is off or its c is not > 0.  pinn_trainer_run_lbfgs refuses
 * (PINN_ENOTSUP) to evaluate an importance batch. */
int pinn_trainer_set_importance(pinn_trainer* t, int on);
/* Held-out validation loss during training.  This call draws the held-out set once, by the trainer's sampler with its box,
 * cutoff and bcutoff: it is pinn_sample(n_val, seed, 0, ...) bit for bit.  (Take a seed other than the training seed:
 * batch 0 of the training seed is the first training batch.)  From then on, every optimizer step of pinn_trainer_run that
 * brings the steps done since the run (re)started to a multiple of `every` is followed by one pinn_loss_eval of the set
 * at the float32 parameters that step left (weights: the counted sets, mask: the set's), two launches.  It writes row k
 * = {optimizer steps done, Ltot, Lpde, Lbc} of a device history of `capacity` rows (evaluations past it are counted, not
 * stored) and updates a best-on-validation record {best_val_loss, best_val_theta (float64), best_val_step}, which starts
 * at +inf / the trainer's current theta / -1 and takes an evaluation only when its Ltot is strictly lower (a NaN is never
 * taken).  Adam's history and best-model record, the batch sequence and every trainer state are unchanged by it; the
 * evaluation reads no batch buffer.  With use_graph = 1 the evaluations are plain launches between the step graphs (the
 * same bits).  The set, its rows and the record are allocated here, never in pinn_trainer_run; every = 0 turns
 * validation off and frees them.  pinn_trainer_load_state restarts the rows and the record.  PINN_EINVAL for every < 0,
 * or n_val <= 0 or capacity < 0 with every > 0; PINN_ENOTSUP while the data-parallel exchange is on (pinn_trainer_run
 * also refuses a trainer with validation on then). */
int pinn_trainer_set_validation(pinn_trainer* t, int64_t n_val, uint64_t seed, int64_t every, int64_t capacity);
/* One validation evaluation now, at the current theta32 (a step-0 point, or after pinn_trainer_run_lbfgs): a row and the
 * record as above.  PINN_EINVAL when validation is off. */
int pinn_trainer_validate(pinn_trainer* t);
/* Synchronise and read: up to max_rows rows of 4 doubles, best_val_theta (1521 doubles), scalars = {evaluations
 * recorded, best_val_loss, best_val_step}.  Any pointer may be NULL.  PINN_EINVAL when validation is off. */
int pinn_trainer_read_validation(pinn_trainer* t, double* rows, int64_t max_rows, double* best_val_theta, double* scalars);
void* pinn_trainer_stream(pinn_trainer* t);

/*
 * L-BFGS: torch.optim.LBFGS.step(closure) of torch 2.11 (torch/optim/lbfgs.py with _strong_wolfe and _cubic_interpolate)
 * in float64 on the device, decision for decision, as a machine that advances by ONE closure evaluation per launch and
 * needs no host synchronisation inside a .step() call.  The closure is Ltot and its gradient at theta.
 *
 * The state is caller-owned device memory of pinn_lbfgs_state_bytes(history_size) bytes; all zero bytes is a fresh
 * optimizer (torch's empty state), and d, t, the history, H_diag, prev_flat_grad, prev_loss, n_iter and func_evals
 * persist in it across calls.  Keep history_size the same for the life of a state.  Its first 8 doubles are the status:
 *   [0] n_iter (torch's state["n_iter"])   [1] func_evals (state["func_evals"])   [2] evaluations in this call
 *   [3] done (1 once the call has finished)  [4] reason (PINN_LBFGS_*)   [5] loss (torch's `loss` when it finished)
 *   [6] iterations in this call            [7] step length of the point requested last (0 for the first evaluation)
 * A call:  pinn_lbfgs_begin requests an evaluation at theta (it writes theta32 = (float)theta).  Then, until done: evaluate
 * the loss and gradient at the requested point (sums[0] = loss, grad = its 1521 doubles; a frozen entry has gradient 0, as
 * torch's _gather_flat_grad gives for a parameter without .grad) and call pinn_lbfgs_advance, which consumes it and
 * writes the next point to evaluate into theta (float64) and theta32, or finishes: theta = torch's final iterate.  After
 * done, pinn_lbfgs_advance changes nothing.  A call takes at most max_eval evaluations, or max_eval + 1 with the line
 * search (torch's line search always evaluates its first trial, even when max_eval has been reached).
 * Every reduction has a fixed order: the same inputs give the same bits on every run and under graph replay.
 * All pointers are device memory; PINN_EINVAL, with nothing launched, for a NULL pointer or a bad config.
 */
typedef struct pinn_lbfgs_config {
  double lr;                /* torch: lr = 1 */
  int max_iter;             /* 20; >= 1 */
  int max_eval;             /* <= 0: torch's default max_iter * 5 / 4 */
  int history_size;         /* 100; >= 1 */
  int line_search;          /* 0: line_search_fn = None (fixed step); 1: "strong_wolfe" */
  double tolerance_grad;    /* 1e-7 */
  double tolerance_change;  /* 1e-9 (the line search keeps its own 1e-9, like torch) */
} pinn_lbfgs_config;
/* status[4]: why the call finished, in the order torch tests */
#define PINN_LBFGS_RUNNING 0
#define PINN_LBFGS_OPTIMAL_AT_START 1         /* max|g| <= tolerance_grad at the first evaluation */
#define PINN_LBFGS_DIRECTIONAL_DERIVATIVE 2   /* g.d > -tolerance_change */
#define PINN_LBFGS_MAX_ITER 3
#define PINN_LBFGS_MAX_EVAL 4
#define PINN_LBFGS_TOLERANCE_GRAD 5           /* max|g| <= tolerance_grad after a step */
#define PINN_LBFGS_STEP_CHANGE 6              /* lack of progress: max|t d| <= tolerance_change */
#define PINN_LBFGS_LOSS_CHANGE 7              /* lack of progress: |loss - prev_loss| < tolerance_change */
#define PINN_LBFGS_SLOTS_EXHAUSTED 8          /* safety stop: more evaluations than the call can take (not expected) */
size_t pinn_lbfgs_state_bytes(int history_size); /* 0 for history_size < 1 */
int pinn_lbfgs_begin(pinn_handle* h, void* state, const pinn_lbfgs_config* cfg, const double* theta, float* theta32,
                     void* stream);
int pinn_lbfgs_advance(pinn_handle* h, void* state, const double* sums, const double* grad, double* theta, float* theta32,
                       void* stream);
/* One .step() call of the trainer on its current batch (resample = 1: the trainer's sampler draws the next batch first;
 * 0: the batch is kept, PINN_EINVAL if there is none yet).  Each evaluation is the step kernel at theta32, the reduction
 * (no Adam, no batch drawn) and the L-BFGS kernel, with the trainer's grad_mask.  use_graph = 0 enqueues every slot the
 * call may take (max_eval, + 1 with the line search): slots after termination change no state, but their step kernels
 * still run.  use_graph = 1 replays one evaluation as the body of a CUDA conditional WHILE node, and the L-BFGS kernel
 * ends the loop when the call finishes, so nothing runs past the end.  The first L-BFGS evaluation of a trainer runs as
 * plain launches.  Adam's moments and step counter, the best-model record and the history are not touched, so Adam can
 * run again afterwards; pinn_trainer_load_state resets the L-BFGS state.  The state is allocated on first use and again
 * (fresh) when history_size changes, in this call.  PINN_ENOTSUP with the data-parallel exchange on, and for resample = 1
 * with adaptive sampling on. */
int pinn_trainer_run_lbfgs(pinn_trainer* t, const pinn_lbfgs_config* cfg, int resample, int use_graph);
/* Synchronise; status: the 8 doubles above (all 0 before the first call); trace: up to `rows` rows of the last call,
 * one per evaluation: {Ltot, Lpde, Lbc, step length of the point}.  Either may be NULL. */
int pinn_trainer_read_lbfgs(pinn_trainer* t, double* status, double* trace, int64_t rows);

/*
 * E(R) of the E-net with its first and second derivative (autograd in poc/main.py:1324-1332) and the gate g(R)
 * (returnGate, poc/main.py:164-176; energy.py:26-31 evaluates the same E-net).  theta: device float32 [1521];
 * R: device float64 [n]; outputs device float64 [n], any may be NULL.
 */
int pinn_enet_curve(pinn_handle* h, const float* theta, const double* R, int n, double* E, double* dE, double* d2E, double* gate,
                    void* stream);

/*
 * Dense-grid quadrature at one R: replaces the grid evaluation + integra3d of energy_from_psi,
 * energy_from_psi_LCAO and dEdR_int (poc/main.py:438-494, 646-676, 179-186) without materialising the grid.
 * Grid = meshgrid('ij') of linspace(lim[0],lim[1],nx) x linspace(lim[2],lim[3],ny) x linspace(lim[4],lim[5],nz);
 * wx, wy, wz: device float64 1-D quadrature weights (Simpson; the product rule equals the nested simps calls).
 * out (device, 8 double): {sum w psi H psi, sum w psi^2, sum w lcao H lcao, sum w lcao^2, sum w dV/dR psi^2, E_net(R), 0, 0}
 * so that E_int = out[0]/out[1], E_lcao = out[2]/out[3], dE/dR|HF = out[4]/out[1] - 1/(2 R^2).
 */
int pinn_grid_reduce(pinn_handle* h, int variant, const float* theta, int nx, int ny, int nz, const double lim[6], double R,
                     const double* wx, const double* wy, const double* wz, double* out, void* stream);

/*
 * Converged E(R): the Rayleigh-quotient sums of pinn_grid_reduce for a whole sweep of R in one launch (+ one finishing
 * reduction), on a prolate-spheroidal node set instead of a Cartesian grid.  With the nuclei at x = +-R,
 * s = (r1 + r2)/2 - R >= 0 and nu = (r2 - r1)/(2R) in [-1, 1], the point of node (s_i, nu_j) at R is
 *     x = R (1 + s/R) nu,  y = sqrt(s (2R + s) (1 - nu^2)),  z = 0      (each operation in double, rounded as written)
 * with weight 2 pi ws_i wnu_j ((R + s)^2 - (R nu)^2): the volume element r1 r2 ds dnu dphi cancels every 1/r of H psi and
 * tensor Gauss-Legendre nodes converge exponentially (the model depends on (x,y,z) through r1, r2 only).
 * R: device float64 [nR], every value > 0 - a row with R <= 0 is all NaN (R is not read on the host).
 * s, ws: device float64 [ns]; nu, wnu: device float64 [nnu].  A node with s = 0 and nu = +-1 sits on a nucleus and gives
 * NaN sums, like a grid point on a nucleus in pinn_grid_reduce.
 * out (device, [nR][8] double): the row layout of pinn_grid_reduce per R, except slot 4 (the Hellmann-Feynman integrand
 * is not smooth in these coordinates) = 0.  Rows are deterministic: row k is the same bits as a call with R[k] alone.
 * nR * ceil(ns * nnu / 128) * 128 must stay below 2^31.  The call keeps 256 bytes per 128 node slots of one R for the largest
 * sweep made so far on the stream (grown on a larger call, which is therefore not CUDA-graph capturable: make the largest call
 * once outside the capture first).
 */
int pinn_spheroidal_reduce(pinn_handle* h, int variant, const float* theta, int nR, const double* R, int ns, const double* s,
                           const double* ws, int nnu, const double* nu, const double* wnu, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PINN_B200_H */
