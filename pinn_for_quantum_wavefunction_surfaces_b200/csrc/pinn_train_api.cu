// C ABI of the rows next to the hot path (include/pinn_b200.h, "training loop" and "analysis" sections):
// sampler, fused Adam, the device-resident trainer (CUDA-graph replay of sample -> loss -> Adam), the E(R)/gate
// curve and the dense-grid quadrature sums.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>

#include "pinn_handle.h"
#include "pinn_train.h"

namespace {
__global__ void set_u64_kernel(unsigned long long* p, unsigned long long v) { *p = v; }
}  // namespace

struct pinn_trainer {
  pinn_handle* h = nullptr;
  pinn_train_config cfg{};
  cudaStream_t st = nullptr;
  // two batch buffers: the step works on buffer `cur` while the sampler blocks riding in its reduction kernel draw the
  // next batch into the other one
  float *x[2] = {nullptr, nullptr}, *y[2] = {nullptr, nullptr}, *z[2] = {nullptr, nullptr}, *R[2] = {nullptr, nullptr};
  uint8_t* mask[2] = {nullptr, nullptr};
  double* weights[2] = {nullptr, nullptr};
  unsigned long long* counts[2] = {nullptr, nullptr};  // per buffer {|set1|, |set2|, sampler ticket, -}
  int cur = 0;
  bool next_ready = false;  // buffer cur^1 holds the batch of the next step
  float *E = nullptr, *theta32 = nullptr;
  unsigned long long *batch = nullptr, *step = nullptr, *adam_ticket = nullptr;
  long long* best_step = nullptr;
  double *theta = nullptr, *m = nullptr, *v = nullptr, *grad = nullptr, *sums = nullptr;
  double *best_loss = nullptr, *best_theta = nullptr, *hist = nullptr;
  cudaGraphExec_t graph[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [cur][draw the next batch too]
  bool warmed = false;  // one plain step has run: one-time kernel attributes are set outside any capture
  int64_t steps_issued = 0;
  int64_t step_base = 0;  // optimizer steps done when the run (re)started (pinn_trainer_load_state)
  bool have_batch = false;
  // residual-adaptive sampling (pinn_trainer_set_adaptive): pool_factor * n candidates per resampling step; off at 0
  int pool_factor = 0;
  float ad_k = 1.0f, ad_c = 1.0f;
  // importance weights (pinn_trainer_set_importance): the adaptive draw also writes omega into pw (n floats, allocated by
  // the first call that turns it on), and every step whose batch came from such a draw (pw_batch) runs the weighted
  // training evaluation on it
  bool importance = false, pw_batch = false;
  float* pw = nullptr;
  float *px = nullptr, *py = nullptr, *pz = nullptr, *pR = nullptr, *pres = nullptr;
  uint8_t* pmask = nullptr;
  double *pcdf = nullptr, *pweights = nullptr, *ppart = nullptr;
  unsigned long long* pcounts = nullptr;  // {|set1|, |set2|, ticket} of the pool's draw, [3] scratch batch word of the selection
  cudaGraphExec_t graph_ad[2] = {nullptr, nullptr};  // [cur]: adaptive draw + step
  cudaGraphExec_t graph_w[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // as graph[][], on an importance batch
  bool ad_warmed = false;  // one plain adaptive step has run (the inference kernel's attributes are set)
  // L-BFGS (pinn_trainer_run_lbfgs): state of lb_hist pairs, trace [lb_trace_rows][4], the WHILE graph of one evaluation
  unsigned char* lb_state = nullptr;
  int lb_hist = 0;
  double* lb_trace = nullptr;
  int64_t lb_trace_rows = 0;
  cudaGraphExec_t graph_lb[2] = {nullptr, nullptr};  // [cur]
  bool lb_warmed = false;  // one plain L-BFGS evaluation has run
  // held-out validation (pinn_trainer_set_validation): val_n fixed points, evaluated every val_every steps; off at 0
  int64_t val_every = 0, val_n = 0, val_cap = 0;
  float *vx = nullptr, *vy = nullptr, *vz = nullptr, *vR = nullptr;
  uint8_t* vmask = nullptr;
  unsigned long long* vwords = nullptr;  // {|set1|, |set2|, batch index, ticket} of the set's draw; [4] evaluations recorded
  double *vweights = nullptr, *vpart = nullptr, *vsums = nullptr, *vrows = nullptr;
  double *vbest_loss = nullptr, *vbest_theta = nullptr;
  long long* vbest_step = nullptr;
};

// Launches of one adaptive draw on top of the pool's sampler: the pool's residual and the four selection kernels
constexpr int ADAPTIVE_LAUNCHES = 6;

// Pool of pool.n points (launch_sample), its residual at theta (the inference instance of the step kernel), then the
// selection of a.out.n points (pinn_adaptive.cu).  The handle mutex is held by the caller.
static int adaptive_enqueue(pinn_handle* h, int nev, const VariantCoef& vc, const float* theta, const SampleParams& pool,
                            bool zero_pool_counts, const AdaptiveParams& a, cudaStream_t st) {
  CU(h, launch_sample(pool, zero_pool_counts, st));
  StepParams p{};
  p.vc = vc; p.x = pool.x; p.y = pool.y; p.z = pool.z; p.R = pool.R; p.n = pool.n; p.theta = theta;
  p.res = const_cast<float*>(a.res);
  CU(h, launch_step_tc(nev, false, p, grid_for(h, pool.n), st));
  CU(h, launch_adaptive_select(a, st));
  h->launches += ADAPTIVE_LAUNCHES + (zero_pool_counts ? 1 : 0);
  return 0;
}

static SampleParams sampler_params(pinn_trainer* t, int buf) {
  pinn_handle* h = t->h;
  const pinn_train_config& c = t->cfg;
  SampleParams s{};
  s.n = c.n; s.seed = c.seed; s.batch_counter = t->batch;
  s.xL = c.xL; s.xR = c.xR; s.yL = c.yL; s.yR = c.yR; s.zL = c.zL; s.zR = c.zR; s.RL = c.RL; s.RR = c.RR;
  s.cutoff = c.cutoff; s.bcutoff = c.bcutoff;
  s.x = t->x[buf]; s.y = t->y[buf]; s.z = t->z[buf]; s.R = t->R[buf]; s.mask = t->mask[buf]; s.counts = t->counts[buf];
  // data-parallel: rank r draws points [r n, (r+1) n) of the global batch of world*n points, so the union over the
  // ranks is exactly the batch a single GPU would draw for n_global = world*n
  s.dp = dp_active(h);
  s.index_offset = (long long)s.dp.rank * c.n;
  s.weights = t->weights[buf]; s.ticket = t->counts[buf] + 2; s.reset_counts = 1;
  return s;
}

// One optimizer step on buffer t->cur.  sample_now: draw its batch first with the stand-alone sampler kernel (the first
// resampling step of a run); presample_next: the reduction kernel also draws the batch of the NEXT step into the other buffer.
static int trainer_enqueue(pinn_trainer* t, bool sample_now, bool adaptive_now, bool presample_next, cudaStream_t st) {
  pinn_handle* h = t->h;
  const pinn_train_config& c = t->cfg;
  const int b = t->cur;
  if (sample_now) {
    const SampleParams s = sampler_params(t, b);
    CU(h, launch_sample(s, false, st));
    h->launches += 1;
  }
  if (adaptive_now) {
    // the pool takes the trainer's batch index (and moves it on); the selection writes buffer b like the sampler would
    SampleParams pool = sampler_params(t, b);
    pool.n = (long long)t->pool_factor * c.n; pool.index_offset = 0;
    pool.x = t->px; pool.y = t->py; pool.z = t->pz; pool.R = t->pR; pool.mask = t->pmask;
    pool.counts = t->pcounts; pool.ticket = t->pcounts + 2; pool.weights = t->pweights;
    AdaptiveParams a{};
    a.pool = pool.n; a.k = t->ad_k; a.c = t->ad_c;
    a.px = t->px; a.py = t->py; a.pz = t->pz; a.pR = t->pR; a.pmask = t->pmask; a.res = t->pres;
    a.cdf = t->pcdf; a.part = t->ppart; a.pool_batch = t->batch; a.idx = nullptr;
    a.out = sampler_params(t, b);
    a.out.index_offset = 0; a.out.batch_counter = t->pcounts + 3;
    if (t->importance) {  // the selection reads the pool's set sizes, then zeroes them
      a.point_w = t->pw; a.pool_counts = t->pcounts;
      pool.reset_counts = 0;
    }
    VariantCoef vc;
    int nev = 0;
    variant_coef(c.variant, &vc, &nev);
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = adaptive_enqueue(h, nev, vc, t->theta32, pool, false, a, st)) return rc;
  }
  AdamParams a{};
  a.theta = t->theta; a.m = t->m; a.v = t->v; a.grad = t->grad; a.sums = t->sums; a.theta32 = t->theta32;
  a.step = t->step; a.best_loss = t->best_loss; a.best_theta = t->best_theta; a.best_step = t->best_step;
  a.hist = t->hist; a.hist_cap = c.history_capacity;
  a.n = c.n * std::max(1, dp_active(h).world);  // mean E of the history is over the global batch
  a.lr = c.lr; a.beta1 = c.beta1; a.beta2 = c.beta2; a.eps = c.eps; a.best_after = (double)c.best_after;
  a.grad_mask = c.grad_mask; a.best_mode = c.best_mode; a.hist_mean_E = c.history_mean_E;
  a.step_base = (unsigned long long)t->step_base;
  SampleParams next{};
  if (presample_next) next = sampler_params(t, b ^ 1);
  // the optimizer step (and the next batch) ride in the reduction kernel: two launches per step
  LossCall lc;
  lc.variant = c.variant; lc.n = c.n; lc.x = t->x[b]; lc.y = t->y[b]; lc.z = t->z[b]; lc.R = t->R[b]; lc.in_dtype = PINN_F32;
  lc.mask = t->mask[b]; lc.theta = t->theta32; lc.weights = t->weights[b]; lc.grad_mask = c.grad_mask; lc.bcutoff = c.bcutoff;
  lc.sums = t->sums; lc.dtheta = t->grad; lc.E_out = t->E; lc.adam = &a; lc.adam_ticket = t->adam_ticket;
  lc.presample = presample_next ? &next : nullptr;
  if (adaptive_now ? t->importance : t->pw_batch) lc.point_w = t->pw;
  int rc = loss_fwd_bwd_impl(h, lc, st);
  if (rc) return rc;
  return 0;
}

// One L-BFGS evaluation on buffer t->cur: the step kernel at theta32, the reduction (no Adam, no batch drawn), the L-BFGS
// kernel.  cond: the WHILE node of a graph body, or NULL.
static int lbfgs_eval_enqueue(pinn_trainer* t, const cudaGraphConditionalHandle* cond, cudaStream_t st) {
  pinn_handle* h = t->h;
  const pinn_train_config& c = t->cfg;
  const int b = t->cur;
  LossCall lc;
  lc.variant = c.variant; lc.n = c.n; lc.x = t->x[b]; lc.y = t->y[b]; lc.z = t->z[b]; lc.R = t->R[b]; lc.in_dtype = PINN_F32;
  lc.mask = t->mask[b]; lc.theta = t->theta32; lc.weights = t->weights[b]; lc.grad_mask = c.grad_mask; lc.bcutoff = c.bcutoff;
  lc.sums = t->sums; lc.dtheta = t->grad; lc.E_out = t->E;
  if (int rc = loss_fwd_bwd_impl(h, lc, st)) return rc;
  CU(h, launch_lbfgs_advance(t->lb_state, t->sums, t->grad, t->theta, t->theta32, t->lb_trace, t->lb_trace_rows, cond, st));
  h->launches += 1;
  return 0;
}

// The graph of one .step() call: a kernel that sets the condition to "not finished", then a conditional WHILE node whose
// body is one evaluation; the L-BFGS kernel clears the condition when the call finishes, so no evaluation runs past it.
static int lbfgs_capture(pinn_trainer* t, cudaGraphExec_t* out) {
  pinn_handle* h = t->h;
  cudaGraph_t g = nullptr;
  CU(h, cudaGraphCreate(&g, 0));
  cudaGraphConditionalHandle cond;
  cudaGraphNodeParams np = {};
  cudaGraphNode_t first = nullptr, node = nullptr;
  size_t nfirst = 1;
  cudaGraph_t body = nullptr;
  int rc = 0;
  cudaError_t e = cudaGraphConditionalHandleCreate(&cond, g, 0, 0);
  if (e == cudaSuccess) e = cudaStreamBeginCaptureToGraph(t->st, g, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal);
  if (e == cudaSuccess) {
    e = launch_lbfgs_cond(t->lb_state, cond, t->st);
    cudaGraph_t same = nullptr;
    const cudaError_t e2 = cudaStreamEndCapture(t->st, &same);
    if (e == cudaSuccess) e = e2;
  }
  if (e == cudaSuccess) e = cudaGraphGetNodes(g, &first, &nfirst);
  if (e == cudaSuccess) {
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = cond;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    e = cudaGraphAddNode(&node, g, &first, 1, &np);
  }
  if (e == cudaSuccess) e = cudaStreamBeginCaptureToGraph(t->st, np.conditional.phGraph_out[0], nullptr, nullptr, 0,
                                                         cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { cudaGraphDestroy(g); return fail(h, (int)e, "pinn_trainer_run_lbfgs: conditional graph"); }
  const int64_t launches_before = h->launches;
  rc = lbfgs_eval_enqueue(t, &cond, t->st);
  h->launches = launches_before;
  e = cudaStreamEndCapture(t->st, &body);
  if (rc) { cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) { cudaGraphDestroy(g); return fail(h, (int)e, "pinn_trainer_run_lbfgs: cudaStreamEndCapture"); }
  e = cudaGraphInstantiate(out, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return fail(h, (int)e, "pinn_trainer_run_lbfgs: cudaGraphInstantiate");
  return 0;
}

static void trainer_free_lbfgs(pinn_trainer* t) {
  for (cudaGraphExec_t& g : t->graph_lb)
    if (g) { cudaGraphExecDestroy(g); g = nullptr; }
  cudaFree(t->lb_state); cudaFree(t->lb_trace);
  t->lb_state = nullptr; t->lb_trace = nullptr;
  t->lb_hist = 0; t->lb_trace_rows = 0;
}

// One validation evaluation at theta32 on the held-out set: the LOSS instance of the step kernel and the finishing block,
// which also writes the row and updates the best-on-validation record.  Reads no batch buffer.
static int validation_enqueue(pinn_trainer* t) {
  pinn_handle* h = t->h;
  StepParams p{};
  int nev = 0;
  variant_coef(t->cfg.variant, &p.vc, &nev);
  p.x = t->vx; p.y = t->vy; p.z = t->vz; p.R = t->vR; p.mask = t->vmask; p.n = t->val_n; p.bcut = t->cfg.bcutoff;
  p.theta = t->theta32;
  p.grid.partials = t->vpart;
  const int grid = grid_for(h, t->val_n);
  LossValidation v{};
  v.on = 1; v.step = t->step; v.count = t->vwords + 4; v.rows = t->vrows; v.cap = t->val_cap;
  v.best_loss = t->vbest_loss; v.best_step = t->vbest_step; v.best_theta = t->vbest_theta; v.theta = t->theta;
  std::lock_guard<std::mutex> lk(h->mu);
  CU(h, launch_loss_tc(nev, p, grid, t->st));
  CU(h, launch_loss_finish(t->vpart, grid, t->val_n, nullptr, t->vsums, &v, t->st));
  h->launches += 2;
  return 0;
}

// The validation rows and record start again (the stream is idle): no rows, best loss +inf, best step -1, best theta =
// the trainer's current theta.
static int validation_reset(pinn_trainer* t) {
  pinn_handle* h = t->h;
  const double inf = INFINITY;
  const long long neg1 = -1;
  CU(h, cudaMemset(t->vwords + 4, 0, 8));
  CU(h, cudaMemset(t->vrows, 0, (size_t)t->val_cap * 4 * 8));
  CU(h, cudaMemcpy(t->vbest_loss, &inf, 8, cudaMemcpyHostToDevice));
  CU(h, cudaMemcpy(t->vbest_step, &neg1, 8, cudaMemcpyHostToDevice));
  CU(h, cudaMemcpy(t->vbest_theta, t->theta, NTHETA * 8, cudaMemcpyDeviceToDevice));
  return 0;
}

// Held-out set, rows and record (the stream is idle)
static void trainer_free_validation(pinn_trainer* t) {
  cudaFree(t->vx); cudaFree(t->vy); cudaFree(t->vz); cudaFree(t->vR); cudaFree(t->vmask); cudaFree(t->vwords);
  cudaFree(t->vweights); cudaFree(t->vpart); cudaFree(t->vsums); cudaFree(t->vrows);
  cudaFree(t->vbest_loss); cudaFree(t->vbest_theta); cudaFree(t->vbest_step);
  t->vx = t->vy = t->vz = t->vR = nullptr;
  t->vmask = nullptr;
  t->vwords = nullptr;
  t->vweights = t->vpart = t->vsums = t->vrows = t->vbest_loss = t->vbest_theta = nullptr;
  t->vbest_step = nullptr;
  t->val_every = t->val_n = t->val_cap = 0;
}

static int trainer_capture(pinn_trainer* t, bool adaptive_now, bool presample_next, cudaGraphExec_t* out) {
  pinn_handle* h = t->h;
  cudaGraph_t g = nullptr;
  CU(h, cudaStreamBeginCapture(t->st, cudaStreamCaptureModeThreadLocal));
  const int64_t launches_before = h->launches;
  int rc = trainer_enqueue(t, false, adaptive_now, presample_next, t->st);
  h->launches = launches_before;  // capture does not launch; replays are counted in pinn_trainer_run
  cudaError_t e = cudaStreamEndCapture(t->st, &g);
  if (rc) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) return fail(h, (int)e, "cudaStreamEndCapture");
  e = cudaGraphInstantiate(out, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return fail(h, (int)e, "cudaGraphInstantiate");
  return 0;
}

// Pool buffers and the adaptive graphs (the stream is idle)
// (the importance flag goes with the pool; pw and an importance batch in use stay: its remaining steps keep their weights)
static void trainer_free_adaptive(pinn_trainer* t) {
  for (cudaGraphExec_t& g : t->graph_ad)
    if (g) { cudaGraphExecDestroy(g); g = nullptr; }
  t->importance = false;
  cudaFree(t->px); cudaFree(t->py); cudaFree(t->pz); cudaFree(t->pR); cudaFree(t->pres); cudaFree(t->pmask);
  cudaFree(t->pcdf); cudaFree(t->pweights); cudaFree(t->ppart); cudaFree(t->pcounts);
  t->px = t->py = t->pz = t->pR = t->pres = nullptr;
  t->pmask = nullptr;
  t->pcdf = t->pweights = t->ppart = nullptr;
  t->pcounts = nullptr;
  t->pool_factor = 0;
}

extern "C" {

int pinn_sample(pinn_handle* h, int64_t n, uint64_t seed, uint64_t batch, const float box[8], float cutoff, float bcutoff,
                float* x, float* y, float* z, float* R, uint8_t* mask, uint64_t* counts, double* weights, void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (n <= 0 || !box || !x || !y || !z || !R || !mask || !counts || !weights)
    return fail(h, PINN_EINVAL, "pinn_sample: bad argument");
  DevGuard dev_guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  pinn_workspace* ws = ws_for(h, st, h->sm_count);
  if (!ws) return PINN_EINVAL;
  unsigned long long* batch_counter = ws->counts + 2;  // [2] batch index, [3] block ticket of the sampler
  set_u64_kernel<<<1, 1, 0, st>>>(batch_counter, (unsigned long long)batch);
  SampleParams s{};
  s.n = n; s.seed = seed; s.batch_counter = batch_counter;
  s.xL = box[0]; s.xR = box[1]; s.yL = box[2]; s.yR = box[3]; s.zL = box[4]; s.zR = box[5]; s.RL = box[6]; s.RR = box[7];
  s.cutoff = cutoff; s.bcutoff = bcutoff;
  s.x = x; s.y = y; s.z = z; s.R = R; s.mask = mask; s.counts = (unsigned long long*)counts;
  s.index_offset = 0;
  s.weights = weights; s.ticket = batch_counter + 1; s.reset_counts = 0;
  CU(h, launch_sample(s, true, st));
  h->launches += 2;
  return 0;
}

}  // extern "C"

// pinn_sample_adaptive and its importance form (point_w != NULL); `fn` names the entry in error messages
static int sample_adaptive_impl(const char* fn, pinn_handle* h, int variant, const float* theta, int64_t n, int64_t pool,
                                uint64_t seed, uint64_t batch, const float box[8], float cutoff, float bcutoff, float k, float c,
                                float* pool_x, float* pool_y, float* pool_z, float* pool_R, uint8_t* pool_mask, float* pool_res,
                                double* pool_cdf, float* x, float* y, float* z, float* R, uint8_t* mask, int64_t* idx,
                                uint64_t* counts, double* weights, float* point_w, void* stream) {
  std::lock_guard<std::mutex> lk(h->mu);
  std::string e = std::string(fn) + ": ";
  if (n <= 0 || pool < n) return fail(h, PINN_EINVAL, (e + "need 0 < n <= pool").c_str());
  if (!(k >= 0.0f) || !std::isfinite(k) || !(c >= 0.0f) || !std::isfinite(c))
    return fail(h, PINN_EINVAL, (e + "k and c must be finite and >= 0").c_str());
  // Lbc weights psi^2, not res^2: a candidate with zero residual must keep a positive probability
  if (point_w && !(c > 0.0f)) return fail(h, PINN_EINVAL, (e + "importance weights need c > 0").c_str());
  if (!theta || !box || !pool_x || !pool_y || !pool_z || !pool_R || !pool_mask || !pool_res || !pool_cdf || !x || !y || !z ||
      !R || !mask || !counts || !weights)
    return fail(h, PINN_EINVAL, (e + "NULL pointer argument").c_str());
  VariantCoef vc;
  int nev = 0;
  if (variant_coef(variant, &vc, &nev)) return fail(h, PINN_EINVAL, (e + "unknown variant").c_str());
  DevGuard dev_guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  const long long scratch_rows = (adaptive_scratch_doubles(pool) + NPART - 1) / NPART;
  if (scratch_rows > 0x7fffffffll) return fail(h, PINN_EINVAL, (e + "pool too large").c_str());
  pinn_workspace* ws = ws_for(h, st, std::max(h->sm_count, (int)scratch_rows));
  if (!ws) return PINN_EINVAL;
  unsigned long long* batch_counter = ws->counts + 2;  // [0..1] the pool's set sizes, [2] its batch index, [3] block ticket
  set_u64_kernel<<<1, 1, 0, st>>>(batch_counter, (unsigned long long)batch);
  CU(h, cudaGetLastError());
  h->launches += 1;
  SampleParams ps{};
  ps.n = pool; ps.seed = seed; ps.batch_counter = batch_counter;
  ps.xL = box[0]; ps.xR = box[1]; ps.yL = box[2]; ps.yR = box[3]; ps.zL = box[4]; ps.zR = box[5]; ps.RL = box[6]; ps.RR = box[7];
  ps.cutoff = cutoff; ps.bcutoff = bcutoff;
  ps.x = pool_x; ps.y = pool_y; ps.z = pool_z; ps.R = pool_R; ps.mask = pool_mask; ps.counts = ws->counts;
  ps.weights = ws->weights; ps.ticket = batch_counter + 1; ps.reset_counts = 0;
  AdaptiveParams a{};
  a.pool = pool; a.k = k; a.c = c;
  a.px = pool_x; a.py = pool_y; a.pz = pool_z; a.pR = pool_R; a.pmask = pool_mask; a.res = pool_res;
  a.cdf = pool_cdf; a.part = ws->partials; a.pool_batch = batch_counter; a.idx = reinterpret_cast<long long*>(idx);
  a.point_w = point_w; a.pool_counts = ws->counts;
  a.out = ps;
  a.out.n = n; a.out.x = x; a.out.y = y; a.out.z = z; a.out.R = R; a.out.mask = mask;
  a.out.counts = (unsigned long long*)counts; a.out.weights = weights;
  // rad_scan_kernel has read the pool's batch index by the time the selection's finish moves this word on again
  a.out.batch_counter = batch_counter;
  return adaptive_enqueue(h, nev, vc, theta, ps, true, a, st);
}

extern "C" {

int pinn_sample_adaptive(pinn_handle* h, int variant, const float* theta, int64_t n, int64_t pool, uint64_t seed, uint64_t batch,
                         const float box[8], float cutoff, float bcutoff, float k, float c, float* pool_x, float* pool_y,
                         float* pool_z, float* pool_R, uint8_t* pool_mask, float* pool_res, double* pool_cdf, float* x,
                         float* y, float* z, float* R, uint8_t* mask, int64_t* idx, uint64_t* counts, double* weights,
                         void* stream) {
  if (!h) return PINN_EINVAL;
  return sample_adaptive_impl("pinn_sample_adaptive", h, variant, theta, n, pool, seed, batch, box, cutoff, bcutoff, k, c, pool_x,
                              pool_y, pool_z, pool_R, pool_mask, pool_res, pool_cdf, x, y, z, R, mask, idx, counts, weights,
                              nullptr, stream);
}

int pinn_sample_adaptive_importance(pinn_handle* h, int variant, const float* theta, int64_t n, int64_t pool, uint64_t seed,
                                    uint64_t batch, const float box[8], float cutoff, float bcutoff, float k, float c,
                                    float* pool_x, float* pool_y, float* pool_z, float* pool_R, uint8_t* pool_mask,
                                    float* pool_res, double* pool_cdf, float* x, float* y, float* z, float* R, uint8_t* mask,
                                    int64_t* idx, uint64_t* counts, double* weights, float* point_w, void* stream) {
  if (!h) return PINN_EINVAL;
  if (!point_w) return fail(h, PINN_EINVAL, "pinn_sample_adaptive_importance: NULL pointer argument");
  return sample_adaptive_impl("pinn_sample_adaptive_importance", h, variant, theta, n, pool, seed, batch, box, cutoff, bcutoff,
                              k, c, pool_x, pool_y, pool_z, pool_R, pool_mask, pool_res, pool_cdf, x, y, z, R, mask, idx, counts,
                              weights, point_w, stream);
}

int pinn_adam_step(pinn_handle* h, double* theta, double* m, double* v, const double* grad, const double* sums, float* theta32,
                   uint64_t* step, double* best_loss, double* best_theta, int64_t* best_step, double* hist, int64_t hist_cap,
                   int64_t n, double lr, double beta1, double beta2, double eps, uint32_t grad_mask, int best_mode,
                   int64_t best_after, int history_mean_E, void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!theta || !m || !v || !grad || !sums || !theta32 || !step || !best_loss || !best_theta || !best_step)
    return fail(h, PINN_EINVAL, "pinn_adam_step: NULL pointer argument");
  DevGuard dev_guard(h->device);
  AdamParams a{};
  a.theta = theta; a.m = m; a.v = v; a.grad = grad; a.sums = sums; a.theta32 = theta32;
  a.step = (unsigned long long*)step; a.best_loss = best_loss; a.best_theta = best_theta; a.best_step = (long long*)best_step;
  a.hist = hist; a.hist_cap = hist_cap; a.n = n; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps;
  a.best_after = (double)best_after; a.grad_mask = grad_mask; a.best_mode = best_mode; a.hist_mean_E = history_mean_E;
  CU(h, launch_adam(a, (cudaStream_t)stream));
  h->launches += 1;
  return 0;
}

int pinn_measure_fp32_peak(pinn_handle* h, double* fma_per_s, double* ms, double* sm_mhz) {
  if (!h || !fma_per_s || !ms || !sm_mhz) return PINN_EINVAL;
  DevGuard dev_guard(h->device);
  CU(h, measure_fp32_peak(h->sm_count, h->s_main, fma_per_s, ms, sm_mhz));
  return 0;
}

// Effective SM clock of the LAST training evaluation enqueued on `stream` through this handle: CTA 0 of the step kernel
// times itself (clock64 and %globaltimer, entry to the end of its tile loop).  Synchronises the stream.
int pinn_step_kernel_clock(pinn_handle* h, void* stream, double* cycles, double* ns) {
  if (!h || !cycles || !ns) return PINN_EINVAL;
  DevGuard dev_guard(h->device);
  const double* src = nullptr;
  {
    std::lock_guard<std::mutex> lk(h->mu);
    for (const pinn_workspace& w : h->ws)
      if (w.stream == (cudaStream_t)stream && w.partials) src = w.partials + (NPART - 2);
  }
  if (!src) return fail(h, PINN_EINVAL, "pinn_step_kernel_clock: no training evaluation has run on this stream");
  CU(h, cudaStreamSynchronize((cudaStream_t)stream));
  double v[2];
  CU(h, cudaMemcpy(v, src, sizeof(v), cudaMemcpyDeviceToHost));
  *cycles = v[0]; *ns = v[1];
  return 0;
}

int pinn_enet_curve(pinn_handle* h, const float* theta, const double* R, int n, double* E, double* dE, double* d2E, double* gate,
                    void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!theta || !R || n <= 0) return fail(h, PINN_EINVAL, "pinn_enet_curve: bad argument");
  DevGuard dev_guard(h->device);
  CU(h, launch_enet_curve(theta, R, n, E, dE, d2E, gate, (cudaStream_t)stream));
  h->launches += 1;
  return 0;
}

int pinn_grid_reduce(pinn_handle* h, int variant, const float* theta, int nx, int ny, int nz, const double lim[6], double R,
                     const double* wx, const double* wy, const double* wz, double* out, void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!theta || !lim || !wx || !wy || !wz || !out) return fail(h, PINN_EINVAL, "pinn_grid_reduce: NULL pointer argument");
  if (nx < 2 || ny < 2 || nz < 2) return fail(h, PINN_EINVAL, "pinn_grid_reduce: every axis needs at least 2 points");
  StepParams p{};
  int nev = 0;
  if (variant_coef(variant, &p.vc, &nev)) return fail(h, PINN_EINVAL, "pinn_grid_reduce: unknown variant");
  DevGuard dev_guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  pinn_workspace* ws = ws_for(h, st, h->sm_count);
  if (!ws) return PINN_EINVAL;
  p.n = (long long)nx * ny * nz;
  p.theta = theta;
  p.grid.on = 1; p.grid.nx = nx; p.grid.ny = ny; p.grid.nz = nz;
  p.grid.x0 = lim[0]; p.grid.dx = (lim[1] - lim[0]) / (nx - 1);
  p.grid.y0 = lim[2]; p.grid.dy = (lim[3] - lim[2]) / (ny - 1);
  p.grid.z0 = lim[4]; p.grid.dz = (lim[5] - lim[4]) / (nz - 1);
  p.grid.R = R; p.grid.wx = wx; p.grid.wy = wy; p.grid.wz = wz; p.grid.partials = ws->grid_partials;
  const int grid = grid_for(h, p.n);
  CU(h, launch_step_tc(nev, false, p, grid, st));  // the dense-grid mode lives in the tcgen05 kernel
  CU(h, launch_grid_finish(ws->grid_partials, grid, out, st));
  h->launches += 2;
  return 0;
}

int pinn_spheroidal_reduce(pinn_handle* h, int variant, const float* theta, int nR, const double* R, int ns, const double* s,
                           const double* ws, int nnu, const double* nu, const double* wnu, double* out, void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!theta || !R || !s || !ws || !nu || !wnu || !out) return fail(h, PINN_EINVAL, "pinn_spheroidal_reduce: NULL pointer argument");
  if (nR < 1 || ns < 1 || nnu < 1) return fail(h, PINN_EINVAL, "pinn_spheroidal_reduce: nR, ns and nnu must be at least 1");
  StepParams p{};
  int nev = 0;
  if (variant_coef(variant, &p.vc, &nev)) return fail(h, PINN_EINVAL, "pinn_spheroidal_reduce: unknown variant");
  // every R owns whole super-tiles; the kernel's index arithmetic is 32-bit
  const long long tiles_per_R = ((long long)ns * nnu + 127) / 128;
  const long long tiles = tiles_per_R * nR;
  if (tiles * 128 >= 0x80000000ll)
    return fail(h, PINN_EINVAL, "pinn_spheroidal_reduce: nR * ceil(ns * nnu / 128) * 128 must stay below 2^31 points");
  DevGuard dev_guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  pinn_workspace* wk = ws_for(h, st, h->sm_count);
  if (!wk) return PINN_EINVAL;
  if (!ws_sph_rows(h, wk, st, (int)(tiles * 4))) return PINN_EINVAL;
  p.n = tiles * 128;
  p.theta = theta;
  p.grid.on = 1; p.grid.sph = 1;
  p.grid.ns = ns; p.grid.nnu = nnu; p.grid.tiles_per_R = (int)tiles_per_R;
  p.grid.Rs = R; p.grid.s = s; p.grid.ws = ws; p.grid.nu = nu; p.grid.wnu = wnu;
  p.grid.partials = wk->sph_partials;
  const int grid = grid_for(h, p.n);
  CU(h, launch_step_tc(nev, false, p, grid, st));
  CU(h, launch_sph_finish(wk->sph_partials, nR, (int)tiles_per_R * 4, R, out, st));
  h->launches += 2;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// device-resident trainer
// ---------------------------------------------------------------------------------------------
// pinn_trainer_create: a failing CUDA call releases the partially built trainer
#define TRAINER_CU(call)                                  \
  do {                                                    \
    cudaError_t e__ = (call);                             \
    if (e__ != cudaSuccess) {                             \
      pinn_trainer_destroy(t);                            \
      return fail(h, (int)e__, "pinn_trainer_create: " #call); \
    }                                                     \
  } while (0)

int pinn_trainer_create(pinn_handle* h, const pinn_train_config* cfg, const double* theta0_host, pinn_trainer** out) {
  if (!h) return PINN_EINVAL;
  if (!cfg || !theta0_host || !out) return fail(h, PINN_EINVAL, "pinn_trainer_create: NULL pointer argument");
  if (cfg->n <= 0 || cfg->sc_sampling <= 0 || cfg->history_capacity < 0)
    return fail(h, PINN_EINVAL, "pinn_trainer_create: n and sc_sampling must be positive");
  if (cfg->variant != PINN_VARIANT_POC && cfg->variant != PINN_VARIANT_TRAINPY)
    return fail(h, PINN_EINVAL, "pinn_trainer_create: unknown variant");
  DevGuard dev_guard(h->device);
  pinn_trainer* t = new pinn_trainer();
  t->h = h; t->cfg = *cfg;
  *out = nullptr;
  const size_t n = (size_t)cfg->n;
  TRAINER_CU(cudaStreamCreateWithFlags(&t->st, cudaStreamNonBlocking));
  for (int b = 0; b < 2; b++) {
    TRAINER_CU(cudaMalloc(&t->x[b], n * 4)); TRAINER_CU(cudaMalloc(&t->y[b], n * 4)); TRAINER_CU(cudaMalloc(&t->z[b], n * 4));
    TRAINER_CU(cudaMalloc(&t->R[b], n * 4)); TRAINER_CU(cudaMalloc(&t->mask[b], n));
    TRAINER_CU(cudaMalloc(&t->weights[b], 4 * 8));
    TRAINER_CU(cudaMalloc(&t->counts[b], 32)); TRAINER_CU(cudaMemset(t->counts[b], 0, 32));
  }
  TRAINER_CU(cudaMalloc(&t->E, n * 4));
  TRAINER_CU(cudaMalloc(&t->theta32, NPART * 4));
  TRAINER_CU(cudaMalloc(&t->batch, 8)); TRAINER_CU(cudaMalloc(&t->step, 8)); TRAINER_CU(cudaMalloc(&t->best_step, 8));
  TRAINER_CU(cudaMalloc(&t->adam_ticket, 8)); TRAINER_CU(cudaMemset(t->adam_ticket, 0, 8));
  TRAINER_CU(cudaMalloc(&t->theta, NPART * 8)); TRAINER_CU(cudaMalloc(&t->m, NPART * 8)); TRAINER_CU(cudaMalloc(&t->v, NPART * 8));
  TRAINER_CU(cudaMalloc(&t->grad, NPART * 8)); TRAINER_CU(cudaMalloc(&t->sums, 8 * 8));
  TRAINER_CU(cudaMalloc(&t->best_loss, 8)); TRAINER_CU(cudaMalloc(&t->best_theta, NPART * 8));
  if (cfg->history_capacity > 0) {
    TRAINER_CU(cudaMalloc(&t->hist, (size_t)cfg->history_capacity * 4 * 8));
    TRAINER_CU(cudaMemset(t->hist, 0, (size_t)cfg->history_capacity * 4 * 8));
  }
  TRAINER_CU(cudaMemset(t->m, 0, NPART * 8)); TRAINER_CU(cudaMemset(t->v, 0, NPART * 8));
  TRAINER_CU(cudaMemset(t->batch, 0, 8)); TRAINER_CU(cudaMemset(t->step, 0, 8));
  const long long neg1 = -1;
  TRAINER_CU(cudaMemcpy(t->best_step, &neg1, 8, cudaMemcpyHostToDevice));
  const double llim = 10.0;  // poc/main.py:370 Llim = 10; train.py takes the first loss unconditionally
  TRAINER_CU(cudaMemcpy(t->best_loss, &llim, 8, cudaMemcpyHostToDevice));
  TRAINER_CU(cudaMemcpy(t->theta, theta0_host, NTHETA * 8, cudaMemcpyHostToDevice));
  TRAINER_CU(cudaMemcpy(t->best_theta, theta0_host, NTHETA * 8, cudaMemcpyHostToDevice));
  float th32[NTHETA];
  for (int i = 0; i < NTHETA; i++) th32[i] = (float)theta0_host[i];
  TRAINER_CU(cudaMemcpy(t->theta32, th32, NTHETA * 4, cudaMemcpyHostToDevice));
  *out = t;
  return 0;
}

int pinn_trainer_destroy(pinn_trainer* t) {
  if (!t) return 0;
  DevGuard dev_guard(t->h->device);
  if (t->st) cudaStreamSynchronize(t->st);
  for (int a = 0; a < 2; a++)
    for (int b = 0; b < 2; b++) {
      if (t->graph[a][b]) cudaGraphExecDestroy(t->graph[a][b]);
      if (t->graph_w[a][b]) cudaGraphExecDestroy(t->graph_w[a][b]);
    }
  trainer_free_adaptive(t);
  cudaFree(t->pw);
  trainer_free_lbfgs(t);
  trainer_free_validation(t);
  for (int b = 0; b < 2; b++) {
    cudaFree(t->x[b]); cudaFree(t->y[b]); cudaFree(t->z[b]); cudaFree(t->R[b]); cudaFree(t->mask[b]);
    cudaFree(t->weights[b]); cudaFree(t->counts[b]);
  }
  cudaFree(t->E); cudaFree(t->theta32); cudaFree(t->batch); cudaFree(t->step); cudaFree(t->best_step); cudaFree(t->adam_ticket);
  cudaFree(t->theta); cudaFree(t->m); cudaFree(t->v); cudaFree(t->grad); cudaFree(t->sums);
  cudaFree(t->best_loss); cudaFree(t->best_theta); cudaFree(t->hist);
  if (t->st) {
    {
      std::lock_guard<std::mutex> lk(t->h->mu);
      ws_release(t->h, t->st);  // the stream handle dies here: its workspace (referenced by the graphs above) goes with it
    }
    cudaStreamDestroy(t->st);
  }
  delete t;
  return 0;
}

// Optimizer state / a resumed run: theta, m, v are 1521 host doubles (m, v may be NULL = zeros), `step` optimizer steps done.
int pinn_trainer_load_state(pinn_trainer* t, const double* theta, const double* m, const double* v, int64_t step) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (!theta || step < 0) return fail(h, PINN_EINVAL, "pinn_trainer_load_state: bad argument");
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  CU(h, cudaMemcpy(t->theta, theta, NTHETA * 8, cudaMemcpyHostToDevice));
  float th32[NTHETA];
  for (int i = 0; i < NTHETA; i++) th32[i] = (float)theta[i];
  CU(h, cudaMemcpy(t->theta32, th32, NTHETA * 4, cudaMemcpyHostToDevice));
  if (m) CU(h, cudaMemcpy(t->m, m, NTHETA * 8, cudaMemcpyHostToDevice)); else CU(h, cudaMemset(t->m, 0, NPART * 8));
  if (v) CU(h, cudaMemcpy(t->v, v, NTHETA * 8, cudaMemcpyHostToDevice)); else CU(h, cudaMemset(t->v, 0, NPART * 8));
  const unsigned long long s = (unsigned long long)step;
  CU(h, cudaMemcpy(t->step, &s, 8, cudaMemcpyHostToDevice));
  // a resumed run starts its own best-model record and history: the loaded parameters are the best known so far, the
  // loss limit is back at its initial value, history row 0 is the first step after the resume
  CU(h, cudaMemcpy(t->best_theta, theta, NTHETA * 8, cudaMemcpyHostToDevice));
  const double llim = 10.0;
  const long long neg1 = -1;
  CU(h, cudaMemcpy(t->best_loss, &llim, 8, cudaMemcpyHostToDevice));
  CU(h, cudaMemcpy(t->best_step, &neg1, 8, cudaMemcpyHostToDevice));
  if (t->hist) CU(h, cudaMemset(t->hist, 0, (size_t)t->cfg.history_capacity * 4 * 8));
  t->steps_issued = step;
  t->step_base = step;
  // captured graphs carry the old step_base in their kernel parameters
  for (int a = 0; a < 2; a++)
    for (int b = 0; b < 2; b++) {
      if (t->graph[a][b]) { cudaGraphExecDestroy(t->graph[a][b]); t->graph[a][b] = nullptr; }
      if (t->graph_w[a][b]) { cudaGraphExecDestroy(t->graph_w[a][b]); t->graph_w[a][b] = nullptr; }
    }
  for (cudaGraphExec_t& g : t->graph_ad)
    if (g) { cudaGraphExecDestroy(g); g = nullptr; }
  // the L-BFGS state restarts fresh (torch's empty state), like a new optimizer on the loaded parameters
  // on the trainer's stream (created non-blocking), so the next call's kernels are ordered after it
  if (t->lb_state) CU(h, cudaMemsetAsync(t->lb_state, 0, lbfgs_state_bytes(t->lb_hist), t->st));
  // the validation rows and record restart with the history (the memset above is on the non-blocking trainer stream)
  if (t->val_every > 0) {
    CU(h, cudaStreamSynchronize(t->st));
    if (int rc = validation_reset(t)) return rc;
  }
  return 0;
}

int pinn_trainer_set_validation(pinn_trainer* t, int64_t n_val, uint64_t seed, int64_t every, int64_t capacity) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (every < 0 || (every > 0 && (n_val <= 0 || capacity < 0)))
    return fail(h, PINN_EINVAL, "pinn_trainer_set_validation: need every >= 0, and n_val > 0 and capacity >= 0 when every > 0");
  if (every > 0 && dp_active(h).world > 1)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_set_validation: validation is not available with the data-parallel exchange");
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  trainer_free_validation(t);
  if (every == 0) return 0;
  const size_t n = (size_t)n_val;
#define VAL_CU(call)                                                           \
  do {                                                                         \
    cudaError_t e__ = (call);                                                  \
    if (e__ != cudaSuccess) {                                                  \
      trainer_free_validation(t);                                              \
      return fail(h, (int)e__, "pinn_trainer_set_validation: " #call);         \
    }                                                                          \
  } while (0)
  VAL_CU(cudaMalloc(&t->vx, n * 4)); VAL_CU(cudaMalloc(&t->vy, n * 4)); VAL_CU(cudaMalloc(&t->vz, n * 4));
  VAL_CU(cudaMalloc(&t->vR, n * 4)); VAL_CU(cudaMalloc(&t->vmask, n));
  VAL_CU(cudaMalloc(&t->vwords, 5 * 8)); VAL_CU(cudaMemset(t->vwords, 0, 5 * 8));
  VAL_CU(cudaMalloc(&t->vweights, 4 * 8));
  VAL_CU(cudaMalloc(&t->vpart, (size_t)(h->sm_count + 1) * 8 * 8));
  VAL_CU(cudaMalloc(&t->vsums, 8 * 8));
  VAL_CU(cudaMalloc(&t->vrows, (size_t)std::max<int64_t>(capacity, 1) * 4 * 8));
  VAL_CU(cudaMalloc(&t->vbest_loss, 8)); VAL_CU(cudaMalloc(&t->vbest_theta, NPART * 8)); VAL_CU(cudaMalloc(&t->vbest_step, 8));
#undef VAL_CU
  t->val_every = every; t->val_n = n_val; t->val_cap = capacity;
  // the held-out set: pinn_sample(n_val, seed, 0, box, cutoff, bcutoff), drawn once, here
  const pinn_train_config& c = t->cfg;
  SampleParams s{};
  s.n = n_val; s.seed = seed; s.batch_counter = t->vwords + 2;
  s.xL = c.xL; s.xR = c.xR; s.yL = c.yL; s.yR = c.yR; s.zL = c.zL; s.zR = c.zR; s.RL = c.RL; s.RR = c.RR;
  s.cutoff = c.cutoff; s.bcutoff = c.bcutoff;
  s.x = t->vx; s.y = t->vy; s.z = t->vz; s.R = t->vR; s.mask = t->vmask; s.counts = t->vwords;
  s.index_offset = 0;
  s.weights = t->vweights; s.ticket = t->vwords + 3; s.reset_counts = 0;
  int rc = 0;
  cudaError_t e = launch_sample(s, true, t->st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(t->st);
  if (e != cudaSuccess) rc = fail(h, (int)e, "pinn_trainer_set_validation: drawing the held-out set");
  if (!rc) rc = validation_reset(t);
  if (rc) { trainer_free_validation(t); return rc; }
  {
    std::lock_guard<std::mutex> lk(h->mu);
    h->launches += 1;
  }
  return 0;
}

int pinn_trainer_validate(pinn_trainer* t) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (t->val_every <= 0) return fail(h, PINN_EINVAL, "pinn_trainer_validate: validation is off (pinn_trainer_set_validation)");
  if (dp_active(h).world > 1)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_validate: validation is not available with the data-parallel exchange");
  DevGuard dev_guard(h->device);
  return validation_enqueue(t);
}

int pinn_trainer_read_validation(pinn_trainer* t, double* rows, int64_t max_rows, double* best_val_theta, double* scalars) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (t->val_every <= 0) return fail(h, PINN_EINVAL, "pinn_trainer_read_validation: validation is off");
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  if (rows && max_rows > 0) {
    const int64_t r = std::min(max_rows, t->val_cap);
    if (r > 0) CU(h, cudaMemcpy(rows, t->vrows, (size_t)r * 4 * 8, cudaMemcpyDeviceToHost));
  }
  if (best_val_theta) CU(h, cudaMemcpy(best_val_theta, t->vbest_theta, NTHETA * 8, cudaMemcpyDeviceToHost));
  if (scalars) {
    unsigned long long k = 0;
    long long bs = 0;
    double bl = 0.0;
    CU(h, cudaMemcpy(&k, t->vwords + 4, 8, cudaMemcpyDeviceToHost));
    CU(h, cudaMemcpy(&bl, t->vbest_loss, 8, cudaMemcpyDeviceToHost));
    CU(h, cudaMemcpy(&bs, t->vbest_step, 8, cudaMemcpyDeviceToHost));
    scalars[0] = (double)k; scalars[1] = bl; scalars[2] = (double)bs;
  }
  return 0;
}

int pinn_trainer_set_adaptive(pinn_trainer* t, int pool_factor, float k, float c) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (pool_factor < 0 || !(k >= 0.0f) || !std::isfinite(k) || !(c >= 0.0f) || !std::isfinite(c))
    return fail(h, PINN_EINVAL, "pinn_trainer_set_adaptive: pool_factor, k and c must be finite and >= 0");
  if (pool_factor > 0 && (int64_t)pool_factor > INT64_MAX / 8 / t->cfg.n)
    return fail(h, PINN_EINVAL, "pinn_trainer_set_adaptive: pool_factor * n too large");
  if (dp_active(h).world > 1)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_set_adaptive: adaptive sampling is not available with the data-parallel exchange");
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  trainer_free_adaptive(t);
  if (pool_factor == 0) return 0;
  const size_t N = (size_t)pool_factor * (size_t)t->cfg.n;
#define AD_CU(call)                                                            \
  do {                                                                         \
    cudaError_t e__ = (call);                                                  \
    if (e__ != cudaSuccess) {                                                  \
      trainer_free_adaptive(t);                                                \
      return fail(h, (int)e__, "pinn_trainer_set_adaptive: " #call);           \
    }                                                                          \
  } while (0)
  AD_CU(cudaMalloc(&t->px, N * 4)); AD_CU(cudaMalloc(&t->py, N * 4)); AD_CU(cudaMalloc(&t->pz, N * 4));
  AD_CU(cudaMalloc(&t->pR, N * 4)); AD_CU(cudaMalloc(&t->pres, N * 4)); AD_CU(cudaMalloc(&t->pmask, N));
  AD_CU(cudaMalloc(&t->pcdf, N * 8)); AD_CU(cudaMalloc(&t->pweights, 4 * 8));
  AD_CU(cudaMalloc(&t->ppart, (size_t)adaptive_scratch_doubles((long long)N) * 8));
  AD_CU(cudaMalloc(&t->pcounts, 32)); AD_CU(cudaMemset(t->pcounts, 0, 32));
#undef AD_CU
  t->pool_factor = pool_factor; t->ad_k = k; t->ad_c = c;
  t->ad_warmed = false;
  return 0;
}

int pinn_trainer_set_importance(pinn_trainer* t, int on) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (on && t->pool_factor <= 0)
    return fail(h, PINN_EINVAL, "pinn_trainer_set_importance: adaptive sampling is off (pinn_trainer_set_adaptive)");
  if (on && !(t->ad_c > 0.0f))
    return fail(h, PINN_EINVAL, "pinn_trainer_set_importance: importance weights need c > 0");
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  if (on && !t->pw) CU(h, cudaMalloc(&t->pw, (size_t)t->cfg.n * 4));
  if ((on != 0) != t->importance) {
    // the adaptive graphs were captured with the other selection and step; the first draw in the new mode runs plain
    for (cudaGraphExec_t& g : t->graph_ad)
      if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    t->ad_warmed = false;
  }
  t->importance = on != 0;
  return 0;
}

// Caller-provided batch instead of the sampler (parity runs feed the reference's own points): device float32 columns,
// mask bytes and the weights {1/n, 1/|set1|, 1/|set2|}; stays in use until the next resampling step.
int pinn_trainer_set_batch(pinn_trainer* t, const float* x, const float* y, const float* z, const float* R, const uint8_t* mask,
                           const double* weights_host) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (!x || !y || !z || !R || !mask || !weights_host) return fail(h, PINN_EINVAL, "pinn_trainer_set_batch: NULL pointer argument");
  DevGuard dev_guard(h->device);
  const size_t n = (size_t)t->cfg.n;
  const int b = t->cur;
  CU(h, cudaMemcpyAsync(t->x[b], x, n * 4, cudaMemcpyDefault, t->st));
  CU(h, cudaMemcpyAsync(t->y[b], y, n * 4, cudaMemcpyDefault, t->st));
  CU(h, cudaMemcpyAsync(t->z[b], z, n * 4, cudaMemcpyDefault, t->st));
  CU(h, cudaMemcpyAsync(t->R[b], R, n * 4, cudaMemcpyDefault, t->st));
  CU(h, cudaMemcpyAsync(t->mask[b], mask, n, cudaMemcpyDefault, t->st));
  CU(h, cudaMemcpyAsync(t->weights[b], weights_host, 3 * 8, cudaMemcpyDefault, t->st));
  CU(h, cudaStreamSynchronize(t->st));
  t->have_batch = true;
  t->pw_batch = false;
  return 0;
}

// Enqueue `steps` optimizer steps.  Step tt resamples iff tt % sc_sampling == 0 and tt < freeze_after (poc/main.py:396;
// train.py:25) - or never, when resample == 0 (the batch of pinn_trainer_set_batch is kept).  The batch of a resampling
// step is drawn by sampler blocks inside the reduction kernel of the step before it (into the other batch buffer) when
// that step belongs to the same call; the first resampling step of a call uses the stand-alone sampler kernel.  The
// sequence of batches is the same either way.  use_graph: steps without a stand-alone sampler replay one of four captured
// CUDA graphs (which buffer x whether the next batch is drawn) instead of launching their two kernels.
int pinn_trainer_run(pinn_trainer* t, int64_t steps, int resample, int use_graph) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  if (steps < 0) return fail(h, PINN_EINVAL, "pinn_trainer_run: steps must be >= 0");
  if (!resample && !t->have_batch) return fail(h, PINN_EINVAL, "pinn_trainer_run: no batch yet (resample = 0 needs pinn_trainer_set_batch or an earlier sampled step)");
  DevGuard dev_guard(h->device);
  const bool adaptive = t->pool_factor > 0;
  if (adaptive && dp_active(h).world > 1)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_run: adaptive sampling is not available with the data-parallel exchange");
  if (t->val_every > 0 && dp_active(h).world > 1)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_run: validation is not available with the data-parallel exchange");
  auto resamples = [&](int64_t tt) { return resample && (tt % t->cfg.sc_sampling == 0) && (tt < t->cfg.freeze_after); };
  for (int64_t k = 0; k < steps; k++) {
    const int64_t tt = t->steps_issued;
    const bool rs = resamples(tt);
    bool sample_now = false;
    // adaptive: the draw needs the parameters this step starts from, so it goes in front of the step, never in the
    // reduction kernel of the step before
    const bool adaptive_now = rs && adaptive;
    if (rs && !adaptive) {
      if (t->next_ready) { t->cur ^= 1; t->next_ready = false; }  // drawn while the previous step was reduced
      else sample_now = true;
    }
    if (rs) t->pw_batch = adaptive_now && t->importance;  // the batch of this step, and of the steps up to the next draw
    const bool presample_next = !adaptive && (k + 1 < steps) && resamples(tt + 1);
    if (use_graph && t->warmed && !sample_now && (!adaptive_now || t->ad_warmed)) {
      cudaGraphExec_t& g = adaptive_now ? t->graph_ad[t->cur]
                           : t->pw_batch ? t->graph_w[t->cur][presample_next ? 1 : 0] : t->graph[t->cur][presample_next ? 1 : 0];
      if (!g) {
        int rc = trainer_capture(t, adaptive_now, presample_next, &g);
        if (rc) return rc;
      }
      CU(h, cudaGraphLaunch(g, t->st));
      h->launches += adaptive_now ? 2 + ADAPTIVE_LAUNCHES : 2;
    } else {
      // plain launches: the first step ever and the first adaptive step (one-time kernel attributes are set outside any
      // capture) and steps that start with the stand-alone sampler
      int rc = trainer_enqueue(t, sample_now, adaptive_now, presample_next, t->st);
      if (rc) return rc;
      t->warmed = true;
      if (adaptive_now) t->ad_warmed = true;
    }
    if (presample_next) t->next_ready = true;
    if (rs) t->have_batch = true;
    t->steps_issued++;
    // held-out validation after every step that brings the steps done since the run (re)started to a multiple of
    // val_every, at the parameters this step left; plain launches between the steps' launches or graph replays
    if (t->val_every > 0 && (t->steps_issued - t->step_base) % t->val_every == 0)
      if (int rc = validation_enqueue(t)) return rc;
  }
  return 0;
}

int pinn_trainer_run_lbfgs(pinn_trainer* t, const pinn_lbfgs_config* cfg, int resample, int use_graph) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  pinn_lbfgs_config c;
  {
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = lbfgs_resolve_config(h, cfg, &c)) return rc;
  }
  if (!resample && !t->have_batch)
    return fail(h, PINN_EINVAL, "pinn_trainer_run_lbfgs: no batch yet (resample = 0 needs pinn_trainer_set_batch or an earlier sampled step)");
  if (dp_active(h).world > 1)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_run_lbfgs: L-BFGS is not available with the data-parallel exchange");
  if (resample && t->pool_factor > 0)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_run_lbfgs: L-BFGS does not draw adaptive batches");
  if (!resample && t->pw_batch)
    return fail(h, PINN_ENOTSUP, "pinn_trainer_run_lbfgs: L-BFGS does not evaluate importance-weighted batches");
  DevGuard dev_guard(h->device);
  const int64_t slots = lbfgs_slots(c);
  if (!t->lb_state || t->lb_hist != c.history_size || t->lb_trace_rows < slots) {
    // (re)allocation happens here, outside any capture; a new history size is a fresh optimizer
    CU(h, cudaStreamSynchronize(t->st));
    for (cudaGraphExec_t& g : t->graph_lb)
      if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    if (!t->lb_state || t->lb_hist != c.history_size) {
      cudaFree(t->lb_state);
      t->lb_state = nullptr; t->lb_hist = 0;
      const size_t bytes = lbfgs_state_bytes(c.history_size);
      CU(h, cudaMalloc(&t->lb_state, bytes));
      CU(h, cudaMemsetAsync(t->lb_state, 0, bytes, t->st));  // ordered before the begin kernel on the same stream
      t->lb_hist = c.history_size;
    }
    if (t->lb_trace_rows < slots) {
      cudaFree(t->lb_trace);
      t->lb_trace = nullptr; t->lb_trace_rows = 0;
      CU(h, cudaMalloc(&t->lb_trace, (size_t)slots * 4 * 8));
      t->lb_trace_rows = slots;
    }
  }
  if (resample) {
    const SampleParams s = sampler_params(t, t->cur);
    CU(h, launch_sample(s, false, t->st));
    h->launches += 1;
    t->have_batch = true;
    t->pw_batch = false;
  }
  CU(h, cudaMemsetAsync(t->lb_trace, 0, (size_t)t->lb_trace_rows * 4 * 8, t->st));
  CU(h, launch_lbfgs_begin(t->lb_state, c, t->theta, t->theta32, t->st));
  h->launches += 1;
  int64_t k = 0;
  if (!t->lb_warmed) {  // one-time kernel attributes are set outside any capture
    if (int rc = lbfgs_eval_enqueue(t, nullptr, t->st)) return rc;
    t->lb_warmed = true;
    k = 1;
  }
  if (use_graph) {
    cudaGraphExec_t& g = t->graph_lb[t->cur];
    if (!g) {
      if (int rc = lbfgs_capture(t, &g)) return rc;
    }
    CU(h, cudaGraphLaunch(g, t->st));
    h->launches += 4;  // the condition kernel and one evaluation: how many evaluations run is decided on the device
  } else {
    for (; k < slots; k++)
      if (int rc = lbfgs_eval_enqueue(t, nullptr, t->st)) return rc;
  }
  return 0;
}

int pinn_trainer_read_lbfgs(pinn_trainer* t, double* status, double* trace, int64_t rows) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  if (status) {
    if (t->lb_state) CU(h, cudaMemcpy(status, t->lb_state, 8 * 8, cudaMemcpyDeviceToHost));
    else std::memset(status, 0, 8 * 8);
  }
  if (trace && rows > 0 && t->lb_trace) {
    const int64_t r = rows < t->lb_trace_rows ? rows : t->lb_trace_rows;
    CU(h, cudaMemcpy(trace, t->lb_trace, (size_t)r * 4 * 8, cudaMemcpyDeviceToHost));
  }
  return 0;
}

// Synchronise and read back.  Any pointer may be NULL.  scalars: {steps done, best loss, best step, batches drawn}.
int pinn_trainer_read(pinn_trainer* t, double* theta, double* m, double* v, double* best_theta, double* scalars, double* history,
                      int64_t history_rows) {
  if (!t) return PINN_EINVAL;
  pinn_handle* h = t->h;
  DevGuard dev_guard(h->device);
  CU(h, cudaStreamSynchronize(t->st));
  if (theta) CU(h, cudaMemcpy(theta, t->theta, NTHETA * 8, cudaMemcpyDeviceToHost));
  if (m) CU(h, cudaMemcpy(m, t->m, NTHETA * 8, cudaMemcpyDeviceToHost));
  if (v) CU(h, cudaMemcpy(v, t->v, NTHETA * 8, cudaMemcpyDeviceToHost));
  if (best_theta) CU(h, cudaMemcpy(best_theta, t->best_theta, NTHETA * 8, cudaMemcpyDeviceToHost));
  if (scalars) {
    unsigned long long s = 0, b = 0;
    long long bs = 0;
    double bl = 0.0;
    CU(h, cudaMemcpy(&s, t->step, 8, cudaMemcpyDeviceToHost));
    CU(h, cudaMemcpy(&b, t->batch, 8, cudaMemcpyDeviceToHost));
    CU(h, cudaMemcpy(&bs, t->best_step, 8, cudaMemcpyDeviceToHost));
    CU(h, cudaMemcpy(&bl, t->best_loss, 8, cudaMemcpyDeviceToHost));
    scalars[0] = (double)s; scalars[1] = bl; scalars[2] = (double)bs; scalars[3] = (double)b;
  }
  if (history && history_rows > 0) {
    const int64_t rows = history_rows < t->cfg.history_capacity ? history_rows : t->cfg.history_capacity;
    if (rows > 0) CU(h, cudaMemcpy(history, t->hist, (size_t)rows * 4 * 8, cudaMemcpyDeviceToHost));
  }
  if (dp_active(h).world > 1) {  // a data-parallel run whose exchange failed stopped updating: say so
    bool failed = false;
    if (int rc = dp_read_status(h, nullptr, &failed)) return rc;
    if (failed)
      return fail(h, PINN_ETIMEDOUT, "pinn_trainer_read: a data-parallel peer did not deliver its partial sums; the optimizer "
                                     "steps from the failed exchange on were skipped (values read are those before it)");
  }
  return 0;
}

// Device pointers of the current batch (x, y, z, R float32; mask bytes), e.g. to inspect what the sampler drew.
int pinn_trainer_batch(pinn_trainer* t, float** x, float** y, float** z, float** R, uint8_t** mask) {
  if (!t) return PINN_EINVAL;
  const int b = t->cur;  // the batch of the last enqueued step
  if (x) *x = t->x[b];
  if (y) *y = t->y[b];
  if (z) *z = t->z[b];
  if (R) *R = t->R[b];
  if (mask) *mask = t->mask[b];
  return 0;
}

void* pinn_trainer_stream(pinn_trainer* t) { return t ? (void*)t->st : nullptr; }

}  // extern "C"
