// C ABI of the rows next to the hot path (include/pinn_b200.h, "training loop" and "analysis" sections):
// sampler, fused Adam, the device-resident trainer (CUDA-graph replay of sample -> loss -> Adam), the E(R)/gate
// curve and the dense-grid quadrature sums.
#include <algorithm>
#include <cstdlib>
#include <cstring>

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
};

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
static int trainer_enqueue(pinn_trainer* t, bool sample_now, bool presample_next, cudaStream_t st) {
  pinn_handle* h = t->h;
  const pinn_train_config& c = t->cfg;
  const int b = t->cur;
  if (sample_now) {
    const SampleParams s = sampler_params(t, b);
    CU(h, launch_sample(s, false, st));
    h->launches += 1;
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
  int rc = loss_fwd_bwd_impl(h, lc, st);
  if (rc) return rc;
  return 0;
}

static int trainer_capture(pinn_trainer* t, bool presample_next, cudaGraphExec_t* out) {
  pinn_handle* h = t->h;
  cudaGraph_t g = nullptr;
  CU(h, cudaStreamBeginCapture(t->st, cudaStreamCaptureModeThreadLocal));
  const int64_t launches_before = h->launches;
  int rc = trainer_enqueue(t, false, presample_next, t->st);
  h->launches = launches_before;  // capture does not launch; replays are counted in pinn_trainer_run
  cudaError_t e = cudaStreamEndCapture(t->st, &g);
  if (rc) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) return fail(h, (int)e, "cudaStreamEndCapture");
  e = cudaGraphInstantiate(out, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return fail(h, (int)e, "cudaGraphInstantiate");
  return 0;
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
    for (int b = 0; b < 2; b++)
      if (t->graph[a][b]) cudaGraphExecDestroy(t->graph[a][b]);
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
    for (int b = 0; b < 2; b++)
      if (t->graph[a][b]) { cudaGraphExecDestroy(t->graph[a][b]); t->graph[a][b] = nullptr; }
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
  auto resamples = [&](int64_t tt) { return resample && (tt % t->cfg.sc_sampling == 0) && (tt < t->cfg.freeze_after); };
  for (int64_t k = 0; k < steps; k++) {
    const int64_t tt = t->steps_issued;
    const bool rs = resamples(tt);
    bool sample_now = false;
    if (rs) {
      if (t->next_ready) { t->cur ^= 1; t->next_ready = false; }  // drawn while the previous step was reduced
      else sample_now = true;
    }
    const bool presample_next = (k + 1 < steps) && resamples(tt + 1);
    if (use_graph && t->warmed && !sample_now) {
      cudaGraphExec_t& g = t->graph[t->cur][presample_next ? 1 : 0];
      if (!g) {
        int rc = trainer_capture(t, presample_next, &g);
        if (rc) return rc;
      }
      CU(h, cudaGraphLaunch(g, t->st));
      h->launches += 2;
    } else {
      // plain launches: the first step ever (one-time kernel attributes are set outside any capture) and steps that
      // start with the stand-alone sampler
      int rc = trainer_enqueue(t, sample_now, presample_next, t->st);
      if (rc) return rc;
      t->warmed = true;
    }
    if (presample_next) t->next_ready = true;
    if (rs) t->have_batch = true;
    t->steps_issued++;
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
