// C ABI of the PINN hot path (see include/pinn_b200.h for the contract).
#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "pinn_handle.h"
#include "pinn_train.h"

std::string g_create_err;

static const int kOffsets[17] = {O_W1, O_B1, O_W2, O_B2, O_WO, O_BO, O_WE1, O_BE1, O_WE2, O_BE2, O_WE, O_BE,
                                 O_WGL, O_BGL, O_WG, O_BG, NTHETA};

extern "C" {

int pinn_version(void) { return 100; }
int pinn_theta_size(void) { return NTHETA; }
void pinn_theta_offsets(int* out) { memcpy(out, kOffsets, sizeof(kOffsets)); }

// pinn_create: a failing CUDA call releases what was built so far; the message goes to the create-error slot
#define CREATE_CU(call)                                    \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) {                              \
      pinn_destroy(h);                                     \
      return fail(nullptr, (int)e__, "pinn_create: " #call); \
    }                                                      \
  } while (0)

int pinn_create(int device, pinn_handle** out) {
  if (!out) return fail(nullptr, PINN_EINVAL, "pinn_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess) return fail(nullptr, (int)e, "cudaGetDeviceCount");
  if (device < 0 || device >= ndev) return fail(nullptr, PINN_EINVAL, "pinn_create: no such CUDA device");
  cudaDeviceProp prop;
  CU(nullptr, cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(nullptr, PINN_ENOTSUP, "pinn_create: this library only carries sm_100a code (B200); no fallback exists");
  DevGuard dev_guard(device);
  pinn_handle* h = new pinn_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  CREATE_CU(cudaMalloc(&h->theta_dev, NTHETA * sizeof(float)));
  CREATE_CU(cudaHostAlloc(&h->out_pinned, NPART * sizeof(double), cudaHostAllocMapped));
  CREATE_CU(cudaHostGetDevicePointer(&h->out_mapped, h->out_pinned, 0));
  CREATE_CU(cudaMallocHost(&h->theta_pinned, NTHETA * sizeof(float)));
  CREATE_CU(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
  CREATE_CU(cudaStreamCreateWithFlags(&h->s_main, cudaStreamNonBlocking));
  for (int c = 0; c < 4; c++) CREATE_CU(cudaEventCreateWithFlags(&h->ev_chunk[c], cudaEventDisableTiming));
  // the workspace of the *_host entry's stream holds the rows of up to 4 chunk launches
  if (!ws_for(h, h->s_main, 4 * h->sm_count)) {
    const std::string msg = h->err;
    pinn_destroy(h);
    g_create_err = "pinn_create: " + msg;
    return PINN_EINVAL;
  }
  *out = h;
  return 0;
}

}  // extern "C"

static void ws_free(pinn_workspace& w) {
  cudaFree(w.partials); cudaFree(w.weights); cudaFree(w.counts); cudaFree(w.grid_partials); cudaFree(w.sph_partials);
  w = pinn_workspace();
}

// The owner of `st` is about to destroy it (a trainer): drain it and give the workspace back.
void ws_release(pinn_handle* h, cudaStream_t st) {
  for (pinn_workspace& c : h->ws)
    if (c.stream == st && c.partials) {
      cudaStreamSynchronize(st);
      ws_free(c);
    }
}

bool stream_is_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); return false; }
  return cap != cudaStreamCaptureStatusNone;
}

pinn_workspace* ws_for(pinn_handle* h, cudaStream_t st, int rows) {
  constexpr size_t MAX_WS = 32;
  pinn_workspace* w = nullptr;
  for (pinn_workspace& c : h->ws)
    if (c.stream == st && c.partials) { w = &c; break; }
  if (w && w->rows >= rows) {
    // a CUDA graph captured from this stream carries the workspace's addresses: from then on it is never recycled
    if (!w->in_graph && stream_is_capturing(st)) w->in_graph = true;
    w->last_use = ++h->ws_clock;
    return w;
  }
  // first call on this stream (or more rows than before): allocate.  Not possible while the stream is being captured
  // into a CUDA graph - the caller has to make one plain call first.
  if (stream_is_capturing(st)) {
    fail(h, PINN_EINVAL, "first call on a stream under CUDA-graph capture: call once on this stream outside the capture first");
    return nullptr;
  }
  if (!w) {
    for (pinn_workspace& c : h->ws)
      if (!c.partials) { w = &c; break; }  // a released slot
    if (!w && h->ws.size() >= MAX_WS) {  // streams come and go in the caller: recycle the least recently used workspace
      size_t lru = h->ws.size();
      for (size_t i = 0; i < h->ws.size(); i++)
        if (!h->ws[i].in_graph && h->ws[i].stream != h->s_main && (lru == h->ws.size() || h->ws[i].last_use < h->ws[lru].last_use)) lru = i;
      if (lru == h->ws.size()) {
        fail(h, PINN_EINVAL, "more than 32 streams with captured graphs or trainers on one handle");
        return nullptr;
      }
      cudaDeviceSynchronize();      // its last kernels may still be running
      ws_free(h->ws[lru]);
      w = &h->ws[lru];
    } else if (!w) {
      h->ws.emplace_back();
      w = &h->ws.back();
    }
  } else {
    if (w->in_graph) {
      fail(h, PINN_EINVAL, "this stream's workspace is referenced by a captured graph and cannot grow");
      return nullptr;
    }
    cudaStreamSynchronize(st);
    ws_free(*w);
  }
  w->stream = st;
  cudaError_t e = cudaMalloc(&w->partials, (size_t)rows * NPART * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&w->weights, 4 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&w->counts, 4 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemset(w->counts, 0, 4 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&w->grid_partials, (size_t)(h->sm_count + 1) * 8 * sizeof(double));
  if (e != cudaSuccess) {
    ws_free(*w);
    fail(h, (int)e, "workspace allocation (cudaMalloc)");
    return nullptr;
  }
  w->rows = rows;
  w->last_use = ++h->ws_clock;
  return w;
}

bool ws_sph_rows(pinn_handle* h, pinn_workspace* w, cudaStream_t st, int rows) {
  if (w->sph_rows >= rows) return true;
  if (stream_is_capturing(st)) {
    fail(h, PINN_EINVAL, "spheroidal sweep larger than any earlier one on a stream under CUDA-graph capture: make the largest "
                         "call once on this stream outside the capture first");
    return false;
  }
  if (w->in_graph) {
    fail(h, PINN_EINVAL, "this stream's workspace is referenced by a captured graph and cannot grow");
    return false;
  }
  cudaStreamSynchronize(st);  // the old rows may still be read by queued kernels
  cudaFree(w->sph_partials);
  w->sph_partials = nullptr;
  w->sph_rows = 0;
  cudaError_t e = cudaMalloc(&w->sph_partials, (size_t)rows * 8 * sizeof(double));
  if (e != cudaSuccess) {
    w->sph_partials = nullptr;
    fail(h, (int)e, "spheroidal workspace allocation (cudaMalloc)");
    return false;
  }
  w->sph_rows = rows;
  return true;
}

extern "C" {

int pinn_destroy(pinn_handle* h) {
  if (!h) return 0;
  DevGuard dev_guard(h->device);
  dp_release(h);
  cudaDeviceSynchronize();
  for (pinn_workspace& w : h->ws) ws_free(w);
  cudaFree(h->theta_dev); cudaFree(h->stage_dev);
  cudaFreeHost(h->out_pinned); cudaFreeHost(h->theta_pinned);
  if (h->s_copy) cudaStreamDestroy(h->s_copy);
  if (h->s_main) cudaStreamDestroy(h->s_main);
  for (int c = 0; c < 4; c++) if (h->ev_chunk[c]) cudaEventDestroy(h->ev_chunk[c]);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  delete h;
  return 0;
}

const char* pinn_last_error(pinn_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }
int64_t pinn_launch_count(pinn_handle* h) { return h ? h->launches : 0; }

int pinn_set_engine(pinn_handle* h, int engine) {
  if (!h) return PINN_EINVAL;
  if (engine == PINN_ENGINE_TCGEN05) return 0;
  std::lock_guard<std::mutex> lk(h->mu);
  if (engine == PINN_ENGINE_FFMA) return fail(h, PINN_ENOTSUP, "pinn_set_engine: this library carries the tcgen05 engine only");
  return fail(h, PINN_EINVAL, "pinn_set_engine: unknown engine");
}
int pinn_get_engine(pinn_handle* h) { return h ? PINN_ENGINE_TCGEN05 : PINN_EINVAL; }

int pinn_host_timing(pinn_handle* h, double* out4) {
  if (!h || !out4) return PINN_EINVAL;
  memcpy(out4, h->host_us, sizeof(h->host_us));
  return 0;
}

int pinn_profile_begin(pinn_handle* h) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  h->profiling = true;
  h->ev_used = 0;
  return 0;
}

int pinn_profile_collect(pinn_handle* h, double* total_ms, int* launches) {
  if (!h || !total_ms || !launches) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  DevGuard dev_guard(h->device);
  double tot = 0.0;
  for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
    CU(h, cudaEventSynchronize(h->ev_pool[i + 1]));
    float ms = 0.0f;
    CU(h, cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]));
    tot += ms;
  }
  *total_ms = tot;
  *launches = (int)(h->ev_used / 2);
  h->profiling = false;
  h->ev_used = 0;
  return 0;
}

// Device-visible alias of a page-locked host pointer, or false when the memory is pageable / not host memory.
static bool map_pinned(const void* p, const void** dev) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  if (a.type != cudaMemoryTypeHost || !a.devicePointer) return false;
  *dev = a.devicePointer;
  return true;
}

// Enqueue the fused step kernel for points [first, first + cnt) of a batch; its per-CTA rows go to partial rows
// [row0, row0 + *rows).  The handle mutex is held by the caller.
static int enqueue_step_chunk(pinn_handle* h, pinn_workspace* ws, int nev, StepParams p, int64_t first, int64_t cnt, int row0,
                              int* rows, cudaStream_t st) {
  const size_t es = p.in_f64 ? 8 : 4;
  p.x = (const char*)p.x + first * es; p.y = (const char*)p.y + first * es;
  p.z = (const char*)p.z + first * es; p.R = (const char*)p.R + first * es;
  if (p.mask) p.mask += first;
  if (p.point_w) p.point_w += first;
  if (p.E_out) p.E_out += first;
  p.n = cnt;
  p.partials = ws->partials + (size_t)row0 * NPART;
  const int grid = train_grid_for(h, cnt);
  if (row0 + grid > ws->rows) return fail(h, PINN_EINVAL, "internal: partial-row workspace exceeded");
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (h->profiling) {
    while (h->ev_pool.size() < h->ev_used + 2) {
      cudaEvent_t e;
      CU(h, cudaEventCreate(&e));
      h->ev_pool.push_back(e);
    }
    e0 = h->ev_pool[h->ev_used++];
    e1 = h->ev_pool[h->ev_used++];
    CU(h, cudaEventRecord(e0, st));
  }
  CU(h, launch_step_tc(nev, true, p, grid, st));
  if (e1) CU(h, cudaEventRecord(e1, st));
  h->launches++;
  *rows = grid;
  return 0;
}

}  // extern "C"

// The training evaluation on device buffers (or mapped page-locked columns): the set-count kernels when no loss weights
// are given, one step launch per chunk of the plan, one reduction over the partial rows of all chunks.
int loss_fwd_bwd_impl(pinn_handle* h, const LossCall& c, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(h->mu);
  StepParams p{};
  int nev = 0;
  if (variant_coef(c.variant, &p.vc, &nev)) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd: unknown variant");
  if (c.n <= 0) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd: n must be positive");
  if (!c.x || !c.y || !c.z || !c.R || (!c.theta && !c.theta_inline && !c.theta_tensors) || !c.sums || !c.dtheta)
    return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd: NULL pointer argument");
  if (c.in_dtype != PINN_F32 && c.in_dtype != PINN_F64) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd: bad in_dtype");
  if (c.point_w && (c.theta_inline || c.nchunk))
    return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_weighted: per-point weights need device-resident inputs");
  const int nchunk = c.nchunk ? c.nchunk : 1;
  int need_rows = 0;  // one partial row per CTA of every chunk launch
  for (int k = 0; k < nchunk; k++) need_rows += train_grid_for(h, c.nchunk ? c.chunk[k].count : c.n);
  DevGuard dev_guard(h->device);
  pinn_workspace* ws = ws_for(h, st, need_rows);
  if (!ws) return PINN_EINVAL;
  if (int rc = dp_serialize(h, st)) return rc;
  p.x = c.x; p.y = c.y; p.z = c.z; p.R = c.R; p.mask = c.mask; p.n = c.n; p.in_f64 = c.in_dtype == PINN_F64;
  p.point_w = c.point_w;
  p.bcut = c.bcutoff; p.E_out = static_cast<float*>(c.E_out); p.E_f64 = c.E_f64;
  p.base_grads = (c.grad_mask & 0x003Fu) != 0;
  p.gate_grads = (c.grad_mask & 0xF000u) != 0;
  const double* weights = c.weights;
  if (c.theta_inline) {
    p.theta_inline = c.theta_inline;
  } else if (c.theta_tensors) {
    for (int k = 0; k < 16; k++) {
      if (!c.theta_tensors[k]) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_tensors: NULL parameter tensor");
      p.theta_tensors[k] = c.theta_tensors[k];
    }
    p.theta_from_tensors = 1; p.tensors_f64 = c.tensors_f64; p.tensors_in_out = c.tensors_in_out;
  } else {
    p.theta = c.theta;
  }
  if (c.weights_inline) {
    p.weights_inline = c.weights_inline;
  } else if (!weights) {
    CU(h, launch_count(p, ws->counts, ws->weights, st));
    h->launches += 2;
    weights = ws->weights;
  }
  p.weights = weights;
  int rows = 0;
  for (int k = 0; k < nchunk; k++) {
    const LossCall::Chunk ck = c.nchunk ? c.chunk[k] : LossCall::Chunk{0, c.n, nullptr};
    if (ck.ready) CU(h, cudaStreamWaitEvent(st, ck.ready, 0));
    int r = 0;
    if (int rc = enqueue_step_chunk(h, ws, nev, p, ck.first, ck.count, rows, &r, st)) return rc;
    rows += r;
  }
  CU(h, launch_reduce(ws->partials, rows, weights, c.weights_inline, c.grad_mask, c.dtheta, c.sums, p.E_out, c.n,
                      dp_active(h), st, c.adam, c.adam_ticket, c.presample, c.E_f64, c.dtheta_in_out));
  h->launches++;
  return 0;
}

extern "C" {

int pinn_loss_fwd_bwd(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z,
                      const void* R, int in_dtype, const uint8_t* mask, const float* theta, const double* weights,
                      uint32_t grad_mask, float bcutoff, double* sums, double* dtheta, float* E_out, void* stream) {
  if (!h) return PINN_EINVAL;
  if (!theta) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd: NULL pointer argument");
  LossCall c;
  c.variant = variant; c.n = n; c.x = x; c.y = y; c.z = z; c.R = R; c.in_dtype = in_dtype; c.mask = mask;
  c.theta = theta; c.weights = weights; c.grad_mask = grad_mask; c.bcutoff = bcutoff; c.sums = sums; c.dtheta = dtheta;
  c.E_out = E_out;
  return loss_fwd_bwd_impl(h, c, (cudaStream_t)stream);
}

int pinn_loss_fwd_bwd_weighted(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z,
                               const void* R, int in_dtype, const uint8_t* mask, const float* theta, const double* weights,
                               const float* point_w, uint32_t grad_mask, float bcutoff, double* sums, double* dtheta,
                               float* E_out, void* stream) {
  if (!h) return PINN_EINVAL;
  if (!theta || !point_w) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_weighted: NULL pointer argument");
  LossCall c;
  c.variant = variant; c.n = n; c.x = x; c.y = y; c.z = z; c.R = R; c.in_dtype = in_dtype; c.mask = mask;
  c.theta = theta; c.weights = weights; c.point_w = point_w; c.grad_mask = grad_mask; c.bcutoff = bcutoff; c.sums = sums;
  c.dtheta = dtheta; c.E_out = E_out;
  return loss_fwd_bwd_impl(h, c, (cudaStream_t)stream);
}

int pinn_loss_fwd_bwd_tensors(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z,
                              const void* R, int in_dtype, const uint8_t* mask, const void* const* params, int param_dtype,
                              int param_layout, const double* weights_host, uint32_t grad_mask, float bcutoff, double* sums,
                              double* dtheta, void* E_out, int E_dtype, void* stream) {
  if (!h) return PINN_EINVAL;
  if (!params) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_tensors: NULL pointer argument");
  if ((param_dtype != PINN_F32 && param_dtype != PINN_F64) || (E_dtype != PINN_F32 && E_dtype != PINN_F64) ||
      (param_layout != PINN_VARIANT_POC && param_layout != PINN_VARIANT_TRAINPY))
    return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_tensors: bad dtype / layout code");
  // canonical order of the 16 tensors; train.py keeps the gate (L1a..L2b) in front of the E-net (train.py:108-109)
  static const int kTrainpyToCanonical[16] = {0, 1, 2, 3, 4, 5, 12, 13, 14, 15, 6, 7, 8, 9, 10, 11};
  const void* canon[16];
  for (int k = 0; k < 16; k++) canon[param_layout == PINN_VARIANT_TRAINPY ? kTrainpyToCanonical[k] : k] = params[k];
  LossCall c;
  c.variant = variant; c.n = n; c.x = x; c.y = y; c.z = z; c.R = R; c.in_dtype = in_dtype; c.mask = mask;
  c.theta_tensors = canon; c.tensors_f64 = param_dtype == PINN_F64; c.tensors_in_out = param_layout == PINN_VARIANT_TRAINPY;
  c.weights_inline = weights_host; c.grad_mask = grad_mask; c.bcutoff = bcutoff; c.sums = sums; c.dtheta = dtheta;
  c.E_out = E_out; c.E_f64 = E_dtype == PINN_F64; c.dtheta_in_out = c.tensors_in_out;
  return loss_fwd_bwd_impl(h, c, (cudaStream_t)stream);
}

int pinn_mask_from_index_sets(pinn_handle* h, int64_t n, const int64_t* idx1, int64_t n1, const int64_t* idx2, int64_t n2,
                              uint8_t* mask, void* stream) {
  if (!h) return PINN_EINVAL;
  if (n <= 0 || n1 < 0 || n2 < 0 || !mask || (n1 > 0 && !idx1) || (n2 > 0 && !idx2) || ((uintptr_t)mask & 3u))
    return fail(h, PINN_EINVAL, "pinn_mask_from_index_sets: bad argument (mask must be 4-byte aligned with room for n rounded up to 4)");
  DevGuard dev_guard(h->device);
  CU(h, launch_mask_from_index_sets(reinterpret_cast<const long long*>(idx1), n1, reinterpret_cast<const long long*>(idx2), n2,
                                    mask, n, (cudaStream_t)stream));
  std::lock_guard<std::mutex> lk(h->mu);
  h->launches += 1;
  return 0;
}

int pinn_fields(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z, const void* R,
                int in_dtype, const float* theta, float* psi, float* lap, float* hpsi, float* res, float* E,
                void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  StepParams p{};
  int nev = 0;
  if (variant_coef(variant, &p.vc, &nev)) return fail(h, PINN_EINVAL, "pinn_fields: unknown variant");
  if (n <= 0) return fail(h, PINN_EINVAL, "pinn_fields: n must be positive");
  if (!x || !y || !z || !R || !theta) return fail(h, PINN_EINVAL, "pinn_fields: NULL pointer argument");
  if (in_dtype != PINN_F32 && in_dtype != PINN_F64) return fail(h, PINN_EINVAL, "pinn_fields: bad in_dtype");
  DevGuard dev_guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  p.x = x; p.y = y; p.z = z; p.R = R; p.n = n; p.in_f64 = in_dtype == PINN_F64;
  p.psi = psi; p.lap = lap; p.hpsi = hpsi; p.res = res; p.E_out = E; p.theta = theta;
  CU(h, launch_step_tc(nev, false, p, grid_for(h, n), st));
  h->launches++;
  return 0;
}

int pinn_loss_eval(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z, const void* R,
                   int in_dtype, const uint8_t* mask, const float* theta, const double* weights, float bcutoff, double* sums,
                   void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  StepParams p{};
  int nev = 0;
  if (variant_coef(variant, &p.vc, &nev)) return fail(h, PINN_EINVAL, "pinn_loss_eval: unknown variant");
  if (n <= 0) return fail(h, PINN_EINVAL, "pinn_loss_eval: n must be positive");
  if (!x || !y || !z || !R || !theta || !sums) return fail(h, PINN_EINVAL, "pinn_loss_eval: NULL pointer argument");
  if (in_dtype != PINN_F32 && in_dtype != PINN_F64) return fail(h, PINN_EINVAL, "pinn_loss_eval: bad in_dtype");
  DevGuard dev_guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  pinn_workspace* ws = ws_for(h, st, h->sm_count);
  if (!ws) return PINN_EINVAL;
  p.x = x; p.y = y; p.z = z; p.R = R; p.mask = mask; p.n = n; p.in_f64 = in_dtype == PINN_F64; p.bcut = bcutoff;
  p.theta = theta;
  p.grid.partials = ws->grid_partials;  // the LOSS instance's per-CTA rows (p.grid.on stays 0)
  const int grid = grid_for(h, n);
  CU(h, launch_loss_tc(nev, p, grid, st));
  CU(h, launch_loss_finish(ws->grid_partials, grid, n, weights, sums, nullptr, st));
  h->launches += 2;
  return 0;
}

int pinn_loss_fwd_bwd_host(pinn_handle* h, int variant, int64_t n, const void* x, const void* y, const void* z,
                           const void* R, int in_dtype, const uint8_t* mask, const double* theta_host,
                           const double* weights_host, uint32_t grad_mask, float bcutoff, double* sums_host,
                           double* dtheta_host, float* E_out_host) {
  if (!h) return PINN_EINVAL;
  if (n <= 0) return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_host: n must be positive");
  if (!x || !y || !z || !R || !theta_host || !sums_host || !dtheta_host)
    return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_host: NULL pointer argument");
  if (in_dtype != PINN_F32 && in_dtype != PINN_F64)
    return fail(h, PINN_EINVAL, "pinn_loss_fwd_bwd_host: bad in_dtype");
  std::lock_guard<std::mutex> host_lock(h->host_mu);
  const auto t_enter = std::chrono::steady_clock::now();
  DevGuard dev_guard(h->device);
  const size_t es = in_dtype == PINN_F64 ? 8 : 4;
  // Page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) inputs are read by the kernel in place: the
  // step kernel requests the coordinates of its next super-tile one tile ahead, which hides the PCIe latency, and
  // the 16 B/point crossing the bus overlap the whole kernel instead of preceding it.  Pageable inputs are staged.
  const void* mapped[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  const bool zero_copy = map_pinned(x, &mapped[0]) && map_pinned(y, &mapped[1]) &&
                         map_pinned(z, &mapped[2]) && map_pinned(R, &mapped[3]) && (!mask || map_pinned(mask, &mapped[4]));
  const size_t col = zero_copy ? 0 : ((size_t)n * es + 255) & ~(size_t)255;
  const size_t mcol = zero_copy ? 0 : ((size_t)n + 255) & ~(size_t)255;
  const size_t ecol = ((size_t)n * 4 + 255) & ~(size_t)255;
  const size_t need = 4 * col + mcol + ecol;
  {
    std::lock_guard<std::mutex> lk(h->mu);
    if (need > h->stage_bytes) {  // grows geometrically; steady-state steps do not allocate
      CU(h, cudaStreamSynchronize(h->s_main));
      if (h->stage_dev) CU(h, cudaFree(h->stage_dev));
      h->stage_dev = nullptr;
      const size_t cap = need + need / 4;
      CU(h, cudaMalloc(&h->stage_dev, cap));
      h->stage_bytes = cap;
    }
  }
  char* base = (char*)h->stage_dev;
  cudaStream_t st = h->s_main;
  for (int i = 0; i < NTHETA; i++) h->theta_pinned[i] = (float)theta_host[i];
  float* edev = (float*)(base + 4 * col + mcol);
  LossCall c;
  c.variant = variant; c.n = n; c.in_dtype = in_dtype; c.grad_mask = grad_mask; c.bcutoff = bcutoff; c.E_out = edev;
  // the 8 sums and 1521 gradients are written by the reduction kernel straight into mapped page-locked memory
  c.sums = h->out_mapped; c.dtheta = h->out_mapped + 8;
  // With known weights theta and the weights ride in the kernel parameters and nothing is uploaded first.  Without them
  // theta is uploaded, and the set sizes are counted on the device.
  if (weights_host) {
    c.theta_inline = h->theta_pinned;
    c.weights_inline = weights_host;
  } else {
    CU(h, cudaMemcpyAsync(h->theta_dev, h->theta_pinned, NTHETA * sizeof(float), cudaMemcpyHostToDevice, st));
    c.theta = h->theta_dev;
  }
  if (zero_copy) {
    c.x = mapped[0]; c.y = mapped[1]; c.z = mapped[2]; c.R = mapped[3]; c.mask = (const uint8_t*)mapped[4];
  } else {
    uint8_t* mdev = mask ? (uint8_t*)(base + 4 * col) : nullptr;
    c.x = base; c.y = base + col; c.z = base + 2 * col; c.R = base + 3 * col; c.mask = mdev;
    // With the weights known up front the batch is processed in 4 chunks so that the copy of chunk k+1 (copy stream)
    // overlaps the kernel of chunk k.  Chunks are whole rounds of super-tiles (sm_count x 128 points) so that no launch
    // ends on a partial wave; the first chunk is short (2 rounds) to start computing early.
    // Without weights the set sizes must be counted over the whole batch first: one chunk, copied on the main stream.
    const int64_t unit = (int64_t)h->sm_count * 128;
    const int64_t rounds = (n + unit - 1) / unit;
    c.nchunk = 1;
    c.chunk[0] = {0, n, nullptr};
    if (weights_host && rounds >= 8) {
      c.nchunk = 4;
      const int64_t rest = rounds - 2;
      const int64_t r[4] = {2, rest / 3, rest / 3, rest - 2 * (rest / 3)};
      int64_t at = 0;
      for (int k = 0; k < 4; k++) {
        c.chunk[k] = {at, k == 3 ? n - at : r[k] * unit, h->ev_chunk[k]};
        at += c.chunk[k].count;
      }
    }
    const void* src[4] = {x, y, z, R};
    for (int k = 0; k < c.nchunk; k++) {
      const LossCall::Chunk& ck = c.chunk[k];
      cudaStream_t sc = ck.ready ? h->s_copy : st;
      for (int j = 0; j < 4; j++)
        CU(h, cudaMemcpyAsync(base + j * col + ck.first * es, (const char*)src[j] + ck.first * es, (size_t)ck.count * es,
                              cudaMemcpyHostToDevice, sc));
      if (mask) CU(h, cudaMemcpyAsync(mdev + ck.first, mask + ck.first, (size_t)ck.count, cudaMemcpyHostToDevice, sc));
      if (ck.ready) CU(h, cudaEventRecord(ck.ready, sc));
    }
  }
  if (int rc = loss_fwd_bwd_impl(h, c, st)) return rc;
  if (E_out_host) CU(h, cudaMemcpyAsync(E_out_host, edev, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  const auto t_submitted = std::chrono::steady_clock::now();
  CU(h, cudaStreamSynchronize(st));
  const auto t_done = std::chrono::steady_clock::now();
  memcpy(sums_host, h->out_pinned, 8 * sizeof(double));
  memcpy(dtheta_host, h->out_pinned + 8, NTHETA * sizeof(double));
  const auto t_exit = std::chrono::steady_clock::now();
  auto us = [](auto a, auto b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
  h->host_us[0] = us(t_enter, t_submitted); h->host_us[1] = us(t_submitted, t_done); h->host_us[2] = us(t_done, t_exit);
  h->host_us[3] = us(t_enter, t_exit);
  return 0;
}

}  // extern "C"
