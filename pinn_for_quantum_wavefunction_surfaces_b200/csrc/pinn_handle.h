// Private to the library: the handle behind the C ABI (include/pinn_b200.h) and the error helpers.
#pragma once
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/pinn_b200.h"
#include "pinn_common.cuh"
#include "pinn_dp.cuh"
#include "pinn_launch.h"

using namespace pinn;

// The handle's data-parallel exchange (pinn_dp.cu)
struct DpState {
  unsigned char* buf = nullptr;  // own exchange buffer
  DpArgs args;                   // rank, world, every rank's buffer as mapped on this device, time-out
  bool on = false;               // calls exchange
  cudaStream_t stream = nullptr;  // the exchange buffers carry ONE sequence of steps: the stream of the last exchanging call
  bool stream_set = false;
  bool opened[DP_MAX_WORLD] = {false, false, false, false, false, false, false, false};  // args.peer[r] came from cudaIpcOpenMemHandle
};

// Scratch memory of the calls ENQUEUED ON ONE STREAM.  Kernels of one stream run in order, so they may share it; calls
// that arrive on different streams (torch's current stream, the *_host entry's private stream, every trainer's own
// stream) may overlap on the device and therefore get one workspace each (ws_for, pinn_capi.cu).
struct pinn_workspace {
  cudaStream_t stream = nullptr;
  double* partials = nullptr;       // [rows][NPART] per-CTA rows of the step kernel
  int rows = 0;
  double* weights = nullptr;        // 4 doubles: the output of the set-count kernels when the caller passes no loss weights
  unsigned long long* counts = nullptr;  // [0..1] boundary-set sizes, [2] batch index of pinn_sample, [3] its block ticket
  double* grid_partials = nullptr;  // [sm_count + 1][8] dense-grid quadrature rows
  double* sph_partials = nullptr;   // [sph_rows][8] rows of the spheroidal sweep (ws_sph_rows: grows, never shrinks)
  int sph_rows = 0;
  uint64_t last_use = 0;
  bool in_graph = false;            // a call on this stream was captured into a CUDA graph: the addresses above must stay valid
};

struct pinn_handle {
  int device = 0;
  int sm_count = 0;
  std::vector<pinn_workspace> ws;  // one per stream that has called in (guarded by mu)
  uint64_t ws_clock = 0;
  // *_host entry
  float* theta_pinned = nullptr;   // theta as float: kernel parameters, or the source of the upload below
  float* theta_dev = nullptr;      // theta uploaded for calls without loss weights
  void* stage_dev = nullptr;       // coordinates + mask
  size_t stage_bytes = 0;
  double* out_pinned = nullptr;    // mapped page-locked: the reduction kernel of the *_host entry writes it directly
  double* out_mapped = nullptr;    // its device alias
  cudaStream_t s_copy = nullptr, s_main = nullptr;
  cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr};  // *_host entry: copy of chunk c complete
  DpState dp;
  double host_us[4] = {0, 0, 0, 0};   // last pinn_loss_fwd_bwd_host call: submit, wait, copy-out, total (microseconds)
  int64_t launches = 0;
  bool profiling = false;          // pinn_profile_begin/collect: CUDA events around the fused step kernel
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  std::string err;
  std::mutex mu;
  std::mutex host_mu;  // pinn_loss_fwd_bwd_host calls on one handle share its staging / mapped buffers: one at a time
};

// Every entry point works on the handle's device and leaves the caller's current device as it found it.
struct DevGuard {
  int prev = -1, dev;
  explicit DevGuard(int d) : dev(d) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DevGuard() {
    if (prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
  DevGuard(const DevGuard&) = delete;
  DevGuard& operator=(const DevGuard&) = delete;
};

// The training evaluation behind pinn_loss_fwd_bwd[_tensors] / pinn_loss_fwd_bwd_host / the trainer (pinn_capi.cu).
namespace pinn { struct AdamParams; struct SampleParams; }
struct LossCall {
  int variant = 0;
  int64_t n = 0;
  const void *x = nullptr, *y = nullptr, *z = nullptr, *R = nullptr;  // device (or mapped page-locked host) columns
  int in_dtype = PINN_F32;
  const uint8_t* mask = nullptr;
  const float* point_w = nullptr;  // device float32 [n] per-point loss weights (pinn_loss_fwd_bwd_weighted), or NULL
  // theta: exactly one of - packed float32 device vector; HOST float32[1521] that travels inside the kernel parameters;
  // the caller's 16 tensors (device pointers in canonical order, float32/float64, (out,in) or train.py (in,out) layout)
  const float* theta = nullptr;
  const float* theta_inline = nullptr;
  const void* const* theta_tensors = nullptr;
  int tensors_f64 = 0, tensors_in_out = 0;
  // loss weights: device pointer, or HOST double[3] carried by value, or neither (sets counted on the device first)
  const double* weights = nullptr;
  const double* weights_inline = nullptr;
  uint32_t grad_mask = 0xFFFFu;
  float bcutoff = 17.5f;
  double *sums = nullptr, *dtheta = nullptr;
  void* E_out = nullptr;
  int E_f64 = 0;          // E_out is float64
  int dtheta_in_out = 0;  // 2-D tensors of dtheta in train.py's (in,out) layout
  const pinn::AdamParams* adam = nullptr;       // optimizer step fused behind the reduction (the trainer)
  unsigned long long* adam_ticket = nullptr;
  const pinn::SampleParams* presample = nullptr;  // the trainer's next batch drawn by extra blocks of the reduction kernel
  // Chunk plan: the batch as up to 4 step launches over points [first, first + count), each enqueued after the stream has
  // waited for its event (NULL: no wait; the *_host entry records there that the chunk's copy is complete).  The partial
  // rows of all chunks go to ONE reduction.  nchunk = 0: one launch over the whole batch.
  struct Chunk {
    int64_t first, count;
    cudaEvent_t ready;
  };
  int nchunk = 0;
  Chunk chunk[4] = {};
};
int loss_fwd_bwd_impl(pinn_handle* h, const LossCall& c, cudaStream_t st);
// pinn_lbfgs.cu: torch's defaults for an unset max_eval, then the checks every L-BFGS entry makes (PINN_EINVAL + message)
int lbfgs_resolve_config(pinn_handle* h, const pinn_lbfgs_config* in, pinn_lbfgs_config* out);

// VariantCoef and number of MLP evaluations (1 or 2) of a PINN_VARIANT_*; PINN_EINVAL for an unknown variant
inline int variant_coef(int variant, VariantCoef* vc, int* nev) {
  if (variant == PINN_VARIANT_POC) { *vc = {1.0f, -0.5f, -1.0f, -1.0f}; *nev = 2; return 0; }
  if (variant == PINN_VARIANT_TRAINPY) { *vc = {2.0f, 1.0f, 1.0f, 1.0f}; *nev = 1; return 0; }
  return PINN_EINVAL;
}
// Grid of a step-kernel launch over n points: one persistent CTA per SM, a CTA works on super-tiles of 128 points
inline int grid_for(const pinn_handle* h, long long n) {
  const long long want = (n + 127) / 128;
  return (int)(want < h->sm_count ? (want < 1 ? 1 : want) : h->sm_count);
}
// Grid of a TRAINING launch: the step kernel keeps its gradient and loss sums in float32 registers over every super-tile
// a CTA works on, and their error grows with that count (DESIGN.md section 4).  Past TRAIN_TILES_MAX super-tiles per CTA
// the launch gets sm_count * ceil(T / TRAIN_TILES_MAX) CTAs instead (T = super-tiles per CTA at one CTA per SM); the
// CTAs beyond one per SM run as later waves, each into its own partial row.  Up to 148 x 256 x 128 = 4.8e6 points a
// launch keeps one CTA per SM.
constexpr long long TRAIN_TILES_MAX = 256;
inline int train_grid_for(const pinn_handle* h, long long n) {
  const long long per_cta = ((n + 127) / 128 + h->sm_count - 1) / h->sm_count;
  if (per_cta <= TRAIN_TILES_MAX) return grid_for(h, n);
  return (int)((long long)h->sm_count * ((per_cta + TRAIN_TILES_MAX - 1) / TRAIN_TILES_MAX));
}

// The workspace of stream `st` with room for at least `rows` partial rows (created / grown on first use; the handle mutex
// is held by the caller).  NULL + error message on failure.
pinn_workspace* ws_for(pinn_handle* h, cudaStream_t st, int rows);
// Room for `rows` rows of the spheroidal sweep in w (the workspace of st): allocated only when a call needs more rows than
// any earlier call on the stream, which is refused under CUDA-graph capture.  false + error message on failure.
bool ws_sph_rows(pinn_handle* h, pinn_workspace* w, cudaStream_t st, int rows);
void ws_release(pinn_handle* h, cudaStream_t st);
bool stream_is_capturing(cudaStream_t st);

// pinn_dp.cu.  dp_active: the exchange arguments of a call (world <= 1 unless the exchange is on with world > 1).
// dp_serialize: before a call that may exchange is enqueued on `st`, mutex held.  dp_read_status: this rank's control
// block, read synchronously (the exchange must be initialised).
DpArgs dp_active(const pinn_handle* h);
int dp_serialize(pinn_handle* h, cudaStream_t st);
int dp_read_status(pinn_handle* h, int64_t* exchanges, bool* failed);
void dp_release(pinn_handle* h);

extern std::string g_create_err;

inline int fail(pinn_handle* h, int code, const char* what) {
  char buf[512];
  if (code > 0)
    snprintf(buf, sizeof(buf), "%s: %s (%s)", what, cudaGetErrorString((cudaError_t)code),
             cudaGetErrorName((cudaError_t)code));
  else
    snprintf(buf, sizeof(buf), "%s", what);
  if (h) h->err = buf; else g_create_err = buf;
  return code;
}
#define CU(h, call)                                   \
  do {                                                \
    cudaError_t e__ = (call);                         \
    if (e__ != cudaSuccess) return fail(h, (int)e__, #call); \
  } while (0)

