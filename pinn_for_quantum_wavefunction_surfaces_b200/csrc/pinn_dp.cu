// Host side of the data-parallel exchange (pinn_dp.cuh; include/pinn_b200.h: pinn_dp_*): the exchange buffers, how the
// peers map them, and which calls exchange.
#include <cstring>

#include "pinn_handle.h"

DpArgs dp_active(const pinn_handle* h) { return h->dp.on && h->dp.args.world > 1 ? h->dp.args : DpArgs(); }

// With the data-parallel exchange enabled the handle's exchange buffers carry one sequence of steps: calls must reach the
// device in one order on all ranks.  A call on another stream than the previous exchanging call first waits (on the
// host) for that stream to drain.
int dp_serialize(pinn_handle* h, cudaStream_t st) {
  if (dp_active(h).world <= 1) return 0;
  if (h->dp.stream_set && h->dp.stream != st) {
    if (stream_is_capturing(st))
      return fail(h, PINN_EINVAL, "data-parallel exchange: the previous exchanging call used another stream; cannot switch streams under capture");
    CU(h, cudaStreamSynchronize(h->dp.stream));
  }
  h->dp.stream = st;
  h->dp.stream_set = true;
  return 0;
}

int dp_read_status(pinn_handle* h, int64_t* exchanges, bool* failed) {
  unsigned long long ctl[DP_CTL_SLOTS];
  CU(h, cudaMemcpy(ctl, dp_ctl(h->dp.buf), sizeof(ctl), cudaMemcpyDeviceToHost));
  if (exchanges) *exchanges = (int64_t)ctl[DP_EXCHANGES];
  *failed = ctl[DP_FAILED] != 0ull;
  return 0;
}

void dp_release(pinn_handle* h) {
  for (int r = 0; r < DP_MAX_WORLD; r++)
    if (h->dp.opened[r] && h->dp.args.peer[r]) cudaIpcCloseMemHandle(h->dp.args.peer[r]);
  if (h->dp.buf) cudaFree(h->dp.buf);
  h->dp = DpState();
}

extern "C" {

int pinn_dp_init(pinn_handle* h, int rank, int world, void* ipc_handle_out) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (world < 1 || world > DP_MAX_WORLD || rank < 0 || rank >= world)
    return fail(h, PINN_EINVAL, "pinn_dp_init: need 0 <= rank < world <= 8");
  DevGuard dev_guard(h->device);
  dp_release(h);
  CU(h, cudaMalloc(&h->dp.buf, DP_BUFFER_BYTES));
  CU(h, cudaMemset(h->dp.buf, 0, DP_BUFFER_BYTES));
  CU(h, cudaDeviceSynchronize());
  h->dp.args.rank = rank;
  h->dp.args.world = world;
  h->dp.args.peer[rank] = h->dp.buf;
  if (ipc_handle_out) {
    static_assert(sizeof(cudaIpcMemHandle_t) == PINN_DP_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t ih;
    CU(h, cudaIpcGetMemHandle(&ih, h->dp.buf));
    memcpy(ipc_handle_out, &ih, sizeof(ih));
  }
  return 0;
}

int pinn_dp_connect(pinn_handle* h, const void* all_handles) {
  if (!h || !all_handles) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->dp.buf) return fail(h, PINN_EINVAL, "pinn_dp_connect: call pinn_dp_init first");
  DevGuard dev_guard(h->device);
  for (int r = 0; r < h->dp.args.world; r++) {
    if (r == h->dp.args.rank) continue;
    cudaIpcMemHandle_t ih;
    memcpy(&ih, (const char*)all_handles + (size_t)r * PINN_DP_HANDLE_BYTES, sizeof(ih));
    void* ptr = nullptr;
    CU(h, cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess));
    h->dp.args.peer[r] = (unsigned char*)ptr;
    h->dp.opened[r] = true;
  }
  h->dp.on = true;
  return 0;
}

int pinn_dp_connect_local(pinn_handle* h, pinn_handle* const* peers) {
  if (!h || !peers) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->dp.buf) return fail(h, PINN_EINVAL, "pinn_dp_connect_local: call pinn_dp_init first");
  DevGuard dev_guard(h->device);
  for (int r = 0; r < h->dp.args.world; r++) {
    if (r == h->dp.args.rank) continue;
    pinn_handle* q = peers[r];
    if (!q || !q->dp.buf || q->dp.args.world != h->dp.args.world || q->dp.args.rank != r)
      return fail(h, PINN_EINVAL, "pinn_dp_connect_local: peer handle is not initialised for this rank/world");
    if (q->device != h->device) {
      int can = 0;
      CU(h, cudaDeviceCanAccessPeer(&can, h->device, q->device));
      if (!can) return fail(h, PINN_ENOTSUP, "pinn_dp_connect_local: no peer access between the two devices");
      cudaError_t e = cudaDeviceEnablePeerAccess(q->device, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) return fail(h, (int)e, "cudaDeviceEnablePeerAccess");
    }
    h->dp.args.peer[r] = q->dp.buf;
  }
  h->dp.on = true;
  return 0;
}

int pinn_dp_enable(pinn_handle* h, int on) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (on) {
    for (int r = 0; r < h->dp.args.world; r++)
      if (!h->dp.args.peer[r]) return fail(h, PINN_EINVAL, "pinn_dp_enable: the exchange is not connected");
    if (h->dp.args.world < 1) return fail(h, PINN_EINVAL, "pinn_dp_enable: the exchange is not initialised");
  }
  h->dp.on = on != 0;
  return 0;
}

int pinn_dp_set_timeout(pinn_handle* h, double seconds) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!(seconds > 0.0) || seconds > 3600.0) return fail(h, PINN_EINVAL, "pinn_dp_set_timeout: need 0 < seconds <= 3600");
  if (h->dp.args.world < 1) return fail(h, PINN_EINVAL, "pinn_dp_set_timeout: the exchange is not initialised");
  h->dp.args.timeout_cycles = (long long)(seconds * 2.0e9);  // SM cycles at ~2 GHz: a bound, not a stopwatch
  return 0;
}

int pinn_dp_status(pinn_handle* h, int64_t* exchanges) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->dp.buf) return fail(h, PINN_EINVAL, "pinn_dp_status: the exchange is not initialised");
  DevGuard dev_guard(h->device);
  bool failed = false;
  if (int rc = dp_read_status(h, exchanges, &failed)) return rc;
  if (failed) return fail(h, PINN_ETIMEDOUT, "pinn_dp: a peer did not deliver its partial sums within the time-out");
  return 0;
}

int pinn_dp_shutdown(pinn_handle* h) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  DevGuard dev_guard(h->device);
  CU(h, cudaDeviceSynchronize());
  dp_release(h);
  return 0;
}

}  // extern "C"
