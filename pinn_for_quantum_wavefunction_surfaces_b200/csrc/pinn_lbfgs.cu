// Device-resident L-BFGS: torch.optim.LBFGS.step(closure) of torch 2.11 (torch/optim/lbfgs.py, with _strong_wolfe and
// _cubic_interpolate) restated in float64 as a machine that advances by exactly one closure evaluation per launch.
// The closure is "Ltot and its gradient at theta"; the caller evaluates it between launches (the trainer: the step
// kernel and the reduction on a fixed batch).  A launch reads the loss and gradient of the point just evaluated, runs
// torch's decisions up to the next closure call and writes that point into theta / theta32, or finishes: theta is then
// torch's final iterate and the done flag is set; later launches change nothing.
//
// One block of LB_THREADS threads.  Thread k owns entries k, k + LB_THREADS, ... of every vector, so element-wise updates
// need no barrier; every dot product, max-abs and abs-sum is a block reduction in a fixed order (each thread's entries in
// index order, a fixed xor-shuffle tree per warp, the warp sums in warp order), so the same inputs give the same bits on
// every run.  Every thread keeps its own copy of the scalar state and takes the same decisions; thread 0 writes it back.
// The scalar arithmetic of the line search and of the two-loop recursion is written with explicit round-to-nearest
// intrinsics where a product meets a sum: no contraction into FMA, so it rounds like the Python expressions it restates.
#include "pinn_handle.h"
#include "pinn_train.h"

namespace pinn {
namespace {

constexpr int LB_THREADS = 256;
constexpr int LB_PER = (NTHETA + LB_THREADS - 1) / LB_THREADS;  // entries a thread owns
constexpr int LB_STRIDE = NPART;           // doubles per vector in the state
constexpr size_t LB_SCALAR_BYTES = 1024;   // the scalar block in front of the vectors
constexpr double C1 = 1e-4, C2 = 0.9;      // _strong_wolfe defaults
constexpr double LS_TOL_CHANGE = 1e-9;     // _strong_wolfe's own tolerance_change (not the optimizer's)

enum Phase { PH_START = 0, PH_LS_BRACKET = 1, PH_LS_ZOOM = 2, PH_FIXED = 3, PH_IDLE = 4 };

// The state block.  The first 8 doubles are the status header of include/pinn_b200.h; a block of zero bytes is a fresh
// optimizer (torch's empty state).
struct LbScalars {
  // status header
  double n_iter, func_evals, evals, done, reason, loss, iters, t_eval;
  // configuration of the current .step() call (pinn_lbfgs_begin)
  double lr, tol_grad, tol_change;
  int max_iter, max_eval, hist_size, line_search;
  // optimizer state kept across calls (torch's state dict): t, H_diag, prev_loss; the history ring (oldest pair in slot
  // hist_head, hist_len pairs)
  double t, H_diag, prev_loss;
  int hist_len, hist_head;
  // this call
  int phase, cur_evals, slots;
  // _strong_wolfe
  double f0, gtd0, d_norm, ls_t, t_prev, f_prev, gtd_prev;
  double b[2], bf[2], bgtd[2];
  int max_ls, ls_iter, ls_evals, ls_done, insuf, low, high, ls_first;
};
static_assert(sizeof(LbScalars) <= LB_SCALAR_BYTES, "scalar block");

struct LbVecs {
  double *x_init, *d, *fg, *pfg, *g_prev, *bg0, *bg1, *S, *Y, *ro, *al;
};
__host__ __device__ inline LbVecs lb_vecs(unsigned char* state, int H) {
  double* v = reinterpret_cast<double*>(state + LB_SCALAR_BYTES);
  LbVecs o;
  o.x_init = v; o.d = v + LB_STRIDE; o.fg = v + 2 * LB_STRIDE; o.pfg = v + 3 * LB_STRIDE; o.g_prev = v + 4 * LB_STRIDE;
  o.bg0 = v + 5 * LB_STRIDE; o.bg1 = v + 6 * LB_STRIDE;
  o.S = v + 7 * LB_STRIDE; o.Y = o.S + (size_t)H * LB_STRIDE;
  o.ro = o.Y + (size_t)H * LB_STRIDE; o.al = o.ro + H;
  return o;
}

#define FOR_OWN(i) for (int i = threadIdx.x; i < NTHETA; i += LB_THREADS)

// the owned entries of a vector in registers (entry threadIdx.x + j LB_THREADS; 0 past the end)
__device__ __forceinline__ void load_row(const double* row, double (&r)[LB_PER]) {
#pragma unroll
  for (int j = 0; j < LB_PER; j++) {
    const int i = threadIdx.x + j * LB_THREADS;
    r[j] = i < NTHETA ? row[i] : 0.0;
  }
}
__device__ __forceinline__ void store_row(const double (&r)[LB_PER], double* row) {
#pragma unroll
  for (int j = 0; j < LB_PER; j++) {
    const int i = threadIdx.x + j * LB_THREADS;
    if (i < NTHETA) row[i] = r[j];
  }
}
// this thread's share of a dot product, in the order of FOR_OWN
__device__ __forceinline__ double own_dot(const double (&a)[LB_PER], const double (&b)[LB_PER]) {
  double v = 0.0;
#pragma unroll
  for (int j = 0; j < LB_PER; j++)
    if (threadIdx.x + j * LB_THREADS < NTHETA) v = fma(a[j], b[j], v);
  return v;
}

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }
// Python's max(a, b) / min(a, b): the first argument unless the second compares greater / smaller
__device__ __forceinline__ double pymax(double a, double b) { return b > a ? b : a; }
__device__ __forceinline__ double pymin(double a, double b) { return b < a ? b : a; }

__device__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  for (int w = 0; w < LB_THREADS / 32; w++) r += red[w];
  __syncthreads();
  return r;
}
// max |.| that keeps a NaN, like torch's abs().max()
__device__ __forceinline__ double nanmax(double a, double b) { return (a > b || a != a) ? a : b; }
__device__ double block_absmax(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = nanmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  for (int w = 0; w < LB_THREADS / 32; w++) r = nanmax(r, red[w]);
  __syncthreads();
  return r;
}
__device__ double dot(const double* a, const double* b, double* red) {
  double v = 0.0;
  FOR_OWN(i) v = fma(a[i], b[i], v);
  return block_sum(v, red);
}
__device__ double absmax(const double* a, double* red) {
  double v = 0.0;
  FOR_OWN(i) v = nanmax(v, fabs(a[i]));
  return block_absmax(v, red);
}

// _cubic_interpolate(x1, f1, g1, x2, f2, g2, bounds=(lo, hi)); has_bounds = 0: the bounds are the two points
__device__ double cubic(double x1, double f1, double g1, double x2, double f2, double g2, bool has_bounds, double lo, double hi) {
  if (!has_bounds) { if (x1 <= x2) { lo = x1; hi = x2; } else { lo = x2; hi = x1; } }
  const double d1 = dsub(dadd(g1, g2), ddiv(dmul(3.0, dsub(f1, f2)), dsub(x1, x2)));
  const double d2sq = dsub(dmul(d1, d1), dmul(g1, g2));
  if (d2sq >= 0) {
    const double d2 = __dsqrt_rn(d2sq);
    double min_pos;
    if (x1 <= x2)
      min_pos = dsub(x2, dmul(dsub(x2, x1), ddiv(dsub(dadd(g2, d2), d1), dadd(dsub(g2, g1), dmul(2.0, d2)))));
    else
      min_pos = dsub(x1, dmul(dsub(x1, x2), ddiv(dsub(dadd(g1, d2), d1), dadd(dsub(g1, g2), dmul(2.0, d2)))));
    return pymin(pymax(min_pos, lo), hi);
  }
  return ddiv(dadd(lo, hi), 2.0);
}

enum Next { N_ITER_TOP, N_AFTER, N_BRACKET_CHECK, N_ZOOM_START, N_ZOOM_TOP, N_LS_RETURN, N_FINISH, N_REQUEST };

struct LbArgs {
  unsigned char* state;
  const double* sums;  // sums[0] = the loss of the point just evaluated (sums[1], sums[2] go to the trace)
  const double* grad;  // its gradient [1521]
  double* theta;
  float* theta32;
  double* trace;       // [trace_rows][4] {Ltot, Lpde, Lbc, step length} per evaluation, or NULL
  long long trace_rows;
  cudaGraphConditionalHandle cond;  // use_cond: the WHILE node of the trainer's graph, cleared when the call ends
  int use_cond;
};

__device__ void finish(LbScalars& s, int reason, const LbArgs& a) {
  FOR_OWN(i) a.theta32[i] = (float)a.theta[i];
  s.done = 1.0; s.reason = (double)reason; s.phase = PH_IDLE;
}

__global__ void __launch_bounds__(LB_THREADS) lbfgs_kernel(const LbArgs a) {
  __shared__ double red[LB_THREADS / 32];
  pdl_wait();
  LbScalars s = *reinterpret_cast<const LbScalars*>(a.state);
  if (s.done != 0.0 || s.phase == PH_IDLE) {
    if (a.use_cond && threadIdx.x == 0) cudaGraphSetConditional(a.cond, 0);
    return;
  }
  const int H = s.hist_size;
  const LbVecs v = lb_vecs(a.state, H);
  const double* g = a.grad;
  const double f_new = a.sums[0];
  if (threadIdx.x == 0 && a.trace && (long long)s.evals < a.trace_rows) {
    double* row = a.trace + 4 * (long long)s.evals;
    row[0] = a.sums[0]; row[1] = a.sums[1]; row[2] = a.sums[2]; row[3] = s.t_eval;
  }
  s.evals += 1.0;
  double gtd_new = 0.0;
  int ls_add = 0;         // evaluations torch adds to current_evals at the end of this iteration
  bool opt_cond = false;
  int next = N_FINISH, reason = 0;

  switch (s.phase) {
    case PH_START:  // orig_loss = closure(): the first evaluation of .step()
      s.cur_evals = 1; s.func_evals += 1.0; s.loss = f_new;
      FOR_OWN(i) v.fg[i] = g[i];
      if (absmax(v.fg, red) <= s.tol_grad) { reason = PINN_LBFGS_OPTIMAL_AT_START; next = N_FINISH; }
      else next = N_ITER_TOP;
      break;
    case PH_FIXED:  // line_search_fn=None: the re-evaluation after the fixed step
      s.loss = f_new;
      FOR_OWN(i) v.fg[i] = g[i];
      opt_cond = absmax(v.fg, red) <= s.tol_grad;
      ls_add = 1;
      next = N_AFTER;
      break;
    case PH_LS_BRACKET:
      s.ls_evals++;
      gtd_new = dot(g, v.d, red);
      if (!s.ls_first) s.ls_iter++;
      s.ls_first = 0;
      next = N_BRACKET_CHECK;
      break;
    case PH_LS_ZOOM: {
      s.ls_evals++;
      gtd_new = dot(g, v.d, red);
      s.ls_iter++;
      const int lo = s.low, hi = s.high;
      double* bgl = lo ? v.bg1 : v.bg0;
      double* bgh = hi ? v.bg1 : v.bg0;
      if (f_new > dadd(s.f0, dmul(dmul(C1, s.ls_t), s.gtd0)) || f_new >= s.bf[lo]) {
        s.b[hi] = s.ls_t; s.bf[hi] = f_new; s.bgtd[hi] = gtd_new;
        FOR_OWN(i) bgh[i] = g[i];
        if (s.bf[0] <= s.bf[1]) { s.low = 0; s.high = 1; } else { s.low = 1; s.high = 0; }
      } else {
        if (fabs(gtd_new) <= dmul(-C2, s.gtd0)) s.ls_done = 1;
        else if (dmul(gtd_new, dsub(s.b[hi], s.b[lo])) >= 0) {
          s.b[hi] = s.b[lo]; s.bf[hi] = s.bf[lo]; s.bgtd[hi] = s.bgtd[lo];
          FOR_OWN(i) bgh[i] = bgl[i];
        }
        s.b[lo] = s.ls_t; s.bf[lo] = f_new; s.bgtd[lo] = gtd_new;
        FOR_OWN(i) bgl[i] = g[i];
      }
      next = N_ZOOM_TOP;
      break;
    }
    default:
      break;
  }

  // torch's control flow from here to the next closure call
  double req_t = 0.0;  // N_REQUEST: evaluate x_init + req_t * d (line search) or theta as it stands (fixed step)
  bool req_from_x_init = false;
  for (;;) {
    if (next == N_FINISH) { finish(s, reason, a); break; }
    if (next == N_REQUEST) {
      if (req_from_x_init) FOR_OWN(i) a.theta[i] = fma(req_t, v.d[i], v.x_init[i]);
      FOR_OWN(i) a.theta32[i] = (float)a.theta[i];
      s.t_eval = req_t;
      break;
    }
    switch (next) {
      case N_ITER_TOP: {
        s.iters += 1.0; s.n_iter += 1.0;
        if (s.n_iter == 1.0) {
          FOR_OWN(i) v.d[i] = -v.fg[i];
          s.hist_len = 0; s.hist_head = 0; s.H_diag = 1.0;
        } else {
          // y = flat_grad - prev_flat_grad, s = d * t; the pair enters the history only if y.s > 1e-10
          double part = 0.0;
          FOR_OWN(i) part = fma(v.fg[i] - v.pfg[i], v.d[i] * s.t, part);
          const double ys = block_sum(part, red);
          if (ys > 1e-10) {
            int slot;
            if (s.hist_len == H) { slot = s.hist_head; s.hist_head = (s.hist_head + 1) % H; }
            else { slot = (s.hist_head + s.hist_len) % H; s.hist_len++; }
            double* Ys = v.Y + (size_t)slot * LB_STRIDE;
            double* Ss = v.S + (size_t)slot * LB_STRIDE;
            FOR_OWN(i) { Ys[i] = v.fg[i] - v.pfg[i]; Ss[i] = v.d[i] * s.t; }
            if (threadIdx.x == 0) v.ro[slot] = 1.0 / ys;
            s.H_diag = ys / dot(Ys, Ys, red);
          }
          // two-loop recursion, q and then r in registers; history index k (0 = oldest) lives in slot (head + k) % H.
          // The rows of the next history step are loaded before the reduction of the current one.
          const int num_old = s.hist_len;
          double q[LB_PER], ra[LB_PER], rb[LB_PER], na[LB_PER], nb[LB_PER];
          load_row(v.fg, q);
#pragma unroll
          for (int j = 0; j < LB_PER; j++) q[j] = -q[j];
          auto slot = [&](int k) { return (size_t)((s.hist_head + k) % H); };
          double ro_c = 0.0, ro_n = 0.0, al_c = 0.0, al_n = 0.0;
          if (num_old > 0) {
            load_row(v.S + slot(num_old - 1) * LB_STRIDE, ra); load_row(v.Y + slot(num_old - 1) * LB_STRIDE, rb);
            ro_c = v.ro[slot(num_old - 1)];
          }
          for (int k = num_old - 1; k >= 0; k--) {  // ra = s_k, rb = y_k
            if (k > 0) {
              load_row(v.S + slot(k - 1) * LB_STRIDE, na); load_row(v.Y + slot(k - 1) * LB_STRIDE, nb);
              ro_n = v.ro[slot(k - 1)];
            }
            const double al = block_sum(own_dot(ra, q), red) * ro_c;
            if (threadIdx.x == 0) v.al[slot(k)] = al;
#pragma unroll
            for (int j = 0; j < LB_PER; j++) { q[j] = fma(-al, rb[j], q[j]); ra[j] = na[j]; rb[j] = nb[j]; }
            ro_c = ro_n;
          }
          __syncthreads();  // al of every slot is written
#pragma unroll
          for (int j = 0; j < LB_PER; j++) q[j] = q[j] * s.H_diag;
          if (num_old > 0) {
            load_row(v.Y + slot(0) * LB_STRIDE, ra); load_row(v.S + slot(0) * LB_STRIDE, rb);
            ro_c = v.ro[slot(0)]; al_c = v.al[slot(0)];
          }
          for (int k = 0; k < num_old; k++) {  // ra = y_k, rb = s_k
            if (k + 1 < num_old) {
              load_row(v.Y + slot(k + 1) * LB_STRIDE, na); load_row(v.S + slot(k + 1) * LB_STRIDE, nb);
              ro_n = v.ro[slot(k + 1)]; al_n = v.al[slot(k + 1)];
            }
            const double be = dmul(block_sum(own_dot(ra, q), red), ro_c);
            const double c = dsub(al_c, be);  // torch rounds be_i before the subtraction: no FMA here
#pragma unroll
            for (int j = 0; j < LB_PER; j++) { q[j] = fma(c, rb[j], q[j]); ra[j] = na[j]; rb[j] = nb[j]; }
            ro_c = ro_n; al_c = al_n;
          }
          store_row(q, v.d);
        }
        FOR_OWN(i) v.pfg[i] = v.fg[i];
        s.prev_loss = s.loss;
        if (s.n_iter == 1.0) {
          double part = 0.0;
          FOR_OWN(i) part += fabs(v.fg[i]);
          const double inv = 1.0 / block_sum(part, red);
          s.t = pymin(1.0, inv) * s.lr;
        } else {
          s.t = s.lr;
        }
        const double gtd = dot(v.fg, v.d, red);
        if (gtd > -s.tol_change) { reason = PINN_LBFGS_DIRECTIONAL_DERIVATIVE; next = N_FINISH; break; }
        if (s.line_search) {
          FOR_OWN(i) { v.x_init[i] = a.theta[i]; v.g_prev[i] = v.fg[i]; }
          s.d_norm = absmax(v.d, red);
          s.f0 = s.loss; s.gtd0 = gtd;
          s.ls_t = s.t; s.t_prev = 0.0; s.f_prev = s.loss; s.gtd_prev = gtd;
          s.ls_iter = 0; s.ls_evals = 0; s.ls_done = 0; s.insuf = 0; s.ls_first = 1;
          s.max_ls = s.max_eval - s.cur_evals;
          s.phase = PH_LS_BRACKET;
          req_t = s.ls_t; req_from_x_init = true; next = N_REQUEST;
        } else {
          FOR_OWN(i) a.theta[i] = fma(s.t, v.d[i], a.theta[i]);
          if (s.iters != (double)s.max_iter) {
            s.phase = PH_FIXED;
            req_t = s.t; req_from_x_init = false; next = N_REQUEST;
          } else {
            ls_add = 0; next = N_AFTER;
          }
        }
        break;
      }
      case N_AFTER: {
        s.cur_evals += ls_add; s.func_evals += (double)ls_add;
        if (s.iters == (double)s.max_iter) { reason = PINN_LBFGS_MAX_ITER; next = N_FINISH; break; }
        if (s.cur_evals >= s.max_eval) { reason = PINN_LBFGS_MAX_EVAL; next = N_FINISH; break; }
        if (opt_cond) { reason = PINN_LBFGS_TOLERANCE_GRAD; next = N_FINISH; break; }
        double m = 0.0;
        FOR_OWN(i) m = nanmax(m, fabs(v.d[i] * s.t));
        if (block_absmax(m, red) <= s.tol_change) { reason = PINN_LBFGS_STEP_CHANGE; next = N_FINISH; break; }
        if (fabs(s.loss - s.prev_loss) < s.tol_change) { reason = PINN_LBFGS_LOSS_CHANGE; next = N_FINISH; break; }
        next = N_ITER_TOP;
        break;
      }
      case N_BRACKET_CHECK: {
        const double t = s.ls_t;
        if (s.ls_iter < s.max_ls) {
          const bool armijo_fail = f_new > dadd(s.f0, dmul(dmul(C1, t), s.gtd0)) || (s.ls_iter > 1 && f_new >= s.f_prev);
          const bool wolfe = fabs(gtd_new) <= dmul(-C2, s.gtd0);
          if (armijo_fail || (!wolfe && gtd_new >= 0)) {
            s.b[0] = s.t_prev; s.b[1] = t; s.bf[0] = s.f_prev; s.bf[1] = f_new; s.bgtd[0] = s.gtd_prev; s.bgtd[1] = gtd_new;
            FOR_OWN(i) { v.bg0[i] = v.g_prev[i]; v.bg1[i] = g[i]; }
            next = N_ZOOM_START;
          } else if (wolfe) {
            // one-point bracket [t]: the zoom is skipped and t is returned
            s.b[0] = t; s.bf[0] = f_new; s.b[1] = t; s.bf[1] = f_new;
            FOR_OWN(i) v.bg0[i] = g[i];
            s.ls_done = 1;
            next = N_ZOOM_START;
          } else {
            const double min_step = dadd(t, dmul(0.01, dsub(t, s.t_prev)));
            const double max_step = dmul(t, 10.0);
            s.ls_t = cubic(s.t_prev, s.f_prev, s.gtd_prev, t, f_new, gtd_new, true, min_step, max_step);
            s.t_prev = t; s.f_prev = f_new; s.gtd_prev = gtd_new;
            FOR_OWN(i) v.g_prev[i] = g[i];
            s.phase = PH_LS_BRACKET;
            req_t = s.ls_t; req_from_x_init = true; next = N_REQUEST;
          }
        } else {  // ls_iter == max_ls: bracket [0, t] around the start and the last trial
          s.b[0] = 0.0; s.b[1] = t; s.bf[0] = s.f0; s.bf[1] = f_new;
          FOR_OWN(i) { v.bg0[i] = v.fg[i]; v.bg1[i] = g[i]; }
          next = N_ZOOM_START;
        }
        break;
      }
      case N_ZOOM_START:
        if (s.bf[0] <= s.bf[1]) { s.low = 0; s.high = 1; } else { s.low = 1; s.high = 0; }
        next = N_ZOOM_TOP;
        break;
      case N_ZOOM_TOP: {
        if (s.ls_done || s.ls_iter >= s.max_ls) { next = N_LS_RETURN; break; }
        if (dmul(fabs(dsub(s.b[1], s.b[0])), s.d_norm) < LS_TOL_CHANGE) { next = N_LS_RETURN; break; }
        double t = cubic(s.b[0], s.bf[0], s.bgtd[0], s.b[1], s.bf[1], s.bgtd[1], false, 0.0, 0.0);
        const double bmax = pymax(s.b[0], s.b[1]), bmin = pymin(s.b[0], s.b[1]);
        const double eps = dmul(0.1, dsub(bmax, bmin));
        if (pymin(dsub(bmax, t), dsub(t, bmin)) < eps) {
          if (s.insuf || t >= bmax || t <= bmin) {
            if (fabs(dsub(t, bmax)) < fabs(dsub(t, bmin))) t = dsub(bmax, eps);
            else t = dadd(bmin, eps);
            s.insuf = 0;
          } else {
            s.insuf = 1;
          }
        } else {
          s.insuf = 0;
        }
        s.ls_t = t;
        s.phase = PH_LS_ZOOM;
        req_t = t; req_from_x_init = true; next = N_REQUEST;
        break;
      }
      case N_LS_RETURN: {
        // t = bracket[low]; the optimizer then steps from x_init by t
        const int lo = s.low;
        s.t = s.b[lo]; s.loss = s.bf[lo];
        const double* bgl = lo ? v.bg1 : v.bg0;
        FOR_OWN(i) { v.fg[i] = bgl[i]; a.theta[i] = fma(s.t, v.d[i], v.x_init[i]); }
        opt_cond = absmax(v.fg, red) <= s.tol_grad;
        ls_add = s.ls_evals;
        next = N_AFTER;
        break;
      }
      default:
        next = N_FINISH;
        break;
    }
  }
  // a call never evaluates more than its slots: max_eval, + 1 where the line search's first trial overruns
  if (s.done == 0.0 && s.evals >= (double)s.slots) { s.done = 1.0; s.reason = PINN_LBFGS_SLOTS_EXHAUSTED; s.phase = PH_IDLE; }
  if (a.use_cond && threadIdx.x == 0 && s.done != 0.0) cudaGraphSetConditional(a.cond, 0);
  __syncthreads();
  if (threadIdx.x == 0) *reinterpret_cast<LbScalars*>(a.state) = s;
}

__global__ void __launch_bounds__(LB_THREADS) lbfgs_begin_kernel(unsigned char* state, const pinn_lbfgs_config c, int slots,
                                                                 const double* theta, float* theta32) {
  pdl_wait();
  FOR_OWN(i) theta32[i] = (float)theta[i];
  if (threadIdx.x != 0) return;
  LbScalars* s = reinterpret_cast<LbScalars*>(state);
  s->lr = c.lr; s->tol_grad = c.tolerance_grad; s->tol_change = c.tolerance_change;
  s->max_iter = c.max_iter; s->max_eval = c.max_eval; s->hist_size = c.history_size; s->line_search = c.line_search;
  s->phase = PH_START; s->cur_evals = 0; s->slots = slots;
  s->evals = 0.0; s->done = 0.0; s->reason = 0.0; s->iters = 0.0; s->t_eval = 0.0;
}

// In front of the WHILE node: the loop runs only while the call has not finished
__global__ void lbfgs_cond_kernel(const unsigned char* state, cudaGraphConditionalHandle cond) {
  const LbScalars* s = reinterpret_cast<const LbScalars*>(state);
  cudaGraphSetConditional(cond, (s->done == 0.0 && s->phase != PH_IDLE) ? 1u : 0u);
}

}  // namespace

cudaError_t launch_lbfgs_cond(const unsigned char* state, cudaGraphConditionalHandle cond, cudaStream_t st) {
  lbfgs_cond_kernel<<<1, 1, 0, st>>>(state, cond);
  return cudaGetLastError();
}

size_t lbfgs_state_bytes(int history_size) {
  return LB_SCALAR_BYTES + sizeof(double) * ((size_t)(7 + 2 * (size_t)history_size) * LB_STRIDE + 2 * (size_t)history_size);
}

int lbfgs_slots(const pinn_lbfgs_config& c) { return c.max_eval + (c.line_search ? 1 : 0); }

cudaError_t launch_lbfgs_begin(unsigned char* state, const pinn_lbfgs_config& c, const double* theta, float* theta32,
                               cudaStream_t st) {
  return launch_pdl(lbfgs_begin_kernel, dim3(1), dim3(LB_THREADS), 0, st, state, c, lbfgs_slots(c), theta, theta32);
}

cudaError_t launch_lbfgs_advance(unsigned char* state, const double* sums, const double* grad, double* theta, float* theta32,
                                 double* trace, long long trace_rows, const cudaGraphConditionalHandle* cond, cudaStream_t st) {
  LbArgs a{};
  a.state = state; a.sums = sums; a.grad = grad; a.theta = theta; a.theta32 = theta32; a.trace = trace;
  a.trace_rows = trace_rows; a.use_cond = cond != nullptr; a.cond = cond ? *cond : 0;
  return launch_pdl(lbfgs_kernel, dim3(1), dim3(LB_THREADS), 0, st, a);
}

}  // namespace pinn

// torch's defaults for what the caller left unset, then the checks of every entry
int lbfgs_resolve_config(pinn_handle* h, const pinn_lbfgs_config* in, pinn_lbfgs_config* out) {
  if (!in) return fail(h, PINN_EINVAL, "pinn_lbfgs: NULL config");
  pinn_lbfgs_config c = *in;
  if (c.max_eval <= 0) c.max_eval = c.max_iter * 5 / 4;
  if (!(c.lr >= 0.0) || !std::isfinite(c.lr) || c.max_iter < 1 || c.max_eval < 1 || c.history_size < 1 ||
      (c.line_search != 0 && c.line_search != 1) || !(c.tolerance_grad >= 0.0) || !(c.tolerance_change >= 0.0) ||
      c.max_iter > (1 << 24) || c.max_eval > (1 << 24) || c.history_size > (1 << 16))
    return fail(h, PINN_EINVAL, "pinn_lbfgs: bad config (lr >= 0, max_iter >= 1, history_size >= 1, line_search 0 or 1, "
                                "tolerances >= 0)");
  *out = c;
  return 0;
}

extern "C" {

size_t pinn_lbfgs_state_bytes(int history_size) { return history_size < 1 ? 0 : pinn::lbfgs_state_bytes(history_size); }

int pinn_lbfgs_begin(pinn_handle* h, void* state, const pinn_lbfgs_config* cfg, const double* theta, float* theta32,
                     void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  pinn_lbfgs_config c;
  if (int rc = lbfgs_resolve_config(h, cfg, &c)) return rc;
  if (!state || !theta || !theta32) return fail(h, PINN_EINVAL, "pinn_lbfgs_begin: NULL pointer argument");
  DevGuard dev_guard(h->device);
  CU(h, pinn::launch_lbfgs_begin(static_cast<unsigned char*>(state), c, theta, theta32, (cudaStream_t)stream));
  h->launches += 1;
  return 0;
}

int pinn_lbfgs_advance(pinn_handle* h, void* state, const double* sums, const double* grad, double* theta, float* theta32,
                       void* stream) {
  if (!h) return PINN_EINVAL;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!state || !sums || !grad || !theta || !theta32) return fail(h, PINN_EINVAL, "pinn_lbfgs_advance: NULL pointer argument");
  DevGuard dev_guard(h->device);
  CU(h, pinn::launch_lbfgs_advance(static_cast<unsigned char*>(state), sums, grad, theta, theta32, nullptr, 0, nullptr,
                                   (cudaStream_t)stream));
  h->launches += 1;
  return 0;
}

}  // extern "C"
