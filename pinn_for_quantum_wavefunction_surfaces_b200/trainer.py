"""Device-resident training loop: the reference's two `train()` drivers (train.py:21-72; poc/main.py:359-430) with the
sampler, the fused loss/gradient kernel and Adam all on the GPU, one CUDA-graph replay per step (SURVEY.md 8f-1, 8f-2).

The reference loops stay usable unchanged through `patch_nn_ion` / `run_train_py` (they keep torch's CPU RNG stream,
which parity runs need); this module is the fast path for runs that do not need that stream:

    sample(...)              <->  train.py:26-39; sampling()+radial()+torch.where  poc/main.py:124-156, 390-393
    sample_adaptive(...)        residual-adaptive batches (RAD) drawn from a pool of sample() points
    Trainer.set_validation      held-out validation loss during training (forward-only loss_eval, best-on-validation record)
    adam_step(...)           <->  optimizer.step() + best/history bookkeeping      train.py:58-72; poc/main.py:403-417
    lbfgs_begin/lbfgs_advance   torch.optim.LBFGS.step(closure), one closure evaluation per device launch
    Trainer                  <->  train()                                          train.py:21-72; poc/main.py:359-430
    train_trainpy / train_poc   convenience drivers with the reference's defaults and return values
"""
import ctypes

import numpy as np
import torch

from . import params as P
from ._lib import Handle, LBFGSConfig, PinnError, TrainConfig

INT64_MAX = (1 << 63) - 1
BOX_POC = (-18.0, 18.0, -18.0, 18.0, -18.0, 18.0, 0.2, 4.0)      # set_params() poc/main.py:17-27
BOX_TRAINPY = (-18.0, 18.0, -18.0, 18.0, -18.0, 18.0, 0.2, 3.0)  # train.py:80-83


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _handle(device=None):
    if not torch.cuda.is_available():
        raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
    return Handle.get(torch.cuda.current_device() if device is None else device)


def sample(n, seed, batch, box=BOX_POC, cutoff=0.005, bcutoff=17.5, device=None):
    """One batch of the device sampler -> dict(x, y, z, R float32 CUDA (n,), mask uint8, counts int64[2], weights f64[3])."""
    h = _handle(device)
    dev = torch.device("cuda", h.device)
    out = {k: torch.empty(n, dtype=torch.float32, device=dev) for k in "xyzR"}
    out["mask"] = torch.empty(n, dtype=torch.uint8, device=dev)
    out["counts"] = torch.zeros(2, dtype=torch.int64, device=dev)
    out["weights"] = torch.empty(3, dtype=torch.float64, device=dev)
    b = (ctypes.c_float * 8)(*box)
    stream = torch.cuda.current_stream(dev).cuda_stream
    rc = h.L.pinn_sample(h.h, n, seed, batch, b, cutoff, bcutoff, _ptr(out["x"]), _ptr(out["y"]), _ptr(out["z"]),
                         _ptr(out["R"]), _ptr(out["mask"]), _ptr(out["counts"]), _ptr(out["weights"]),
                         ctypes.c_void_p(stream))
    h.check(rc, "pinn_sample")
    return out


def sample_adaptive(variant, theta, n, pool_factor=4, k=1.0, c=1.0, seed=0, batch=0, box=None, cutoff=0.005, bcutoff=17.5,
                    device=None, importance=False):
    """Residual-adaptive batch (pinn_sample_adaptive): n points out of pool_factor * n uniform candidates
    (= sample(pool_factor * n, seed, batch)), candidate i taken with probability proportional to
    |res_i|^k * N / sum |res|^k + c, res = the residual of `theta` (packed parameters) there, by systematic resampling.
    -> dict(x, y, z, R, mask, counts, weights as sample(); idx int64 (n,) pool index of each point; pool = dict(x, y, z,
    R, mask) of the candidates; res float32 and cdf float64 (N,), the candidates' residuals and weight prefix sums).
    importance=True (pinn_sample_adaptive_importance; needs c > 0): the same batch, plus "point_weights" float32 (n,),
    om_j = 1 / (N P_i) of the candidate each point came from, and "weights" = {1/n, N/(n |set1 of the pool|),
    N/(n |set2 of the pool|)}: loss_and_grad_raw(..., weights, point_weights=...) on it is an unbiased estimate of the
    pool's uniform loss and gradient."""
    variant = {"poc": 0, "trainpy": 1}.get(variant, variant)
    if box is None:
        box = BOX_POC if variant == 0 else BOX_TRAINPY
    h = _handle(device)
    dev = torch.device("cuda", h.device)
    N = int(pool_factor) * int(n)
    th = torch.as_tensor(np.asarray(theta) if not torch.is_tensor(theta) else theta).detach()
    th = th.to(device=dev, dtype=torch.float32).contiguous()
    col = lambda m, dt=torch.float32: torch.empty(m, dtype=dt, device=dev)
    pool = {k_: col(N) for k_ in "xyzR"}
    pool["mask"] = col(N, torch.uint8)
    out = {k_: col(n) for k_ in "xyzR"}
    out["mask"] = col(n, torch.uint8)
    out["counts"] = torch.zeros(2, dtype=torch.int64, device=dev)
    out["weights"] = col(3, torch.float64)
    out["idx"] = col(n, torch.int64)
    out["pool"], out["res"], out["cdf"] = pool, col(N), col(N, torch.float64)
    b = (ctypes.c_float * 8)(*box)
    stream = torch.cuda.current_stream(dev).cuda_stream
    args = [h.h, variant, _ptr(th), n, N, seed, batch, b, cutoff, bcutoff, k, c,
            *[_ptr(pool[k_]) for k_ in ("x", "y", "z", "R", "mask")], _ptr(out["res"]), _ptr(out["cdf"]),
            *[_ptr(out[k_]) for k_ in ("x", "y", "z", "R", "mask", "idx", "counts", "weights")]]
    if importance:
        out["point_weights"] = col(n)
        rc = h.L.pinn_sample_adaptive_importance(*args, _ptr(out["point_weights"]), ctypes.c_void_p(stream))
        h.check(rc, "pinn_sample_adaptive_importance")
        return out
    rc = h.L.pinn_sample_adaptive(*args, ctypes.c_void_p(stream))
    h.check(rc, "pinn_sample_adaptive")
    return out


class AdamState:
    """Device state of the fused Adam step (float64, like the reference's parameters)."""

    def __init__(self, theta0, device=None, history_capacity=0, best_mode=0):
        h = _handle(device)
        self.h = h
        dev = torch.device("cuda", h.device)
        t64 = lambda a: torch.as_tensor(np.asarray(a, np.float64)).to(dev)
        self.theta = t64(theta0).clone()
        self.m = torch.zeros(P.N_THETA, dtype=torch.float64, device=dev)
        self.v = torch.zeros(P.N_THETA, dtype=torch.float64, device=dev)
        self.theta32 = self.theta.float()
        self.step = torch.zeros(1, dtype=torch.int64, device=dev)
        self.best_loss = torch.full((1,), 10.0, dtype=torch.float64, device=dev)  # Llim = 10, poc/main.py:370
        self.best_theta = self.theta.clone()
        self.best_step = torch.full((1,), -1, dtype=torch.int64, device=dev)
        self.hist = torch.zeros(max(history_capacity, 1), 4, dtype=torch.float64, device=dev)
        self.hist_cap = history_capacity
        self.best_mode = best_mode


def adam_step(state, grad, sums, n, lr=8e-3, betas=(0.9, 0.999), eps=1e-8, grad_mask=0xFFFF, best_after=0,
              history_mean_E=True):
    """One fused optimizer step on `state` (AdamState) from the device outputs of loss_and_grad_raw."""
    h = state.h
    stream = torch.cuda.current_stream(state.theta.device).cuda_stream
    rc = h.L.pinn_adam_step(h.h, _ptr(state.theta), _ptr(state.m), _ptr(state.v), _ptr(grad), _ptr(sums), _ptr(state.theta32),
                            _ptr(state.step), _ptr(state.best_loss), _ptr(state.best_theta), _ptr(state.best_step),
                            _ptr(state.hist) if state.hist_cap else None, state.hist_cap, n, lr, betas[0], betas[1], eps,
                            grad_mask, state.best_mode, best_after, int(history_mean_E), ctypes.c_void_p(stream))
    h.check(rc, "pinn_adam_step")


LBFGS_REASONS = {0: "running", 1: "optimal at start", 2: "directional derivative", 3: "max_iter", 4: "max_eval",
                 5: "tolerance_grad", 6: "step change", 7: "loss change", 8: "slots exhausted"}


def lbfgs_config(max_iter=20, max_eval=None, lr=1, tolerance_grad=1e-7, tolerance_change=1e-9, history_size=100,
                 line_search_fn=None):
    """pinn_lbfgs_config from torch.optim.LBFGS's arguments and defaults."""
    if line_search_fn not in (None, "strong_wolfe"):
        raise ValueError("only 'strong_wolfe' is supported")
    c = LBFGSConfig()
    c.lr, c.max_iter, c.history_size = float(lr), int(max_iter), int(history_size)
    c.max_eval = 0 if max_eval is None else int(max_eval)
    c.line_search = 1 if line_search_fn == "strong_wolfe" else 0
    c.tolerance_grad, c.tolerance_change = float(tolerance_grad), float(tolerance_change)
    return c


def lbfgs_status(status):
    """The 8-double status header of an L-BFGS state -> dict."""
    s = [float(x) for x in status]
    return {"n_iter": int(s[0]), "func_evals": int(s[1]), "evals": int(s[2]), "done": bool(s[3]), "reason": int(s[4]),
            "reason_name": LBFGS_REASONS.get(int(s[4]), "?"), "loss": s[5], "iters": int(s[6]), "t": s[7]}


class LBFGSState:
    """Device state of the L-BFGS machine (pinn_lbfgs_*): zero bytes = a fresh torch.optim.LBFGS.  theta (float64) and
    theta32 hold the point the machine asks to be evaluated next, and its final iterate once it is done."""

    def __init__(self, theta0, history_size=100, device=None):
        h = _handle(device)
        self.h = h
        dev = torch.device("cuda", h.device)
        self.history_size = int(history_size)
        nbytes = int(h.L.pinn_lbfgs_state_bytes(self.history_size))
        if nbytes == 0:
            raise ValueError("history_size must be >= 1")
        self.state = torch.zeros(nbytes // 8, dtype=torch.float64, device=dev)
        self.theta = torch.as_tensor(np.asarray(theta0, np.float64)).to(dev).clone()
        self.theta32 = self.theta.float()

    def status(self):
        """Synchronises; -> dict of the status header."""
        return lbfgs_status(self.state[:8].cpu().numpy())


def lbfgs_begin(state, max_iter=20, max_eval=None, lr=1, tolerance_grad=1e-7, tolerance_change=1e-9, line_search_fn=None):
    """Start one .step() call on `state` (LBFGSState): requests an evaluation at state.theta."""
    c = lbfgs_config(max_iter, max_eval, lr, tolerance_grad, tolerance_change, state.history_size, line_search_fn)
    h = state.h
    stream = torch.cuda.current_stream(state.theta.device).cuda_stream
    h.check(h.L.pinn_lbfgs_begin(h.h, _ptr(state.state), ctypes.byref(c), _ptr(state.theta), _ptr(state.theta32),
                                 ctypes.c_void_p(stream)), "pinn_lbfgs_begin")


def lbfgs_advance(state, sums, grad):
    """Consume the evaluation at the requested point (sums[0] = loss, grad: 1521 float64 CUDA tensors) and request the
    next one, or finish."""
    h = state.h
    stream = torch.cuda.current_stream(state.theta.device).cuda_stream
    h.check(h.L.pinn_lbfgs_advance(h.h, _ptr(state.state), _ptr(sums), _ptr(grad), _ptr(state.theta), _ptr(state.theta32),
                                   ctypes.c_void_p(stream)), "pinn_lbfgs_advance")


class Trainer:
    """pinn_trainer: everything of a training run lives on the device until read()."""

    def __init__(self, variant, n, theta0, seed=12345, lr=8e-3, betas=(0.9, 0.999), eps=1e-8, box=None, cutoff=0.005,
                 bcutoff=17.5, grad_mask=0xFFFF, best_mode=None, best_after=0, sc_sampling=1, freeze_after=INT64_MAX,
                 history_capacity=0, history_mean_E=None, device=None, handle=None, adaptive=None, validation=None):
        variant = {"poc": 0, "trainpy": 1}.get(variant, variant)
        self.h = handle if handle is not None else _handle(device)   # default: the cached per-device Handle
        if box is None:
            box = BOX_POC if variant == 0 else BOX_TRAINPY
        c = TrainConfig()
        c.variant, c.n, c.seed = variant, n, seed
        c.best_mode = (1 if variant == 0 else 0) if best_mode is None else best_mode
        c.history_mean_E = (0 if variant == 0 else 1) if history_mean_E is None else int(history_mean_E)
        c.sc_sampling, c.freeze_after, c.best_after, c.history_capacity = sc_sampling, freeze_after, best_after, history_capacity
        c.xL, c.xR, c.yL, c.yR, c.zL, c.zR, c.RL, c.RR = box
        c.cutoff, c.bcutoff, c.grad_mask = cutoff, bcutoff, grad_mask
        c.lr, c.beta1, c.beta2, c.eps = lr, betas[0], betas[1], eps
        self.cfg = c
        th = np.ascontiguousarray(np.asarray(theta0, np.float64).ravel())
        if th.size != P.N_THETA:
            raise ValueError("theta0 must have 1521 entries")
        tp = ctypes.c_void_p()
        rc = self.h.L.pinn_trainer_create(self.h.h, ctypes.byref(c), th.ctypes.data_as(ctypes.c_void_p), ctypes.byref(tp))
        self.h.check(rc, "pinn_trainer_create")
        self.t = tp
        self._step_base = 0
        if adaptive:
            self.set_adaptive(**adaptive)
        self._val_cap = 0
        if validation:
            self.set_validation(**validation)

    def set_adaptive(self, pool_factor=4, k=1.0, c=1.0, importance=False):
        """Residual-adaptive batches (pinn_trainer_set_adaptive): every resampling step draws its n points from
        pool_factor * n candidates in proportion to |res|^k / mean |res|^k + c at the current parameters; pool_factor=0
        turns it off.  Without importance weights the history and best-model record are evaluated on the adaptive
        batches, a residual-weighted mean that is not comparable with a uniform run's; set_validation records a
        held-out loss that is.  importance=True (pinn_trainer_set_importance; needs c > 0) weights every point of an
        adaptive batch by 1 / (N P_i) and takes the pool's set sizes in the loss weights, so that each step's loss and
        gradient are unbiased estimates of the pool's uniform ones."""
        self.h.check(self.h.L.pinn_trainer_set_adaptive(self.t, int(pool_factor), float(k), float(c)),
                     "pinn_trainer_set_adaptive")
        if importance:
            self.h.check(self.h.L.pinn_trainer_set_importance(self.t, 1), "pinn_trainer_set_importance")

    def set_validation(self, n, seed, every, capacity=None):
        """Held-out validation loss (pinn_trainer_set_validation): n points drawn once now, sample(n, seed, 0) with the
        trainer's box and cutoffs, evaluated (pinn_loss_eval, forward only) after every step that brings the steps done
        since the run (re)started to a multiple of `every`, into `capacity` rows (None: 1024) and a best-on-validation
        record.  The seed has no default: batch 0 of the training seed is the first training batch.  every=0 turns it
        off.  Nothing else the trainer computes changes."""
        if every and capacity is None:
            capacity = 1024
        capacity = int(capacity or 0)
        self.h.check(self.h.L.pinn_trainer_set_validation(self.t, int(n), int(seed), int(every), capacity),
                     "pinn_trainer_set_validation")
        self._val_cap = capacity if every else 0

    def validate(self):
        """Enqueue one validation evaluation now, at the current parameters (a step-0 point, or after run_lbfgs)."""
        self.h.check(self.h.L.pinn_trainer_validate(self.t), "pinn_trainer_validate")

    def read_validation(self):
        """-> dict(rows (k, 4): steps done, Ltot, Lpde, Lbc of each evaluation recorded; evaluations; best_val_theta;
        best_val_loss; best_val_step (-1 while no evaluation was taken))."""
        rows = np.zeros((max(self._val_cap, 1), 4), np.float64)
        best = np.empty(P.N_THETA, np.float64)
        sc = np.zeros(3, np.float64)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        self.h.check(self.h.L.pinn_trainer_read_validation(self.t, p(rows), self._val_cap, p(best), p(sc)),
                     "pinn_trainer_read_validation")
        k = int(sc[0])
        return {"rows": rows[:min(k, self._val_cap)], "evaluations": k, "best_val_theta": best,
                "best_val_loss": float(sc[1]), "best_val_step": int(sc[2])}

    def load_state(self, theta, m=None, v=None, step=0):
        """Resume: parameters, Adam moments (None = zeros) and the number of optimizer steps already done.  The resumed run
        starts its own best-model record (best_theta = the loaded parameters until a step qualifies) and its own history
        (row 0 = the first step after the resume); `freeze_after`, `best_after` and `sc_sampling` keep counting absolute steps."""
        a = lambda x: None if x is None else np.ascontiguousarray(np.asarray(x, np.float64).ravel())
        th, mm, vv = a(theta), a(m), a(v)
        p = lambda x: None if x is None else x.ctypes.data_as(ctypes.c_void_p)
        self.h.check(self.h.L.pinn_trainer_load_state(self.t, p(th), p(mm), p(vv), step), "pinn_trainer_load_state")
        self._step_base = int(step)

    def set_batch(self, x, y, z, R, mask, weights):
        """Use caller-provided points (CUDA or CPU float32 tensors) until the next resampling step."""
        cols = [t.detach().reshape(-1).to(torch.float32).contiguous() for t in (x, y, z, R)]
        mask = mask.detach().reshape(-1).to(torch.uint8).contiguous()
        w = np.ascontiguousarray(np.asarray(weights, np.float64))
        rc = self.h.L.pinn_trainer_set_batch(self.t, *[_ptr(c) for c in cols], _ptr(mask), w.ctypes.data_as(ctypes.c_void_p))
        self.h.check(rc, "pinn_trainer_set_batch")

    def run(self, steps, resample=True, use_graph=False):
        """Enqueue `steps` optimizer steps (asynchronous; read() synchronises).  A step is two launches (step kernel,
        reduction + Adam + next batch), chained as programmatic dependents; use_graph=True replays captured CUDA graphs
        instead, which costs the host less (1.5 vs 7 microseconds per step) but breaks the dependent-launch chain between
        replays (measured 147.6 vs 145.5 microseconds per step at 2^18 points)."""
        self.h.check(self.h.L.pinn_trainer_run(self.t, steps, int(resample), int(use_graph)), "pinn_trainer_run")

    def run_lbfgs(self, max_iter=20, max_eval=None, lr=1, tolerance_grad=1e-7, tolerance_change=1e-9, history_size=100,
                  line_search_fn=None, resample=False, use_graph=False):
        """One torch.optim.LBFGS.step(closure) on the device (pinn_trainer_run_lbfgs), with torch's argument names and
        defaults; the closure is Ltot and its gradient (restricted to grad_mask) on the trainer's current batch, which
        stays fixed (resample=True draws a new one first).  The optimizer state persists across calls.  Adam's moments,
        step counter, history and best-model record are left alone.  Synchronises; -> (status dict, trace (evals, 4):
        Ltot, Lpde, Lbc and step length per evaluation)."""
        c = lbfgs_config(max_iter, max_eval, lr, tolerance_grad, tolerance_change, history_size, line_search_fn)
        self.h.check(self.h.L.pinn_trainer_run_lbfgs(self.t, ctypes.byref(c), int(resample), int(use_graph)),
                     "pinn_trainer_run_lbfgs")
        return self.read_lbfgs()

    def read_lbfgs(self):
        """-> (status dict, trace of the last L-BFGS call)."""
        st = np.zeros(8, np.float64)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        self.h.check(self.h.L.pinn_trainer_read_lbfgs(self.t, p(st), None, 0), "pinn_trainer_read_lbfgs")
        s = lbfgs_status(st)
        tr = np.zeros((max(s["evals"], 1), 4), np.float64)
        self.h.check(self.h.L.pinn_trainer_read_lbfgs(self.t, None, p(tr), s["evals"]), "pinn_trainer_read_lbfgs")
        return s, tr[:s["evals"]]

    def read(self, history_rows=None):
        f = lambda: np.empty(P.N_THETA, np.float64)
        theta, m, v, best = f(), f(), f(), f()
        sc = np.zeros(4, np.float64)
        rows = self.cfg.history_capacity if history_rows is None else min(history_rows, self.cfg.history_capacity)
        hist = np.zeros((max(rows, 0), 4), np.float64)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        rc = self.h.L.pinn_trainer_read(self.t, p(theta), p(m), p(v), p(best), p(sc), p(hist) if rows > 0 else None, rows)
        self.h.check(rc, "pinn_trainer_read")
        steps = int(sc[0])
        return {"theta": theta, "m": m, "v": v, "best_theta": best, "steps": steps, "best_loss": float(sc[1]),
                "best_step": int(sc[2]), "batches": int(sc[3]), "history": hist[:max(0, min(rows, steps - self._step_base))]}

    def close(self):
        if self.t:
            self.h.L.pinn_trainer_destroy(self.t)
            self.t = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def init_trainpy(seed=12345):
    """train.py's initialisation (ini(), train.py:13-18, 74, 88-103) -> packed theta (float64, canonical layout)."""
    g = torch.Generator().manual_seed(seed)
    nh, ne, nl = 16, 32, 10
    shapes = [(2, nh), (nh,), (nh, nh), (nh,), (nh, 1), (1,), (1, nl), (nl,), (nl, 1), (1,),
              (1, ne), (ne,), (ne, ne), (ne,), (ne, 1), (1,)]
    ts = []
    for s in shapes:
        t = torch.empty(s, dtype=torch.float64)
        lim = 1 / s[0] ** 0.5
        t.uniform_(-lim, lim, generator=g)
        ts.append(t)
    return P.pack_trainpy(ts, dtype=torch.float64).numpy()


def init_poc(seed=0):
    """A freshly constructed NN_ion (poc/main.py:233-245): `nn.Linear` default initialisation in float64, layers created in
    the reference's order, `Lin_Eout.bias = -1` -> packed theta (float64).  Equals the real class under
    `torch.manual_seed(seed)` (tests/golden/checkpoints.npz: init_seed0)."""
    nh, ne, nl = 16, 32, 10
    state = torch.get_rng_state()
    try:
        torch.manual_seed(seed)
        dims = [(2, nh), (nh, nh), (nh, 1), (1, ne), (ne, ne), (ne, 1), (1, nl), (nl, 1)]
        layers = [torch.nn.Linear(i, o, dtype=torch.float64) for i, o in dims]
    finally:
        torch.set_rng_state(state)
    with torch.no_grad():
        layers[5].bias.fill_(-1.0)
    ts = []
    for L in layers:
        ts += [L.weight, L.bias]
    return P.pack_poc(ts, dtype=torch.float64).numpy()


def _validation_rows(validation, steps):
    """validation dict of train_poc / train_trainpy -> Trainer.set_validation arguments with room for every row of the run
    (the step-0 evaluation and one per `every` steps)"""
    v = dict(validation)
    if v.get("capacity") is None:
        v["capacity"] = steps // max(int(v["every"]), 1) + 1
    return v


def train_trainpy(theta0=None, n=10000, epochs=1000, lr=8e-3, seed=12345, fine_tune=False, use_graph=False, log_every=0,
                  adaptive=None, validation=None):
    """train(params, lr, epochs) of train.py on the device.  Like the reference it evaluates epochs+1 losses, takes `epochs`
    optimizer steps and returns the parameters of the best loss seen (train.py:58-69).  Returns (theta_best, info).
    adaptive: None (uniform batches) or dict(pool_factor, k, c[, importance]) for residual-adaptive batches
    (Trainer.set_adaptive).
    validation: None, or dict(n, seed, every, capacity=None) for a held-out loss (Trainer.set_validation), evaluated at the
    initial parameters and every `every` steps; info then has a "validation" entry (Trainer.read_validation)."""
    if theta0 is None:
        theta0 = init_trainpy(seed)
    mask = P.FINE_TUNE_GRAD_MASK if fine_tune else 0xFFFF  # train.py:111 (commented) trains the E-net tensors only
    tr = Trainer("trainpy", n, theta0, seed=seed, lr=lr, grad_mask=mask, history_capacity=epochs + 1, adaptive=adaptive,
                 validation=_validation_rows(validation, epochs + 1) if validation else None)
    if validation:
        tr.validate()
    done = 0
    while done < epochs:
        k = min(log_every or epochs, epochs - done)
        tr.run(k, use_graph=use_graph)
        done += k
        if log_every:
            r = tr.read()
            print("%8d: %.2e %.2e %.2e (%.2e) [%.5e]" % (done - 1, *r["history"][done - 1], r["best_loss"]))
    # the reference's loop evaluates the loss once more at tt == epochs before it stops (train.py:41-69): one more step
    # whose parameter update is discarded
    before = tr.read()
    tr.run(1, use_graph=use_graph)
    after = tr.read()
    best = after["best_theta"]
    info = {"history": after["history"], "best_loss": after["best_loss"], "best_step": after["best_step"],
            "theta_last": before["theta"], "batches": after["batches"]}
    if validation:
        info["validation"] = tr.read_validation()
    tr.close()
    return best, info


def train_poc(theta0, params=None, freezeUnits=False, seed=0, use_graph=False, adaptive=None, validation=None):
    """train(params, loadWeights, freezeUnits) of poc/main.py:359-430 on the device.  `params` uses the reference's keys
    (set_params(), poc/main.py:14-45).  Returns (theta_last, theta_saved or None, lossDictionary like poc/main.py:422-427).
    adaptive: None (uniform batches) or dict(pool_factor, k, c[, importance]) for residual-adaptive batches
    (Trainer.set_adaptive).
    validation: None, or dict(n, seed, every, capacity=None) for a held-out loss (Trainer.set_validation), evaluated at
    theta0 and every `every` steps; the loss dictionary then has a "validation" entry (Trainer.read_validation)."""
    pr = {"xL": -18, "xR": 18, "yL": -18, "yR": 18, "zL": -18, "zR": 18, "RxL": 0.2, "RxR": 4, "cutOff": 0.005,
          "BCcutoff": 17.5, "sc_sampling": 1, "n_train": 100000, "epochs": 5000, "lr": 8e-3}
    pr.update(params or {})
    P.check_supported_model(pr)
    epochs = int(pr["epochs"])
    box = (pr["xL"], pr["xR"], pr["yL"], pr["yR"], pr["zL"], pr["zR"], pr["RxL"], pr["RxR"])
    # resample while tt < 0.9*epochs (main.py:396); save when tt > 0.5*epochs and Ltot < Llim (main.py:414)
    freeze_after = int(np.ceil(0.9 * epochs))
    best_after = int(np.floor(0.5 * epochs))
    tr = Trainer("poc", int(pr["n_train"]), theta0, seed=seed, lr=pr["lr"], box=box, cutoff=pr["cutOff"],
                 bcutoff=pr["BCcutoff"], grad_mask=P.FINE_TUNE_GRAD_MASK if freezeUnits else 0xFFFF, best_mode=1,
                 best_after=best_after, sc_sampling=int(pr["sc_sampling"]), freeze_after=freeze_after,
                 history_capacity=epochs, history_mean_E=False, adaptive=adaptive,
                 validation=_validation_rows(validation, epochs) if validation else None)
    if validation:
        tr.validate()
    tr.run(epochs, use_graph=use_graph)
    r = tr.read()
    val = tr.read_validation() if validation else None
    tr.close()
    hcol = lambda k: r["history"][:, k:k + 1].copy()
    loss = {"Ltot": hcol(0), "Lpde": hcol(1), "Lbc": hcol(2), "Energy": hcol(3)}
    if validation:
        loss["validation"] = val
    saved = r["best_theta"] if r["best_step"] >= 0 else None
    return r["theta"], saved, loss
