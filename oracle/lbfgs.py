"""torch.optim.LBFGS itself driven on a flat float64 vector (TEST INFRASTRUCTURE ONLY), the way
train_loop.adam_reference drives torch.optim.Adam.  No restatement of the algorithm: torch is the reference.

    run(fg, x0, steps, free=None, **lbfgs_kwargs) -> one record per .step() call: the points at which torch called the
        closure, its counters, the termination reason and the final iterate
    CoverageTracer       the lines of torch/optim/lbfgs.py that ran (sys.settrace), and the termination of each step

fg(x) -> (f, g): the objective at a float64 numpy vector and its gradient.  free: None, or a list of (size, bool) segments
of x: a segment with bool False is a frozen parameter tensor (its .grad stays None, which _gather_flat_grad turns into
zeros - what the device reduction writes for a tensor outside grad_mask).
"""
import inspect
import sys

import numpy as np
import torch
import torch.optim.lbfgs as _lb

LBFGS_FILE = _lb.__file__
_SRC, _FIRST = inspect.getsourcelines(_lb)

# reason codes of include/pinn_b200.h (PINN_LBFGS_*), keyed by the condition line whose `break` / `return` ran
_REASON_LINES = [
    ("if opt_cond:\n", "return orig_loss", 1),
    ("if gtd > -tolerance_change:", "break", 2),
    ("if n_iter == max_iter:", "break", 3),
    ("if current_evals >= max_eval:", "break", 4),
    ("if opt_cond:\n", "break", 5),
    ("if d.mul(t).abs().max() <= tolerance_change:", "break", 6),
    ("if abs(loss - prev_loss) < tolerance_change:", "break", 7),
]


def _reason_map():
    """line number of each terminating statement -> reason code"""
    out = {}
    for cond, stmt, code in _REASON_LINES:
        for k, line in enumerate(_SRC):
            if line.strip() == cond.strip() and _SRC[k + 1].strip() == stmt:
                out[_FIRST + k + 1] = code
                break
        else:
            raise RuntimeError("torch/optim/lbfgs.py: cannot find %r" % cond)
    return out


REASON_LINES = _reason_map()


def function_lines(fn):
    """Executable lines of a function and the functions nested in it."""
    lines = set()
    todo = [inspect.unwrap(fn).__code__]
    while todo:
        co = todo.pop()
        lines.update(ln for _, _, ln in co.co_lines() if ln is not None and ln != co.co_firstlineno)
        todo.extend(c for c in co.co_consts if inspect.iscode(c))
    return lines


class CoverageTracer:
    """Records every line of torch/optim/lbfgs.py that runs while active; `last_reason` is the termination of the last
    .step() call."""

    def __init__(self):
        self.lines = set()
        self.hits = {}  # line -> times it ran
        self.last_reason = 0

    def _trace(self, frame, event, arg):
        if frame.f_code.co_filename != LBFGS_FILE:
            return None
        if event == "line":
            self.lines.add(frame.f_lineno)
            self.hits[frame.f_lineno] = self.hits.get(frame.f_lineno, 0) + 1
            r = REASON_LINES.get(frame.f_lineno)
            if r:
                self.last_reason = r
        return self._trace

    def __enter__(self):
        self._old = sys.gettrace()
        sys.settrace(self._trace)
        return self

    def __exit__(self, *exc):
        sys.settrace(self._old)


def run(fg, x0, steps=1, free=None, tracer=None, **kw):
    """torch.optim.LBFGS(**kw) for `steps` .step() calls from x0.  Returns a list of dicts, one per call:
    points (evals, n) where the closure was called, losses (evals,), evals, n_iter and func_evals (torch's state after the
    call), reason (PINN_LBFGS_*), hist_len (curvature pairs held), x (the iterate after the call)."""
    x0 = np.asarray(x0, np.float64)
    segs = free if free is not None else [(x0.size, True)]
    if sum(s for s, _ in segs) != x0.size:
        raise ValueError("segments do not cover x0")
    params, off = [], 0
    for s, _ in segs:
        params.append(torch.tensor(x0[off:off + s].copy(), dtype=torch.float64, requires_grad=True))
        off += s
    opt = torch.optim.LBFGS(params, **kw)
    tr = tracer if tracer is not None else CoverageTracer()
    out = []
    for _ in range(steps):
        pts, fs = [], []

        def closure():
            x = torch.cat([p.detach() for p in params]).numpy().copy()
            f, g = fg(x)
            pts.append(x)
            fs.append(float(f))
            off = 0
            for p, (s, on) in zip(params, segs):
                p.grad = torch.tensor(np.asarray(g[off:off + s], np.float64).copy()) if on else None
                off += s
            return torch.tensor(float(f), dtype=torch.float64)

        tr.last_reason = 0
        with tr:
            opt.step(closure)
        st = opt.state[params[0]]
        out.append({"points": np.array(pts), "losses": np.array(fs), "evals": len(pts), "n_iter": int(st["n_iter"]),
                    "func_evals": int(st["func_evals"]), "reason": tr.last_reason, "hist_len": len(st.get("old_dirs") or []),
                    "x": torch.cat([p.detach() for p in params]).numpy().copy()})
    return out


# ---- test problems (float64 numpy) ----
def rosenbrock(x):
    """extended Rosenbrock: sum over pairs 100 (x[2i+1] - x[2i]^2)^2 + (1 - x[2i])^2; odd length: the last entry enters
    a plain quadratic"""
    n2 = x.size // 2 * 2
    a, b = x[0:n2:2], x[1:n2:2]
    f = float(np.sum(100.0 * (b - a * a) ** 2 + (1.0 - a) ** 2))
    g = np.zeros_like(x)
    g[0:n2:2] = -400.0 * a * (b - a * a) - 2.0 * (1.0 - a)
    g[1:n2:2] = 200.0 * (b - a * a)
    if x.size > n2:
        f += float(x[-1] ** 2)
        g[-1] = 2.0 * x[-1]
    return f, g


def quadratic(diag, center):
    """0.5 sum diag (x - center)^2"""
    def fg(x):
        r = x - center
        return float(0.5 * np.sum(diag * r * r)), diag * r
    return fg


def nonconvex(x):
    """sum sin(x_i) + 0.05 x_i^2: indefinite curvature, so y.s <= 0 happens under fixed steps"""
    return float(np.sum(np.sin(x) + 0.05 * x * x)), np.cos(x) + 0.1 * x


def pinn_problem(n=1024, mask=0x0FC0):
    """The poc loss of the float64 oracle (closed_form.loss_and_grad) on the first n golden points (float32-rounded
    coordinates, as the device reads them) at the paper re-run's stage-1 parameters, with the tensors outside `mask`
    frozen -> (fg, x0, free segments)"""
    import os
    from . import closed_form as cf
    from . import layout
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
    g = np.load(os.path.join(root, "poc_seed0_n4096.npz"))
    th = np.load(os.path.join(root, "poc_paper_run_seed0.npz"))["theta_stage1_saved"].astype(np.float64)
    m1 = np.zeros(g["x"].size); m1[g["i1"]] = 1
    m2 = np.zeros(g["x"].size); m2[g["i2"]] = 1
    pts = [g[k][:n].astype(np.float32).astype(np.float64) for k in "xyzR"]
    m1, m2 = m1[:n], m2[:n]

    def fg(x):
        o = cf.loss_and_grad("poc", x, *pts, m1, m2)
        return o["Ltot"], o["grad"]
    offs = layout.offsets() + [layout.N_THETA]
    free = [(offs[k + 1] - offs[k], bool((mask >> k) & 1)) for k in range(16)]
    return fg, th, free


def kink(x):
    """sum |x - 0.3|: the slope never shrinks, so the zoom narrows the bracket until it is too small to go on"""
    return float(np.sum(np.abs(x - 0.3))), np.sign(x - 0.3)


def wiggly(a, w):
    """sum 0.5 x^2 + a sin(w x + 1): cubic steps that land at or near a bracket end"""
    def fg(x):
        return float(np.sum(0.5 * x * x + a * np.sin(w * x + 1.0))), x + a * w * np.cos(w * x + 1.0)
    return fg


def problems():
    """name -> (fg, x0, steps, free, torch.optim.LBFGS kwargs): the cases the tests run on torch and on the device.
    Between them every line of _strong_wolfe, _cubic_interpolate and LBFGS.step runs (tests/test_oracle_lbfgs.py)."""
    n = 1521
    x_rosen = np.where(np.arange(n) % 2 == 0, -1.2, 1.0)
    rng = np.random.default_rng(7)
    diag = rng.uniform(1.0, 10.0, n)
    center = rng.standard_normal(n)
    x_nc = rng.uniform(-3.0, 3.0, n)
    fg_pinn, th_pinn, free_pinn = pinn_problem()
    sw = "strong_wolfe"
    return {
        # Rosenbrock amplifies rounding about 100-fold every 5 iterations (torch against itself with 1-ulp gradient
        # noise: 5e-13 of the point after 15 iterations, 1e-8 after 25): the runs stay short enough to compare points
        "rosenbrock_1521": (rosenbrock, x_rosen, 1, None, dict(max_iter=15, history_size=20, line_search_fn=sw)),
        "quadratic_tolerance_grad": (quadratic(diag, center), np.zeros(n), 2, None,
                                     dict(max_iter=100, tolerance_grad=1e-3, history_size=10, line_search_fn=sw)),
        "nonconvex_fixed_step": (nonconvex, x_nc, 1, None, dict(max_iter=40, lr=0.5, history_size=10)),
        "history_3": (rosenbrock, x_rosen[:40], 1, None, dict(max_iter=30, history_size=3, line_search_fn=sw)),
        "max_eval_in_line_search": (quadratic(diag, center), np.zeros(n), 2, None,
                                    dict(lr=1e-4, max_iter=20, max_eval=6, line_search_fn=sw)),
        "persisted_state": (rosenbrock, x_rosen[:100], 3, None, dict(max_iter=4, history_size=5, line_search_fn=sw)),
        "quadratic_directional_derivative": (quadratic(diag, center), np.zeros(n), 1, None,
                                             dict(max_iter=100, tolerance_change=1e-2, line_search_fn=sw)),
        "persisted_state_fixed_step": (rosenbrock, x_rosen[:100] * 0.1, 3, None, dict(max_iter=5, lr=1e-3, history_size=4)),
        "fixed_step_lack_of_progress": (quadratic(diag, center), np.zeros(n), 1, None,
                                        dict(max_iter=10, lr=1e-6, tolerance_change=1e-4)),
        "frozen_mask": (rosenbrock, x_rosen, 1, [(500, True), (521, False), (500, True)],
                        dict(max_iter=25, history_size=10, line_search_fn=sw)),
        "kink_1d": (kink, np.array([-1.0]), 1, None, dict(max_iter=20, max_eval=200, line_search_fn=sw)),
        "wiggly_1d_near_lower_end": (wiggly(0.02, 20.0), np.random.default_rng(0).uniform(-3, 3, 1), 1, None,
                                     dict(max_iter=30, lr=20, line_search_fn=sw)),
        "wiggly_1d_near_upper_end": (wiggly(0.01, 40.0), np.random.default_rng(16).uniform(-3, 3, 1), 1, None,
                                     dict(max_iter=30, lr=10, line_search_fn=sw)),
        "pinn_oracle": (fg_pinn, th_pinn, 1, free_pinn,
                        dict(max_iter=15, history_size=20, tolerance_grad=0, tolerance_change=0, line_search_fn=sw)),
    }
