"""The device L-BFGS (pinn_lbfgs_*, Trainer.run_lbfgs) against torch.optim.LBFGS itself (oracle/lbfgs.py).

Stand-alone entries: the host computes f and g in float64 and the device keeps the state; the points the device asks to
be evaluated must be torch's, point for point, and the counters and the termination reason must be torch's exactly.
Trainer: its evaluations (step kernel + reduction on a fixed batch) are compared with the stand-alone entries fed by
loss_and_grad_raw, bit for bit, in the plain and the graph form."""
import ctypes
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import layout
from oracle import lbfgs as O

pytestmark = pytest.mark.gpu

N = 1521
# Relative bar on the requested points, max|device - torch| / max|torch| over a problem's calls.  The device sums dot
# products in another order than torch's BLAS and fuses its vector updates, so the points differ by rounding, which the
# iterations amplify.  Measured on a B200: at most 4.0e-12 (frozen_mask; torch against itself with 1-ulp gradient noise
# moves that run by 6e-8), 0 to 1.4e-12 on the other 1521-entry runs, 0 on the 1-D ones.  Bar: 25x the largest.
POINT_RTOL = 1e-10


def device_run(fg, x0, steps, free, kw):
    """The problem on the stand-alone entries: x0 padded to 1521 entries whose gradient is 0, frozen segments too."""
    n = x0.size
    theta0 = np.zeros(N)
    theta0[:n] = x0
    on = np.zeros(N, bool)
    off = 0
    for s, f in (free or [(n, True)]):
        on[off:off + s] = f
        off += s
    kw = dict(kw)
    st = pk.LBFGSState(theta0, history_size=kw.pop("history_size", 100))
    dev = st.theta.device
    out = []
    for _ in range(steps):
        pk.lbfgs_begin(st, **kw)
        pts, statuses = [], []
        for _ in range(100000):
            status = st.status()
            if status["done"]:
                break
            x = st.theta.cpu().numpy()
            assert np.array_equal(st.theta32.cpu().numpy(), x.astype(np.float32))
            f, g = fg(x[:n].copy())
            gg = np.zeros(N)
            gg[:n] = g
            gg[~on] = 0.0
            pts.append(x.copy())
            sums = torch.tensor([f, 0, 0, 0, 0, 0, 0, 0], dtype=torch.float64, device=dev)
            pk.lbfgs_advance(st, sums, torch.from_numpy(gg).to(dev))
        out.append({"points": np.array(pts), "status": st.status(), "x": st.theta.cpu().numpy(),
                    "raw": st.state[:8].cpu().numpy()})
    return out


@pytest.fixture(scope="module")
def problems():
    return O.problems()


@pytest.mark.parametrize("name", [
    "rosenbrock_1521", "quadratic_tolerance_grad", "nonconvex_fixed_step", "history_3", "max_eval_in_line_search",
    "persisted_state", "quadratic_directional_derivative", "persisted_state_fixed_step", "fixed_step_lack_of_progress", "frozen_mask", "kink_1d",
    "wiggly_1d_near_lower_end", "wiggly_1d_near_upper_end", "pinn_oracle"])
def test_standalone_matches_torch(problems, name):
    fg, x0, steps, free, kw = problems[name]
    ref = O.run(fg, x0, steps, free, **kw)
    dev = device_run(fg, x0, steps, free, kw)
    n = x0.size
    worst = 0.0
    for k, (r, d) in enumerate(zip(ref, dev)):
        s = d["status"]
        got = (s["evals"], s["n_iter"], s["func_evals"], s["reason"])
        want = (r["evals"], r["n_iter"], r["func_evals"], r["reason"])
        assert got == want, (name, k, got, want)
        assert np.all(d["points"][:, n:] == 0.0)
        scale = max(np.abs(r["points"]).max(), np.abs(r["x"]).max(), 1e-300)
        err = max(np.abs(d["points"][:, :n] - r["points"]).max(), np.abs(d["x"][:n] - r["x"]).max()) / scale
        worst = max(worst, err)
    print("lbfgs point error %-28s %.3e" % (name, worst))
    assert worst <= POINT_RTOL, (name, worst)
    if free:
        x = dev[-1]["x"]
        off = 0
        for s, f in free:
            if not f:
                assert np.array_equal(x[off:off + s], x0[off:off + s])
            off += s


@pytest.mark.parametrize("name", ["rosenbrock_1521", "pinn_oracle"])
def test_standalone_repeats_bit_for_bit(problems, name):
    fg, x0, steps, free, kw = problems[name]
    a = device_run(fg, x0, steps, free, kw)
    b = device_run(fg, x0, steps, free, kw)
    for p, q in zip(a, b):
        assert np.array_equal(p["points"], q["points"]) and np.array_equal(p["raw"], q["raw"])


# ---------------------------------------------------------------------------------------------
# trainer
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def batch(golden_dir):
    g = np.load(os.path.join(golden_dir, "poc_seed0_n4096.npz"))
    n = g["x"].size
    m1 = np.zeros(n); m1[g["i1"]] = 1
    m2 = np.zeros(n); m2[g["i2"]] = 1
    cols = {k: torch.from_numpy(g[k].astype(np.float32)).cuda() for k in "xyzR"}
    cols["mask"] = torch.from_numpy((m1 + 2 * m2).astype(np.uint8)).cuda()
    cols["w"] = np.array([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()])
    cols["n"] = n
    th = np.load(os.path.join(golden_dir, "poc_paper_run_seed0.npz"))["theta_stage1_saved"].astype(np.float64)
    return cols, th


def _trainer(batch, mask=pk.FINE_TUNE_GRAD_MASK):
    b, th = batch
    tr = pk.Trainer("poc", b["n"], th, grad_mask=mask, history_capacity=16)
    tr.set_batch(b["x"], b["y"], b["z"], b["R"], b["mask"], b["w"])
    return tr


LB = {"none": dict(max_iter=6, history_size=4, tolerance_grad=0, tolerance_change=0),
      "strong_wolfe": dict(max_iter=6, history_size=4, tolerance_grad=0, tolerance_change=0, line_search_fn="strong_wolfe")}


@pytest.mark.parametrize("ls", ["none", "strong_wolfe"])
@pytest.mark.parametrize("use_graph", [False, True])
def test_trainer_equals_standalone_fed_by_loss_and_grad_raw(batch, ls, use_graph):
    b, th = batch
    kw = LB[ls]
    tr = _trainer(batch)
    st = pk.LBFGSState(th, history_size=kw["history_size"])
    wd = torch.from_numpy(b["w"]).cuda()
    sums = torch.empty(8, dtype=torch.float64, device="cuda")
    dth = torch.empty(N, dtype=torch.float64, device="cuda")
    E = torch.empty(b["n"], dtype=torch.float32, device="cuda")
    slots = kw["max_iter"] * 5 // 4 + (1 if ls == "strong_wolfe" else 0)
    for call in range(2):  # the second call continues from the persisted state
        s_t, trace = tr.run_lbfgs(use_graph=use_graph, **kw)
        args = {k: v for k, v in kw.items() if k != "history_size"}
        pk.lbfgs_begin(st, **args)
        losses = []
        for _ in range(slots):
            pk.loss_and_grad_raw(0, b["x"], b["y"], b["z"], b["R"], st.theta32, b["mask"], wd,
                                 grad_mask=pk.FINE_TUNE_GRAD_MASK, sums=sums, dtheta=dth, E_out=E)
            losses.append(sums[:3].clone())
            pk.lbfgs_advance(st, sums, dth)
        s_s = st.status()
        assert s_t == s_s, (call, s_t, s_s)
        assert s_t["done"] and s_t["evals"] >= 2
        assert np.array_equal(tr.read()["theta"], st.theta.cpu().numpy())
        assert np.array_equal(trace[:, :3], torch.stack(losses[:s_t["evals"]]).cpu().numpy())
    tr.close()


@pytest.mark.parametrize("ls", ["none", "strong_wolfe"])
def test_graph_equals_plain_launches(batch, ls):
    kw = LB[ls]
    outs = []
    for use_graph in (False, True):
        tr = _trainer(batch)
        res = [tr.run_lbfgs(use_graph=use_graph, **kw) for _ in range(3)]
        outs.append((res, tr.read()["theta"]))
        tr.close()
    (ra, ta), (rb, tb) = outs
    assert np.array_equal(ta, tb)
    for (sa, xa), (sb, xb) in zip(ra, rb):
        assert sa == sb and np.array_equal(xa, xb)


def _step_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, sum(ev.count for ev in prof.key_averages() if "pinn_step_tc_kernel" in ev.key)


def test_graph_runs_no_evaluation_past_the_end(batch):
    tr = _trainer(batch)
    tr.run_lbfgs(**LB["strong_wolfe"])  # warm: the first evaluation of a trainer runs as plain launches
    # terminates early on the loss change, and on the gradient at the first evaluation
    for kw in (dict(max_iter=50, tolerance_change=1e-3, history_size=4, line_search_fn="strong_wolfe"),
               dict(max_iter=50, tolerance_grad=1e3, history_size=4, line_search_fn="strong_wolfe")):
        (s, trace), k = _step_kernels(lambda: tr.run_lbfgs(use_graph=True, **kw))
        assert s["done"] and s["evals"] < 50
        assert k == s["evals"], (kw, k, s)
        (s2, _), k2 = _step_kernels(lambda: tr.run_lbfgs(use_graph=False, **kw))
        assert k2 == 50 * 5 // 4 + 1  # the plain form runs every slot
    tr.close()


def test_adam_state_is_untouched_and_adam_continues(batch):
    tr = _trainer(batch)
    tr.run(3, resample=False)
    r0 = tr.read()
    s, _ = tr.run_lbfgs(**LB["strong_wolfe"])
    r1 = tr.read()
    for k in ("m", "v", "best_theta", "history"):
        assert np.array_equal(r0[k], r1[k]), k
    for k in ("steps", "best_loss", "best_step", "batches"):
        assert r0[k] == r1[k], k
    assert not np.array_equal(r0["theta"], r1["theta"])
    frozen = np.ones(N, bool)
    offs = layout.offsets() + [N]
    for t in range(16):
        if (pk.FINE_TUNE_GRAD_MASK >> t) & 1:
            frozen[offs[t]:offs[t + 1]] = False
    assert np.array_equal(r0["theta"][frozen], r1["theta"][frozen])
    tr.run(2, resample=False)
    r2 = tr.read()
    assert r2["steps"] == 5 and np.all(np.isfinite(r2["theta"])) and not np.array_equal(r2["theta"], r1["theta"])
    # load_state resets the L-BFGS state to a fresh optimizer
    assert tr.read_lbfgs()[0]["n_iter"] > 0
    tr.load_state(r2["theta"])
    s0, _ = tr.read_lbfgs()
    assert s0["n_iter"] == 0 and s0["func_evals"] == 0 and s0["evals"] == 0
    tr.close()


def test_bad_arguments_launch_nothing(batch):
    h = pk.Handle.get(0)
    L = h.L
    st = pk.LBFGSState(np.zeros(N), history_size=3)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    good = pk.trainer.lbfgs_config(history_size=3)
    assert L.pinn_lbfgs_state_bytes(0) == 0
    before = h.launch_count()
    for field, value in (("history_size", 0), ("max_iter", 0), ("line_search", 2), ("lr", -1.0), ("lr", float("nan")),
                         ("tolerance_grad", -1.0)):
        c = pk.trainer.lbfgs_config(history_size=3)
        setattr(c, field, value)
        assert L.pinn_lbfgs_begin(h.h, p(st.state), ctypes.byref(c), p(st.theta), p(st.theta32), None) == -1, field
    assert L.pinn_lbfgs_begin(h.h, None, ctypes.byref(good), p(st.theta), p(st.theta32), None) == -1
    assert L.pinn_lbfgs_begin(h.h, p(st.state), None, p(st.theta), p(st.theta32), None) == -1
    sums = torch.zeros(8, dtype=torch.float64, device="cuda")
    assert L.pinn_lbfgs_advance(h.h, p(st.state), None, p(st.theta), p(st.theta), p(st.theta32), None) == -1
    assert L.pinn_lbfgs_advance(h.h, p(st.state), p(sums), p(st.theta), None, p(st.theta32), None) == -1
    assert h.launch_count() == before
    b, th = batch
    tr = pk.Trainer("poc", b["n"], th)
    assert L.pinn_trainer_run_lbfgs(tr.t, ctypes.byref(good), 0, 0) == -1  # no batch yet
    c = pk.trainer.lbfgs_config(history_size=0)
    assert L.pinn_trainer_run_lbfgs(tr.t, ctypes.byref(c), 1, 0) == -1
    assert h.launch_count() == before
    with pytest.raises(ValueError):
        pk.trainer.lbfgs_config(line_search_fn="backtracking")
    tr.close()


def test_not_supported_with_the_data_parallel_exchange(batch):
    b, th = batch
    h0, h1 = pk.Handle(0), pk.Handle(0)
    try:
        h0.dp_init(0, 2, want_ipc=False)
        h1.dp_init(1, 2, want_ipc=False)
        h0.dp_connect_local([h0, h1])
        h1.dp_connect_local([h0, h1])
        tr = pk.Trainer("poc", 4096, th, handle=h0)
        before = h0.launch_count()
        c = pk.trainer.lbfgs_config()
        assert h0.L.pinn_trainer_run_lbfgs(tr.t, ctypes.byref(c), 1, 0) == -2
        assert h0.launch_count() == before
        tr.close()
    finally:
        h0.dp_shutdown(); h1.dp_shutdown()
        h0.close(); h1.close()


def test_paper_fine_tune_reaches_adam_in_fewer_evaluations(golden_dir):
    """From the paper re-run's stage-1 model, one fixed batch of 100 000 points, E-net free (freezeUnits): L-BFGS with
    strong Wolfe and history 20 reaches a batch Ltot at or below that of 2000 device Adam steps at lr 5e-4, in at most
    400 evaluations (max_eval 399: the line search may take one evaluation past max_eval)."""
    th = np.load(os.path.join(golden_dir, "poc_paper_run_seed0.npz"))["theta_stage1_saved"].astype(np.float64)
    n = 100000
    s = pk.sample(n, seed=2024, batch=0)
    w = s["weights"].cpu().numpy()

    def ltot(theta):
        t32 = torch.from_numpy(np.asarray(theta, np.float32)).cuda()
        sums, _, _ = pk.loss_and_grad_raw(0, s["x"], s["y"], s["z"], s["R"], t32, s["mask"], s["weights"])
        return float(sums[0].item())
    ta = pk.Trainer("poc", n, th, lr=5e-4, grad_mask=pk.FINE_TUNE_GRAD_MASK)
    ta.set_batch(s["x"], s["y"], s["z"], s["R"], s["mask"], w)
    ta.run(2000, resample=False, use_graph=True)
    l_adam = ltot(ta.read()["theta"])
    ta.close()
    tl = pk.Trainer("poc", n, th, grad_mask=pk.FINE_TUNE_GRAD_MASK)
    tl.set_batch(s["x"], s["y"], s["z"], s["R"], s["mask"], w)
    st, trace = tl.run_lbfgs(max_iter=400, max_eval=399, history_size=20, tolerance_grad=0, tolerance_change=0,
                             line_search_fn="strong_wolfe", use_graph=True)
    l_lb = ltot(tl.read()["theta"])
    tl.close()
    print("paper fine-tune, batch Ltot: start %.4e  adam(2000) %.4e  lbfgs(%d evals, %s) %.4e"
          % (ltot(th), l_adam, st["evals"], st["reason_name"], l_lb))
    assert st["evals"] <= 400
    assert l_lb <= l_adam
