"""GPU tests of importance-weighted adaptive batches: the weighted training evaluation (pinn_loss_fwd_bwd_weighted)
against the float64 oracle, the importance draw (pinn_sample_adaptive_importance) against its host restatement, the
unbiasedness of the weighted batch loss over many draws, and the trainer's importance mode against a host loop of the
same calls."""
import ctypes
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import adaptive as ad
from oracle import importance as imp
from oracle import layout
from oracle import ref_autograd as ra

pytestmark = pytest.mark.gpu
OFFS = layout.offsets() + [1521]
TRAINED_LOSS_BAR = 1.5e-4  # the bars of test_gpu_parity.py at the shipped trained weights (its module docstring)
TRAINED_ENET_BAR = 2e-5
AD = dict(pool_factor=4, k=1.0, c=1.0)


def dev():
    return torch.device("cuda:0")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def _np(t):
    return t.cpu().numpy()


@pytest.fixture(scope="module")
def ck(golden_dir):
    return np.load(os.path.join(golden_dir, "checkpoints.npz"))


@pytest.fixture(scope="module")
def init_theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]  # train.py's init rule, seed 12345


_POINTS = {}


def points(variant, n):
    """n float32 points of the reference's sampler, none within 1e-3 of the boundary radius (so the kernel's own set rule
    and the float64 one agree), point 0 in both sets; sets m1, m2 and per-point weights om (float32, some zero)."""
    key = (variant, n)
    if key not in _POINTS:
        g = torch.Generator().manual_seed(1000 + n)
        x, y, z, R, _, _ = ra.sample_box(n + n // 8 + 64, variant, g)
        a = [v.numpy().ravel().astype(np.float32) for v in (x, y, z, R)]
        a[0][0], a[1][0], a[2][0] = 0.0, 15.0, 15.0
        a64 = [v.astype(np.float64) for v in a]
        r1 = np.sqrt((a64[0] - a64[3]) ** 2 + a64[1] ** 2 + a64[2] ** 2)
        r2 = np.sqrt((a64[0] + a64[3]) ** 2 + a64[1] ** 2 + a64[2] ** 2)
        keep = np.flatnonzero((np.abs(r1 - 17.5) > 1e-3) & (np.abs(r2 - 17.5) > 1e-3))[:n]
        assert keep.size == n
        a = [v[keep] for v in a]
        m1, m2 = (r1[keep] >= 17.5).astype(np.float64), (r2[keep] >= 17.5).astype(np.float64)
        om = np.random.default_rng(n).uniform(0.0, 3.0, n).astype(np.float32)
        om[1::11] = 0.0
        om[0] = 1.5
        _POINTS[key] = (a, m1, m2, om)
    return _POINTS[key]


def run_weighted(variant, a, th32, m1, m2, om, dtype, use_mask, grad_mask, weights):
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev())
    mask = t((m1 + 2 * m2).astype(np.uint8)) if use_mask else None
    w = torch.tensor(weights, dtype=torch.float64, device=dev())
    sums, dth, E = pk.loss_and_grad_raw(0 if variant == "poc" else 1, *[t(v.astype(dtype)) for v in a], t(th32), mask, w,
                                        grad_mask, want_E=True, point_weights=t(om))
    torch.cuda.synchronize()
    return _np(sums), _np(dth), _np(E)


_ORACLE = {}


@pytest.mark.parametrize("tune", ["full", "fine_tune"])
@pytest.mark.parametrize("use_mask", [True, False], ids=["mask", "no_mask"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("variant", ["poc", "trainpy"])
@pytest.mark.parametrize("n", [1, 127, 4096, (1 << 18) + 3])
def test_weighted_evaluation_against_the_oracle(n, variant, dtype, use_mask, tune, init_theta, ck):
    a, m1, m2, om = points(variant, n)
    th = init_theta if tune == "full" else ck["ionHsym_fineTune"]
    th32 = th.astype(np.float32)
    gm = 0xFFFF if tune == "full" else pk.FINE_TUNE_GRAD_MASK
    weights = (1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum())
    key = (n, variant, tune)
    if key not in _ORACLE:
        _ORACLE[key] = imp.loss_and_grad(variant, th32.astype(np.float64), *[v.astype(np.float64) for v in a], m1, m2,
                                        *weights, point_weights=om.astype(np.float64))
    ref = _ORACLE[key]
    sums, dth, E = run_weighted(variant, a, th32, m1, m2, om, dtype, use_mask, gm, weights)
    # At the trained (fine-tune) weights psi at the boundary and the residual are cancellations (psi ~ 2e-5 of O(0.1)
    # terms, |res| ~ 1e-3 of its terms), so the float32 loss terms are limited there: the parity bar of Lbc at those
    # weights is TRAINED_LOSS_BAR.  Lpde takes it too: at 1 and 127 points, where no point near a nucleus dominates
    # the sum, it measures 7e-5 (at 4096 and more points, under 1e-5).
    bar = 1e-5 if tune == "full" else TRAINED_LOSS_BAR
    assert abs(sums[1] - ref["Lpde"]) <= bar * abs(ref["Lpde"]), ("Lpde", sums[1], ref["Lpde"])
    assert abs(sums[2] - ref["Lbc"]) <= bar * abs(ref["Lbc"]), ("Lbc", sums[2], ref["Lbc"])
    assert abs(sums[0] - ref["Ltot"]) <= bar * abs(ref["Ltot"]), ("Ltot", sums[0], ref["Ltot"])
    assert abs(sums[3] - ref["sums"]["E"]) <= 1e-5 * abs(ref["sums"]["E"])
    assert rel(E, ref["E"]) < 1e-5
    if tune == "full":
        for i, (nm, _) in enumerate(layout.POC_TENSORS):
            assert rel(dth[OFFS[i]:OFFS[i + 1]], ref["grad"][OFFS[i]:OFFS[i + 1]]) < 1e-5, nm
    else:  # the parity bar of the fine-tune mode (test_gpu_parity.py::test_fine_tune_grad_mask)
        assert np.all(dth[:OFFS[6]] == 0) and np.all(dth[OFFS[12]:] == 0)
        # (one point: the E-net gradient is its seed Ebar = 2 w om cE res psi times dE/dtheta, so it carries the error of
        # the loss terms, 7.5e-5 measured; over many points those errors average out below TRAINED_ENET_BAR)
        bar_e = TRAINED_ENET_BAR if n > 1 else TRAINED_LOSS_BAR
        assert rel(dth[OFFS[6]:OFFS[12]], ref["grad"][OFFS[6]:OFFS[12]]) < bar_e


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("n", [127, 4096, (1 << 18) + 3])
def test_unit_weights_give_the_unweighted_bits(variant, n, init_theta):
    a, m1, m2, _ = points("poc" if variant == 0 else "trainpy", n)
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev())
    cols = [t(v) for v in a]
    mask = t((m1 + 2 * m2).astype(np.uint8))
    th = t(init_theta.astype(np.float32))
    s0, g0, E0 = pk.loss_and_grad_raw(variant, *cols, th, mask, None, want_E=True)
    s1, g1, E1 = pk.loss_and_grad_raw(variant, *cols, th, mask, None, want_E=True,
                                      point_weights=torch.ones(n, dtype=torch.float32, device=dev()))
    assert torch.equal(s0, s1) and torch.equal(g0, g1) and torch.equal(E0, E1)


@pytest.mark.parametrize("variant", [0, 1])
def test_integer_weights_equal_duplicated_points(variant, init_theta):
    n = 20000
    a, m1, m2, _ = points("poc" if variant == 0 else "trainpy", n)
    om = np.random.default_rng(9).integers(0, 4, n)
    om[0] = 1
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev())
    th = t(init_theta.astype(np.float32))
    w = torch.tensor([1.0 / om.sum(), 1.0 / (om * m1).sum(), 1.0 / (om * m2).sum()], dtype=torch.float64, device=dev())
    sa, ga, _ = pk.loss_and_grad_raw(variant, *[t(v) for v in a], th, t((m1 + 2 * m2).astype(np.uint8)), w,
                                     point_weights=t(om.astype(np.float32)))
    rep = lambda v: np.repeat(v, om)
    sb, gb, _ = pk.loss_and_grad_raw(variant, *[t(rep(v)) for v in a], th, t(rep(m1 + 2 * m2).astype(np.uint8)), w)
    sa, ga, sb, gb = _np(sa), _np(ga), _np(sb), _np(gb)
    # two float32 evaluations of one float64 sum, each within the 1e-5 parity bars of it
    for i in range(4):
        assert abs(sa[i] - sb[i]) <= 2e-5 * abs(sb[i]), i
    for i, (nm, _) in enumerate(layout.POC_TENSORS):
        assert rel(ga[OFFS[i]:OFFS[i + 1]], gb[OFFS[i]:OFFS[i + 1]]) < 2e-5, nm


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
@pytest.mark.parametrize("k,c", [(1.0, 1.0), (2.0, 0.1), (1e30, 1.0)])
def test_importance_draw(variant, k, c, ck):
    n, pf, seed, batch = 5000, 4, 77, 9
    N = n * pf
    theta = ck["ionHsym"]
    kw = dict(pool_factor=pf, k=k, c=c, seed=seed, batch=batch)
    a = pk.sample_adaptive(variant, theta, n, **kw)
    b = pk.sample_adaptive(variant, theta, n, importance=True, **kw)
    for key in ("x", "y", "z", "R", "mask", "idx", "counts", "res", "cdf"):
        assert torch.equal(a[key], b[key]), key
    res, cdf, idx = _np(b["res"]), _np(b["cdf"]), _np(b["idx"])
    # omega = float32(T / (N w_idx)), w formed again on the host from the returned residuals (Q summed in another order:
    # within one float32 rounding)
    w = ad.weights(res, k, c)
    want = (cdf[-1] / (N * w[idx])).astype(np.float32)
    got = _np(b["point_weights"])
    ulp = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1 and np.mean(ulp == 0) > 0.99, (ulp.max(), np.mean(ulp == 0))
    assert got.max() <= (1 + np.float32(c)) / np.float32(c) * (1 + 1e-6)
    if k == 1e30:  # uniform fallback
        assert np.all(got == 1.0)
    pm = _np(b["pool"]["mask"])
    c1, c2 = int((pm & 1).sum()), int((pm >> 1 & 1).sum())
    assert _np(b["weights"]).tolist() == imp.importance_loss_weights(n, N, c1, c2).tolist()


def test_weighted_batch_loss_is_unbiased_and_the_plain_one_is_not(ck):
    """Over 256 draws: mean of (batch loss - the pool's own uniform loss_eval) within 3 standard errors of 0 with
    importance weights, for Ltot and Lpde.  Without them the batch loss is a residual-weighted mean.  Its differences
    are so heavy-tailed (a draw that takes a few points of huge residual) that their standard error hides the bias in
    256 draws, so the bias is shown by a sign test instead: the batch exceeds its pool in far more than half the draws
    (3 standard deviations of a fair coin above 1/2)."""
    n, pf = 4096, 4
    th = torch.from_numpy(ck["ionHsym"].astype(np.float32)).to(dev())
    d = {True: [], False: []}
    for b in range(256):
        for imp in (True, False):
            out = pk.sample_adaptive("poc", th, n, seed=123, batch=b, importance=imp, **AD)
            s, _, _ = pk.loss_and_grad_raw(0, out["x"], out["y"], out["z"], out["R"], th, out["mask"], out["weights"],
                                           point_weights=out.get("point_weights"))
            p = out["pool"]
            ref = pk.loss_eval(0, p["x"], p["y"], p["z"], p["R"], th, p["mask"])
            d[imp].append((float(s[0]), float(ref[0]), float(s[1]), float(ref[1])))
    for imp in (True, False):
        v = np.array(d[imp])
        for col, name in ((0, "Ltot"), (2, "Lpde")):
            diff = v[:, col] - v[:, col + 1]
            m, se = diff.mean(), diff.std(ddof=1) / np.sqrt(diff.size)
            print("importance=%s %s: mean over the pools %.6e, mean(batch - pool) %.3e, standard error %.3e, z = %.2f"
                  % (imp, name, v[:, col + 1].mean(), m, se, m / se))
            above = float(np.mean(diff > 0))
            print("    batch above its pool in %.3f of the draws" % above)
            if imp:
                assert abs(m) < 3 * se, name
            else:
                assert above > 0.5 + 3 * 0.5 / np.sqrt(diff.size), name


@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("variant", ["poc", "trainpy"])
def test_trainer_equals_host_loop_bit_for_bit(variant, use_graph, init_theta):
    n, steps, seed = 4096, 20, 17
    box = pk.trainer.BOX_POC if variant == "poc" else pk.trainer.BOX_TRAINPY
    theta0 = pk.init_poc(0) if variant == "poc" else init_theta
    tr = pk.Trainer(variant, n, theta0, seed=seed, lr=8e-3, history_capacity=steps, adaptive=dict(AD, importance=True))
    tr.run(steps, use_graph=use_graph)
    got = tr.read()
    tr.close()
    v = 0 if variant == "poc" else 1
    st = pk.AdamState(theta0, history_capacity=steps, best_mode=1 if v == 0 else 0)
    for t in range(steps):
        out = pk.sample_adaptive(variant, st.theta32, n, seed=seed, batch=t, box=box, importance=True, **AD)
        sums, dth, _ = pk.loss_and_grad_raw(v, out["x"], out["y"], out["z"], out["R"], st.theta32, out["mask"],
                                            out["weights"], want_E=True, point_weights=out["point_weights"])
        pk.adam_step(st, dth, sums, n, lr=8e-3, history_mean_E=(v == 1))
    torch.cuda.synchronize()
    assert np.array_equal(got["theta"], _np(st.theta))
    assert np.array_equal(got["m"], _np(st.m)) and np.array_equal(got["v"], _np(st.v))
    assert np.array_equal(got["best_theta"], _np(st.best_theta))
    assert np.array_equal(got["history"], _np(st.hist)[:steps])


def test_importance_batches_keep_their_weights_between_draws():
    """sc_sampling = 3: the two steps after each importance draw evaluate the same batch with its weights, plain and
    under graph replay alike, and the run differs from the unweighted adaptive one."""
    n, steps = 4096, 9
    res = {}
    for imp, graph in ((True, False), (True, True), (False, True)):
        tr = pk.Trainer("poc", n, pk.init_poc(0), seed=5, lr=8e-3, history_capacity=steps, sc_sampling=3,
                        adaptive=dict(AD, importance=imp))
        tr.run(steps, use_graph=graph)
        res[(imp, graph)] = tr.read()
        tr.close()
    for kk in ("theta", "m", "v", "best_theta", "history"):
        assert np.array_equal(res[(True, False)][kk], res[(True, True)][kk]), kk
    assert not np.array_equal(res[(True, True)]["theta"], res[(False, True)]["theta"])


def test_argument_errors_launch_nothing(init_theta):
    h = pk.Handle.get(0)
    n = 1000
    a, m1, m2, om = points("poc", n)
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev())
    cols = [t(v) for v in a]
    th = t(init_theta.astype(np.float32))
    mask = t((m1 + 2 * m2).astype(np.uint8))
    good = t(om)
    bad = {"length": good[:-1].clone(), "device": good.cpu(), "negative": good.clone().index_fill_(0, t(np.array([3])), -1.0),
           "nan": good.clone().index_fill_(0, t(np.array([5])), float("nan")),
           "inf": good.clone().index_fill_(0, t(np.array([7])), float("inf")), "dtype": good.double()}
    torch.cuda.synchronize()
    for name, w in bad.items():
        before = h.launch_count()
        with pytest.raises(ValueError):
            pk.loss_and_grad_raw(0, *cols, th, mask, None, point_weights=w)
        assert h.launch_count() == before, name
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    sums = torch.empty(8, dtype=torch.float64, device=dev())
    dth = torch.empty(1521, dtype=torch.float64, device=dev())
    before = h.launch_count()
    assert h.L.pinn_loss_fwd_bwd_weighted(h.h, 0, n, *[P(c) for c in cols], 0, P(mask), P(th), None, None, 0xFFFF,
                                          17.5, P(sums), P(dth), None, None) == -1
    assert h.launch_count() == before
    # importance mode needs c > 0
    before = h.launch_count()
    with pytest.raises(pk.PinnError):
        pk.sample_adaptive("poc", init_theta, 512, pool_factor=4, k=1.0, c=0.0, importance=True)
    assert h.launch_count() == before
    tr = pk.Trainer("poc", 512, init_theta, seed=1)
    assert h.L.pinn_trainer_set_importance(tr.t, 1) == -1  # adaptive sampling is off
    tr.set_adaptive(pool_factor=4, k=1.0, c=0.0)
    assert h.L.pinn_trainer_set_importance(tr.t, 1) == -1  # c = 0
    tr.set_adaptive(pool_factor=4, k=1.0, c=1.0, importance=True)
    assert h.L.pinn_trainer_set_importance(tr.t, 0) == 0
    tr.close()
