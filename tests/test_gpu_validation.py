"""GPU tests of the forward-only loss reduction (pinn_loss_eval) and the trainer's held-out validation
(pinn_trainer_set_validation / _validate / _read_validation).

- The per-point values the reduction adds are pinn_fields' bits: its sums equal a float64 sum over pinn_fields' outputs
  within 1e-12, a bar one ulp of any per-point value would miss by five orders.
- Against float64: the parity bars of the training path, and the training path's own sums and set counts.
- No drift at scale: K copies of a block give K times the block's sums, where the training kernel's float32
  accumulators miss their bars (DESIGN.md section 4).
- The trainer with validation on computes every other bit as it did without, and its rows are the stand-alone call."""
import ctypes
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf
from oracle import pointwise as pw
from oracle import validation as va

pytestmark = pytest.mark.gpu
BCUT = 17.5
EINVAL, ENOTSUP = -1, -2
VARIANTS = ["poc", "trainpy"]
VCODE = {"poc": 0, "trainpy": 1}


def dev():
    return torch.device("cuda", torch.cuda.current_device())


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def box_of(variant):
    return pk.trainer.BOX_POC if variant == "poc" else pk.trainer.BOX_TRAINPY


@pytest.fixture(scope="module")
def thetas(golden_dir):
    ck = np.load(os.path.join(golden_dir, "checkpoints.npz"))
    tp = np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]  # train.py's init rule, seed 12345
    return {"init_poc0": pk.init_poc(0), "trainpy_init": tp, "ionHsym": ck["ionHsym"], "ionHsym_fineTune": ck["ionHsym_fineTune"]}


def points(variant, n, seed, f64=False):
    """n sampler points (host) with no point within 1e-5 relative of a boundary radius, so that r >= bcutoff in float64
    and the kernel's ir * bcutoff <= 1 agree; f64: float64 coordinates off the float32 grid."""
    m = 2 * n + 64
    s = pk.sample(m, seed, 0, box=box_of(variant))
    x, y, z, R = [s[k].cpu().numpy() for k in "xyzR"]
    cols = [a.astype(np.float64) for a in (x, y, z, R)]
    if f64:
        rng = np.random.default_rng(seed)
        cols = [a * (1.0 + 1e-9 * rng.standard_normal(m)) for a in cols]
    xd, yd, zd, Rd = cols
    r1 = np.sqrt((xd - Rd) ** 2 + yd ** 2 + zd ** 2)
    r2 = np.sqrt((xd + Rd) ** 2 + yd ** 2 + zd ** 2)
    keep = (np.abs(r1 / BCUT - 1) > 1e-5) & (np.abs(r2 / BCUT - 1) > 1e-5)
    idx = np.nonzero(keep)[0][:n]
    assert idx.size == n
    a = [c[idx] for c in cols] if f64 else [c[idx] for c in (x, y, z, R)]
    return a, (r1[idx] >= BCUT).astype(np.float64), (r2[idx] >= BCUT).astype(np.float64)


def fields64(variant, a, th32):
    f = pk.fields(variant, *[t(c) for c in a], t(th32), want=("psi", "res", "E"))
    return {k: v.cpu().numpy() for k, v in f.items()}


def close(a, b, rtol):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    ok = both_nan | (np.abs(a - b) <= rtol * np.abs(b))
    return bool(ok.all())


# ---------------------------------------------------------------------------------------------------------------------
# 1. exactness against pinn_fields
# ---------------------------------------------------------------------------------------------------------------------
SIZES = [1, 127, 128, 129, 20000, (1 << 18) + 3]


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("weights", ["given", "null"])
@pytest.mark.parametrize("mask", ["given", "null"])
@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_sums_are_a_float64_sum_over_fields(variant, dtype, mask, weights, n, thetas):
    th32 = thetas["ionHsym" if variant == "poc" else "trainpy_init"].astype(np.float32)
    a, m1, m2 = points(variant, n, 1000 + n, f64=dtype == "f64")
    if mask == "given":
        # arbitrary set bits (and the high bits set, which the kernel ignores): the mask is data, read at every byte offset
        bits = np.random.default_rng(n).integers(0, 256, n).astype(np.uint8)
        m1, m2 = (bits & 1).astype(np.float64), ((bits >> 1) & 1).astype(np.float64)
        mk = t(bits)
    else:
        mk = None
    c1, c2 = m1.sum(), m2.sum()
    if weights == "given":
        w = np.array([0.7 / n, 1.3 / max(c1, 1.0), 0.9 / max(c2, 1.0)])
        wt = t(w)
    else:
        with np.errstate(divide="ignore"):
            w = np.array([1.0 / n, 1.0 / c1, 1.0 / c2])
        wt = None
    sums = pk.loss_eval(variant, *[t(c) for c in a], t(th32), mask=mk, weights=wt).cpu().numpy()
    f = fields64(variant, a, th32)
    res, psi, E = [f[k].astype(np.float64) for k in ("res", "psi", "E")]
    r2, p1, p2, sE = (res * res).sum(), (m1 * psi * psi).sum(), (m2 * psi * psi).sum(), E.sum()
    with np.errstate(invalid="ignore"):
        Lpde, Lbc = w[0] * r2, w[1] * p1 + w[2] * p2
    want = [Lpde + Lbc, Lpde, Lbc, sE, r2, p1, p2]
    assert close(np.delete(sums[:7], 3), np.delete(want, 3), 1e-12), (sums[:7], want)
    assert abs(sums[3] - sE) <= 1e-12 * np.abs(E).sum()   # (E may change sign: relative to the sum of |E|)
    assert sums[7] == float(f["E"][n - 1])
    if weights == "null" and (c1 == 0 or c2 == 0):
        assert np.isnan(sums[2])


# ---------------------------------------------------------------------------------------------------------------------
# 2. against float64 and the training path
# ---------------------------------------------------------------------------------------------------------------------
CASES = [("poc", "init_poc0"), ("trainpy", "trainpy_init"), ("poc", "trainpy_init"), ("poc", "ionHsym"),
         ("poc", "ionHsym_fineTune")]


@pytest.mark.parametrize("variant, which", CASES)
def test_against_float64_and_the_training_path(variant, which, thetas):
    """1e-5 on Ltot, Lpde and Lbc.  At the trained checkpoints Lbc is ~1e-9: psi at r >= 17.5 is the small difference of
    gate N and the LCAO part, and float32 psi there carries relative errors of ~1e-4 in pinn_fields and in the training
    kernel alike (this reduction adds pinn_fields' own bits, test above).  Lbc then meets the first-order bound of those
    per-point errors instead, sum over the sets of w 2 |psi| C u M_psi (oracle/pointwise.py), which is printed."""
    th32 = thetas[which].astype(np.float32)
    n = 20000
    a, m1, m2 = points(variant, n, 7)
    cols = [t(c) for c in a]
    mk = t((m1 + 2 * m2).astype(np.uint8))
    a64 = [c.astype(np.float64) for c in a]
    ref = cf.loss_and_grad(variant, th32.astype(np.float64), *a64, m1, m2)
    d = pw.C_KERNEL * pw.U * pw.magnitudes(variant, th32.astype(np.float64), *a64)["psi"]
    ap = np.abs(ref["psi"])
    lbc_bound = (2 * ap * d + d * d) @ (m1 / m1.sum() + m2 / m2.sum())
    for mask in (mk, None):   # the sets from the mask bytes, and by the rule r >= bcutoff
        ev = pk.loss_eval(variant, *cols, t(th32), mask=mask).cpu().numpy()
        for k, key in enumerate(("Ltot", "Lpde")):
            assert abs(ev[k] - ref[key]) <= 1e-5 * abs(ref[key]), (key, ev[k], ref[key])
        err = abs(ev[2] - ref["Lbc"])
        print("\n%s %s: Lbc %.6e oracle %.6e, error %.2e relative, per-point bound %.2e relative"
              % (variant, which, ev[2], ref["Lbc"], err / ref["Lbc"], lbc_bound / ref["Lbc"]))
        assert err <= max(1e-5 * abs(ref["Lbc"]), lbc_bound)
        if which.startswith("init") or which == "trainpy_init":
            assert err <= 1e-5 * abs(ref["Lbc"])
        tr, _, _ = pk.loss_and_grad_raw(VCODE[variant], *cols, t(th32), mask, None, want_E=True)
        tr = tr.cpu().numpy()
        for k in range(7):
            assert abs(ev[k] - tr[k]) <= 1e-5 * abs(tr[k]), (k, ev[k], tr[k])
        assert ev[7] == tr[7]
        # weights NULL: the counted sets are the host's, and the training path's, exactly - its composed loss is the same
        # bits as with the explicit weights {1/n, 1/|set1|, 1/|set2|} of the host's counts
        w = t(np.array([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()]))
        ev_w = pk.loss_eval(variant, *cols, t(th32), mask=mask, weights=w).cpu().numpy()
        tr_w, _, _ = pk.loss_and_grad_raw(VCODE[variant], *cols, t(th32), mask, w)
        assert np.array_equal(ev, ev_w)
        assert np.array_equal(tr[:3], tr_w.cpu().numpy()[:3])


# ---------------------------------------------------------------------------------------------------------------------
# 3. no drift at scale
# ---------------------------------------------------------------------------------------------------------------------
NB = (1 << 16) + 37


@pytest.mark.parametrize("variant, which", [("poc", "init_poc0"), ("poc", "ionHsym"), ("trainpy", "trainpy_init")])
def test_no_drift_over_copies_of_a_block(variant, which, thetas):
    """K copies of a block B (every copy starts at another offset within a super-tile) give K times B's sums.  Bar: a
    float64 sum of m terms in any order is within (m' - 1) u sum|terms| of the exact sum, m' the longest chain of
    additions; here m' <= tiles per lane (K * NB / 128 / 148 < 3600) + 5 shuffle levels + 2 group levels + 148 rows, so
    both sides are within 4e-13 sum|terms|.  1e-11 leaves a factor of 25."""
    th32 = thetas[which].astype(np.float32)
    a, m1, m2 = points(variant, NB, 11)
    cols = [t(c) for c in a]
    mk = t((m1 + 2 * m2).astype(np.uint8))
    one = t(np.ones(3))
    blk = pk.loss_eval(variant, *cols, t(th32), mask=mk, weights=one).cpu().numpy()
    absE = np.abs(fields64(variant, a, th32)["E"].astype(np.float64)).sum()
    scale = np.array([blk[0], blk[1], blk[2], absE, blk[4], blk[5], blk[6]])
    for K in (64, 1024):
        big = pk.loss_eval(variant, *[c.repeat(K) for c in cols], t(th32), mask=mk.repeat(K), weights=one).cpu().numpy()
        err = np.abs(big[:7] - K * blk[:7]) / (K * scale)
        print("\n%s %s K=%d n=%d: worst relative drift %.2e" % (variant, which, K, K * NB, err.max()))
        assert err.max() <= 1e-11, err
        assert big[7] == blk[7]
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# 4. determinism, capture, empty sets, argument errors
# ---------------------------------------------------------------------------------------------------------------------
def test_repeat_calls_and_a_captured_graph_give_the_same_bits(thetas):
    th = t(thetas["ionHsym"].astype(np.float32))
    a, m1, m2 = points("poc", (1 << 18) + 3, 5)
    cols = [t(c) for c in a]
    mk = t((m1 + 2 * m2).astype(np.uint8))
    first = pk.loss_eval("poc", *cols, th, mask=mk)
    for _ in range(3):
        assert torch.equal(pk.loss_eval("poc", *cols, th, mask=mk), first)
    s = torch.cuda.Stream()
    out = torch.full((8,), -1.0, dtype=torch.float64, device=dev())
    with torch.cuda.stream(s):
        pk.loss_eval("poc", *cols, th, mask=mk, sums=out)   # one plain call on the stream first
    s.synchronize()
    assert torch.equal(out, first)
    out.fill_(-1.0)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        pk.loss_eval("poc", *cols, th, mask=mk, sums=out)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, first)


def test_empty_boundary_set_gives_nan_lbc(thetas):
    n = 1000
    rng = np.random.default_rng(3)
    a = [rng.uniform(-2, 2, n).astype(np.float32) for _ in range(3)] + [rng.uniform(0.5, 2, n).astype(np.float32)]
    s = pk.loss_eval("poc", *[t(c) for c in a], t(thetas["ionHsym"].astype(np.float32))).cpu().numpy()
    assert np.isnan(s[0]) and np.isnan(s[2]) and np.isfinite(s[1]) and s[5] == 0.0 and s[6] == 0.0


def test_argument_errors_launch_nothing(thetas):
    h = pk.Handle.get(torch.cuda.current_device())
    n = 256
    a, _, _ = points("poc", n, 2)
    cols = [t(c) for c in a]
    th = t(thetas["ionHsym"].astype(np.float32))
    out = torch.empty(8, dtype=torch.float64, device=dev())
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    good = dict(variant=0, n=n, x=P(cols[0]), y=P(cols[1]), z=P(cols[2]), R=P(cols[3]), dt=0, theta=P(th), sums=P(out))

    def call(**kw):
        c = dict(good, **kw)
        return h.L.pinn_loss_eval(h.h, c["variant"], c["n"], c["x"], c["y"], c["z"], c["R"], c["dt"], None, c["theta"],
                                  None, BCUT, c["sums"], st)
    assert call() == 0
    torch.cuda.synchronize()
    before = h.launch_count()
    for bad in (dict(variant=7), dict(n=0), dict(n=-5), dict(x=None), dict(R=None), dict(dt=3), dict(theta=None),
                dict(sums=None)):
        assert call(**bad) == EINVAL, bad
    assert h.L.pinn_loss_eval(None, 0, n, good["x"], good["y"], good["z"], good["R"], 0, None, good["theta"], None, BCUT,
                              good["sums"], st) == EINVAL
    assert h.launch_count() == before
    with pytest.raises(ValueError):
        pk.loss_eval("poc", cols[0], cols[1], cols[2], cols[3].double(), th)


# ---------------------------------------------------------------------------------------------------------------------
# 5. the trainer with validation on changes nothing else
# ---------------------------------------------------------------------------------------------------------------------
VAL = dict(n=5000, seed=99, every=4)


def trainer_run(th0, adaptive, use_graph, validation, steps=(3, 9, 6)):
    tr = pk.Trainer("poc", 4096, th0, seed=5, sc_sampling=3, freeze_after=11, history_capacity=sum(steps), adaptive=adaptive,
                    validation=validation)
    if validation:
        tr.validate()
    for k in steps:
        tr.run(k, use_graph=use_graph)
    r = tr.read()
    v = tr.read_validation() if validation else None
    tr.close()
    return r, v


@pytest.mark.parametrize("use_graph", [False, True], ids=["plain", "graph"])
@pytest.mark.parametrize("adaptive", [None, dict(pool_factor=4, k=1.0, c=1.0)], ids=["uniform", "adaptive"])
def test_validation_changes_nothing_else(adaptive, use_graph, thetas):
    th0 = thetas["init_poc0"]
    base, _ = trainer_run(th0, adaptive, use_graph, None)
    r, v = trainer_run(th0, adaptive, use_graph, VAL)
    for k in ("theta", "m", "v", "best_theta", "history"):
        assert np.array_equal(r[k], base[k]), k
    for k in ("steps", "best_loss", "best_step", "batches"):
        assert r[k] == base[k], k
    # rows: the step-0 call and every 4th step of 18
    assert v["rows"][:, 0].tolist() == [0, 4, 8, 12, 16]
    if use_graph:  # graph replays and plain launches evaluate the same bits
        _, v_plain = trainer_run(th0, adaptive, False, VAL)
        assert np.array_equal(v["rows"], v_plain["rows"])
        assert np.array_equal(v["best_val_theta"], v_plain["best_val_theta"])


# ---------------------------------------------------------------------------------------------------------------------
# 6. rows are the stand-alone call; the record is the oracle's rule; validate after L-BFGS; load_state; the exchange
# ---------------------------------------------------------------------------------------------------------------------
def standalone(variant, theta64, n_val, seed, box):
    s = pk.sample(n_val, seed, 0, box=box)
    return pk.loss_eval(variant, *[s[k] for k in "xyzR"], t(theta64.astype(np.float32)), mask=s["mask"]).cpu().numpy()


@pytest.mark.parametrize("use_graph", [False, True], ids=["plain", "graph"])
def test_rows_are_the_standalone_call(use_graph, thetas):
    every, n_val, seed = 5, 20000, 31
    box = pk.trainer.BOX_POC
    tr = pk.Trainer("poc", 4096, thetas["init_poc0"], seed=3, lr=2e-2, validation=dict(n=n_val, seed=seed, every=every, capacity=8))
    tr.validate()
    thetas_at = [tr.read()["theta"]]
    for _ in range(6):
        tr.run(every, use_graph=use_graph)
        thetas_at.append(tr.read()["theta"])
    v = tr.read_validation()
    assert v["evaluations"] == 7 and v["rows"].shape == (7, 4)
    for k, th in enumerate(thetas_at):
        want = standalone("poc", th, n_val, seed, box)
        assert v["rows"][k, 0] == every * k
        assert np.array_equal(v["rows"][k, 1:], want[:3]), k
    best, step, idx = va.best_record(v["rows"][:, 1], v["rows"][:, 0])
    assert v["best_val_loss"] == best and v["best_val_step"] == step
    assert np.array_equal(v["best_val_theta"], thetas_at[idx])
    # validate() after L-BFGS: the stand-alone call at the L-BFGS iterate, at the Adam step count
    tr.run_lbfgs(max_iter=4, history_size=5, use_graph=use_graph)
    tr.validate()
    th = tr.read()["theta"]
    v = tr.read_validation()
    assert v["evaluations"] == 8
    assert v["rows"][7, 0] == 30 and np.array_equal(v["rows"][7, 1:], standalone("poc", th, n_val, seed, box)[:3])
    # past the capacity evaluations are counted, not stored
    tr.run(every, use_graph=use_graph)
    v = tr.read_validation()
    assert v["evaluations"] == 9 and v["rows"].shape == (8, 4)
    # load_state restarts the rows and the record; the schedule counts from the resume
    th_loaded = tr.read()["theta"]
    tr.load_state(th_loaded, step=1000)
    v = tr.read_validation()
    assert v["evaluations"] == 0 and v["best_val_loss"] == np.inf and v["best_val_step"] == -1
    assert np.array_equal(v["best_val_theta"], th_loaded)
    tr.run(2 * every + 1, use_graph=use_graph)
    v = tr.read_validation()
    _, rows = va.schedule(every, [("load", 1000), ("run", 2 * every + 1)])
    assert v["rows"][:, 0].tolist() == rows.tolist() == [1005, 1010]
    # every = 0 turns it off
    tr.set_validation(0, 0, 0)
    with pytest.raises(pk.PinnError):
        tr.validate()
    tr.close()


def test_train_drivers_return_validation_only_when_asked(thetas):
    th = thetas["init_poc0"]
    prm = {"n_train": 4096, "epochs": 20}
    a = pk.train_poc(th, prm, seed=1)
    b = pk.train_poc(th, prm, seed=1, validation=dict(n=4096, seed=7, every=5))
    assert "validation" not in a[2] and b[2]["validation"]["rows"][:, 0].tolist() == [0, 5, 10, 15, 20]
    assert np.array_equal(a[0], b[0]) and all(np.array_equal(a[2][k], b[2][k]) for k in a[2])
    _, ia = pk.train_trainpy(n=4096, epochs=10)
    _, ib = pk.train_trainpy(n=4096, epochs=10, validation=dict(n=4096, seed=7, every=5))
    assert "validation" not in ia and ib["validation"]["rows"][:, 0].tolist() == [0, 5, 10]
    assert all(np.array_equal(ia[k], ib[k]) for k in ia)
    with pytest.raises(TypeError):   # the held-out seed has no default
        pk.Trainer("poc", 4096, th, validation=dict(n=4096, every=5))


def test_argument_errors_and_the_data_parallel_exchange(thetas):
    th = thetas["init_poc0"]
    tr = pk.Trainer("poc", 4096, th)
    L = tr.h.L
    assert L.pinn_trainer_set_validation(tr.t, 100, 1, -1, 10) == EINVAL
    assert L.pinn_trainer_set_validation(tr.t, 0, 1, 5, 10) == EINVAL
    assert L.pinn_trainer_set_validation(tr.t, 100, 1, 5, -1) == EINVAL
    assert L.pinn_trainer_validate(tr.t) == EINVAL
    assert L.pinn_trainer_read_validation(tr.t, None, 0, None, None) == EINVAL
    tr.close()
    h0, h1 = pk.Handle(0), pk.Handle(0)
    try:
        h0.dp_init(0, 2, want_ipc=False)
        h1.dp_init(1, 2, want_ipc=False)
        h0.dp_connect_local([h0, h1])
        h1.dp_connect_local([h0, h1])
        tr = pk.Trainer("poc", 4096, th, handle=h0)
        assert h0.L.pinn_trainer_set_validation(tr.t, 4096, 7, 5, 10) == ENOTSUP
        tr.close()
        # validation set while the exchange is off, then the exchange back on: run refuses, launching nothing
        h0.dp_enable(False)
        tr = pk.Trainer("poc", 4096, th, handle=h0, validation=dict(n=4096, seed=7, every=5))
        h0.dp_enable(True)
        before = h0.launch_count()
        assert h0.L.pinn_trainer_run(tr.t, 3, 1, 0) == ENOTSUP
        assert h0.L.pinn_trainer_validate(tr.t) == ENOTSUP
        assert h0.launch_count() == before
        tr.close()
    finally:
        h0.dp_shutdown(); h1.dp_shutdown()
        h0.close(); h1.close()
