"""GPU tests of residual-adaptive collocation (pinn_sample_adaptive, pinn_trainer_set_adaptive) against the numpy
restatement in oracle/adaptive.py: the pool is the uniform sampler's stream, its residual the inference kernel's, the
selection exact, the whole draw deterministic and graph-capturable, and the trainer's adaptive batches those of the
stand-alone call."""
import ctypes
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import adaptive as ad
from oracle import layout
from oracle import philox as ph

pytestmark = pytest.mark.gpu
AD = dict(pool_factor=4, k=1.0, c=1.0)


@pytest.fixture(scope="module")
def thetas(golden_dir):
    ck = np.load(os.path.join(golden_dir, "checkpoints.npz"))
    tp = np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]  # train.py's init rule, seed 12345
    # bo near the float32 maximum: q N overflows near the nuclei and stays finite far from them, so the residual is
    # non-finite on part of every pool
    huge = ck["ionHsym"].astype(np.float32)
    huge[layout.offsets()[5]] = 3.0e38
    return {"trained": ck["ionHsym"], "init": pk.init_poc(0), "trainpy_init": tp, "huge_bo": huge}


def _np(t):
    return t.cpu().numpy()


class _DevCol:
    """A device column of the trainer (pinn_trainer_batch) as a torch tensor, without a copy"""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3,
                                         "strides": None}


def _trainer_batch(tr, n):
    p = [ctypes.c_void_p() for _ in range(5)]
    tr.h.check(tr.h.L.pinn_trainer_batch(tr.t, *[ctypes.byref(q) for q in p]), "pinn_trainer_batch")
    cols = [torch.as_tensor(_DevCol(q.value, n, "<f4"), device="cuda").clone() for q in p[:4]]
    cols.append(torch.as_tensor(_DevCol(p[4].value, n, "|u1"), device="cuda").clone())
    return [_np(c) for c in cols]


# (n, pool_factor, k, c) beyond the plain draw: one output; a pool equal to n; 513 scan blocks (three rounds of the
# offset fold) and the grid-stride loop of the selection; non-integer k; c = 0; k = 1e30, where |res|^k is 0 or inf and
# the draw falls back to uniform weights; and residuals that are not finite on part of the pool
DRAWS = {"": (5000, 4, 1.0, 1.0), "n1": (1, 4, 1.0, 1.0), "pool_eq_n": (4097, 1, 1.0, 1.0),
         "fold3": ((1 << 19) + 3, 4, 1.0, 1.0), "k0.5": (5000, 4, 0.5, 1.0), "k1.7": (5000, 4, 1.7, 1.0),
         "c0": (5000, 4, 1.0, 0.0), "k1e30": (5000, 4, 1e30, 1.0), "nonfinite": (5000, 4, 1.0, 1.0)}
DRAW_CASES = [pytest.param(variant, which, case, id="-".join([variant, which] + ([case] if case else [])))
              for case in DRAWS
              for which in {"k1e30": ["trained", "init", "trainpy_init", "huge_bo"], "nonfinite": ["trained"]}.get(case, ["trained", "init"])
              for variant in ["poc", "trainpy"]]


@pytest.mark.parametrize("variant, which, case", DRAW_CASES)
def test_draw_against_the_oracle(variant, which, case, thetas):
    n, pf, k, c = DRAWS[case]
    seed, batch = 77, 9
    box = pk.trainer.BOX_POC if variant == "poc" else pk.trainer.BOX_TRAINPY
    theta = thetas["huge_bo" if case == "nonfinite" else which]  # (huge_bo at k = 1e30: finite |res| > 1, Q = inf)
    out = pk.sample_adaptive(variant, theta, n, pool_factor=pf, k=k, c=c, seed=seed, batch=batch, box=box)
    N = pf * n
    # the pool is the uniform sampler's batch `batch` of N points, bit for bit
    x, y, z, R, mask, _ = ph.sample_batch(N, seed, batch, box=box)
    pool = {kk: _np(v) for kk, v in out["pool"].items()}
    for kk, want in zip("xyzR", (x, y, z, R)):
        assert np.array_equal(pool[kk].view(np.uint32), want.view(np.uint32)), kk
    assert np.array_equal(pool["mask"], mask)
    # its residual is the one pinn_fields gives at the same points and parameters
    f = pk.fields(variant, *[out["pool"][kk] for kk in "xyzR"], torch.from_numpy(theta.astype(np.float32)).cuda(),
                  want=("res",))
    res = _np(out["res"])
    assert np.array_equal(res.view(np.uint32), _np(f["res"]).view(np.uint32))
    # cdf: the prefix sum of the oracle weights of the device's residuals; never decreasing
    cdf = _np(out["cdf"])
    want_cdf = np.cumsum(ad.weights(res, k, c))
    assert np.all(np.abs(cdf - want_cdf) <= 1e-12 * want_cdf)
    assert np.all(np.diff(cdf) >= 0.0)
    r = np.abs(res.astype(np.float64))
    if case == "k1e30":  # Q = 0 when every finite |res| < 1, inf when one exceeds 1: uniform either way
        rmax = r[np.isfinite(r)].max()
        print("k = 1e30, %s %s: max|res| %.3g -> Q = %s" % (which, variant, rmax, "inf" if rmax > 1 else "0"))
        assert rmax != 1.0 and (rmax > 1.0) == (which == "huge_bo")
        assert np.array_equal(cdf, np.arange(1, N + 1, dtype=np.float64))
    if case == "nonfinite":  # the weight of a non-finite residual is c alone
        fin = np.isfinite(res)
        print("non-finite residuals: %d of %d" % ((~fin).sum(), N))
        assert fin.any() and not fin.all()
        step = np.diff(cdf, prepend=0.0)[~fin]
        assert np.all(np.abs(step - c) <= 4 * np.spacing(cdf[~fin]))
    # selection: exactly the oracle's over the device's own cdf
    idx = _np(out["idx"])
    assert np.array_equal(idx, ad.select(cdf, n, ad.u0(N, seed, batch)))
    for kk in "xyzR":
        assert np.array_equal(_np(out[kk]).view(np.uint32), pool[kk][idx].view(np.uint32)), kk
    m = _np(out["mask"])
    assert np.array_equal(m, pool["mask"][idx])
    c1, c2 = int((m & 1).sum()), int((m >> 1 & 1).sum())
    assert _np(out["counts"]).tolist() == [c1, c2]
    with np.errstate(divide="ignore"):  # a set can be empty at n = 1: its weight is inf
        assert _np(out["weights"]).tolist() == (1.0 / np.array([n, c1, c2], np.float64)).tolist()


def check_counts(thetas, n, pf, k, c):
    out = pk.sample_adaptive("poc", thetas["trained"], n, pool_factor=pf, k=k, c=c, seed=3, batch=1)
    cdf = _np(out["cdf"])
    P = np.diff(cdf, prepend=0.0) / cdf[-1]
    cnt = np.bincount(_np(out["idx"]), minlength=cdf.size)
    lo, hi = ad.count_bounds(P, n, slack=1e-9)
    assert np.all(cnt >= lo) and np.all(cnt <= hi)

    def near(d):
        x, y, z, R = [d[kk] if isinstance(d[kk], np.ndarray) else _np(d[kk]) for kk in "xyzR"]
        r1 = np.sqrt((x - R) ** 2 + y ** 2 + z ** 2)
        r2 = np.sqrt((x + R) ** 2 + y ** 2 + z ** 2)
        return float(np.mean(np.minimum(r1, r2) < 4.0))

    print("share within 4 bohr of a nucleus (trained weights, n=%d, k=%g, c=%g): batch %.4f, pool %.4f"
          % (n, k, c, near(out), near(out["pool"])))


def test_counts_within_floor_and_ceil_at_2_18(thetas):
    check_counts(thetas, 1 << 18, 4, 1.0, 1.0)


@pytest.mark.parametrize("case", [c for c in DRAWS if c not in ("", "k1e30", "nonfinite")])
def test_counts_within_floor_and_ceil_of_other_draws(case, thetas):
    """The count bounds at the draws of DRAWS whose weights are not uniform."""
    check_counts(thetas, *DRAWS[case])


def test_two_calls_and_a_graph_replay_give_the_same_bits(thetas):
    n, kw = 20000, dict(pool_factor=4, k=2.0, c=0.5, seed=5, batch=4)
    keys = ("x", "y", "z", "R", "mask", "idx", "counts", "weights", "res", "cdf")
    snap = lambda o: {kk: o[kk].clone() for kk in keys}
    th = torch.from_numpy(thetas["trained"].astype(np.float32)).cuda()  # no host copy inside the capture below
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        a = snap(pk.sample_adaptive("poc", th, n, **kw))
        b = snap(pk.sample_adaptive("poc", th, n, **kw))
    st.synchronize()
    for kk in keys:
        assert torch.equal(a[kk], b[kk]), kk
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        cap = pk.sample_adaptive("poc", th, n, **kw)
    g.replay()
    torch.cuda.synchronize()
    for kk in keys:
        assert torch.equal(cap[kk], a[kk]), kk


def test_trainer_batch_is_the_stand_alone_draw_at_the_previous_parameters(thetas):
    n, seed = 4096, 31
    tr = pk.Trainer("poc", n, thetas["init"], seed=seed, lr=8e-3, history_capacity=8, adaptive=AD)
    for step in range(3):
        before = tr.read()["theta"]
        tr.run(1)
        tr.read()  # the trainer's stream is done with the step
        got = _trainer_batch(tr, n)
        want = pk.sample_adaptive("poc", before.astype(np.float32), n, seed=seed, batch=step, **AD)
        for kk, g in zip("xyzR", got[:4]):
            assert np.array_equal(g.view(np.uint32), _np(want[kk]).view(np.uint32)), (step, kk)
        assert np.array_equal(got[4], _np(want["mask"])), step
    assert tr.read()["batches"] == 3
    tr.close()


def test_trainer_graph_and_plain_launches_agree():
    n, steps = 4096, 12
    res = {}
    for graph in (True, False):
        tr = pk.Trainer("poc", n, pk.init_poc(0), seed=8, lr=8e-3, history_capacity=steps, sc_sampling=2, adaptive=AD)
        h0 = tr.h.launch_count()
        tr.run(steps, use_graph=graph)
        launched = tr.h.launch_count() - h0
        res[graph] = tr.read()
        tr.close()
        assert launched == 2 * steps + 6 * (steps // 2)  # the step's two launches, six more per adaptive draw
    for kk in ("theta", "m", "v", "best_theta", "history"):
        assert np.array_equal(res[True][kk], res[False][kk]), kk


def test_train_poc_adaptive_is_finite_and_reproducible():
    pr = {"n_train": 4096, "epochs": 50}
    runs = [pk.train_poc(pk.init_poc(0), params=pr, seed=2, adaptive=AD) for _ in range(2)]
    last, _, loss = runs[0]
    for kk in ("Ltot", "Lpde", "Lbc", "Energy"):
        assert loss[kk].shape == (50, 1) and np.all(np.isfinite(loss[kk]))
        assert np.array_equal(loss[kk], runs[1][2][kk])
    assert np.array_equal(last, runs[1][0])


def test_adaptive_turned_off_again_is_a_uniform_trainer(thetas):
    n, steps = 4096, 10
    out = []
    for toggle in (False, True):
        tr = pk.Trainer("poc", n, thetas["init"], seed=6, lr=8e-3, history_capacity=steps)
        if toggle:
            tr.set_adaptive(**AD)
            tr.set_adaptive(pool_factor=0)
        tr.run(steps, use_graph=True)
        out.append(tr.read())
        tr.close()
    for kk in ("theta", "best_theta", "history"):
        assert np.array_equal(out[0][kk], out[1][kk]), kk


def test_bad_arguments_launch_nothing(thetas):
    h = pk.Handle.get(0)
    n, N = 1000, 4000
    f = lambda m, dt=torch.float32: torch.empty(m, dtype=dt, device="cuda")
    th = torch.from_numpy(thetas["init"].astype(np.float32)).cuda()
    bufs = dict(px=f(N), py=f(N), pz=f(N), pR=f(N), pm=f(N, torch.uint8), res=f(N), cdf=f(N, torch.float64), x=f(n),
                y=f(n), z=f(n), R=f(n), m=f(n, torch.uint8), idx=f(n, torch.int64), counts=f(2, torch.int64),
                w=f(3, torch.float64))
    box = (ctypes.c_float * 8)(*pk.trainer.BOX_POC)
    P = lambda t: ctypes.c_void_p(t.data_ptr())

    def call(variant=0, n_=n, N_=N, k=1.0, c=1.0, drop=None):
        ptr = {kk: (None if kk == drop else P(v)) for kk, v in bufs.items()}
        return h.L.pinn_sample_adaptive(h.h, variant, None if drop == "theta" else P(th), n_, N_, 0, 0,
                                        None if drop == "box" else box, 0.005, 17.5, k, c,
                                        *[ptr[kk] for kk in ("px", "py", "pz", "pR", "pm", "res", "cdf", "x", "y", "z", "R",
                                                             "m", "idx", "counts", "w")], None)

    assert call() == 0  # the valid call, for contrast
    torch.cuda.synchronize()
    cases = [dict(n_=0), dict(n_=-5), dict(N_=n - 1), dict(k=-1.0), dict(k=float("nan")), dict(k=float("inf")),
             dict(c=-0.5), dict(c=float("inf")), dict(variant=7), dict(drop="theta"), dict(drop="box")]
    cases += [dict(drop=kk) for kk in bufs if kk != "idx"]
    for kw in cases:
        before = h.launch_count()
        assert call(**kw) == -1, kw
        assert h.launch_count() == before, kw
    assert call(drop="idx") == 0  # idx is optional
    tr = pk.Trainer("poc", 512, thetas["init"], seed=1)
    for args in ((-1, 1.0, 1.0), (4, float("nan"), 1.0), (4, 1.0, -1.0)):
        assert h.L.pinn_trainer_set_adaptive(tr.t, *args) == -1, args
    tr.close()
    torch.cuda.synchronize()
