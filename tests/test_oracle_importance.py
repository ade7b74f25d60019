"""Importance-weighted adaptive batches on the CPU: the weighted closed-form loss and gradient against nested autograd,
integer weights against duplicated points, and the unbiasedness of systematic resampling with omega = 1 / (N P_i) -
the exact expectation over u0 of the counts, and through it of the weighted loss and gradient."""
import os

import numpy as np
import pytest
import torch

from oracle import adaptive as ad
from oracle import closed_form as cf
from oracle import importance as imp


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max()


def _points(golden_dir, n, seed=0):
    g = np.load(os.path.join(golden_dir, "poc_seed0_n4096.npz"))
    rng = np.random.default_rng(seed)
    sel = rng.choice(g["x"].size, n, replace=False)
    m1 = np.zeros(g["x"].size); m1[g["i1"]] = 1
    m2 = np.zeros(g["x"].size); m2[g["i2"]] = 1
    return [g[k][sel].astype(np.float64) for k in "xyzR"], m1[sel], m2[sel]


def _theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"].astype(np.float64)


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
def test_weighted_closed_form_matches_nested_autograd(golden_dir, variant):
    (x, y, z, R), m1, m2 = _points(golden_dir, 48)
    theta = _theta(golden_dir)
    rng = np.random.default_rng(1)
    om = rng.uniform(0.0, 3.0, x.size)
    om[::7] = 0.0
    w = (1.0 / 40, 1.0 / 11, 1.0 / 13)
    ref = imp.loss_and_grad(variant, theta, x, y, z, R, m1, m2, *w, point_weights=om)
    T = lambda a: torch.tensor(a, dtype=torch.float64)
    col = lambda a: T(a).reshape(-1, 1)
    Ltot, Lpde, Lbc, sE, grad = imp.autograd_loss_and_grad(variant, T(theta), col(x), col(y), col(z), col(R), T(m1), T(m2),
                                                          T(om), *w)
    assert abs(ref["Ltot"] - Ltot.item()) <= 1e-12 * abs(Ltot.item())
    assert abs(ref["Lpde"] - Lpde.item()) <= 1e-12 * abs(Lpde.item())
    assert abs(ref["Lbc"] - Lbc.item()) <= 1e-12 * abs(Lbc.item())
    assert abs(ref["sums"]["E"] - sE.item()) <= 1e-12 * abs(sE.item())
    assert _rel(ref["grad"], grad.numpy()) < 1e-12


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
def test_unit_weights_are_the_unweighted_loss(golden_dir, variant):
    (x, y, z, R), m1, m2 = _points(golden_dir, 64, seed=3)
    theta = _theta(golden_dir)
    a = cf.loss_and_grad(variant, theta, x, y, z, R, m1, m2)
    b = imp.loss_and_grad(variant, theta, x, y, z, R, m1, m2, point_weights=np.ones(x.size))
    assert a["Ltot"] == b["Ltot"] and np.array_equal(a["grad"], b["grad"])


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
def test_integer_weights_equal_duplicated_points(golden_dir, variant):
    (x, y, z, R), m1, m2 = _points(golden_dir, 64, seed=4)
    theta = _theta(golden_dir)
    om = np.random.default_rng(2).integers(0, 4, x.size)
    w = (1.0 / 100, 1.0 / 30, 1.0 / 31)
    a = imp.loss_and_grad(variant, theta, x, y, z, R, m1, m2, *w, point_weights=om)
    rep = lambda v: np.repeat(v, om)
    b = cf.loss_and_grad(variant, theta, rep(x), rep(y), rep(z), rep(R), rep(m1), rep(m2), *w)
    assert abs(a["Ltot"] - b["Ltot"]) <= 1e-13 * b["Ltot"]
    assert _rel(a["grad"], b["grad"]) < 1e-13


def _residuals(kind, N, rng):
    r = (rng.standard_normal(N) * np.exp(rng.uniform(-8, 2, N))).astype(np.float32)
    if kind == "zeros_and_nonfinite":
        r[::5] = 0.0
        r[3::17] = np.nan
        r[7::23] = np.inf
        r[11::29] = -np.inf
    elif kind == "uniform_fallback":
        r[:] = 0.0
    return r


@pytest.mark.parametrize("kind", ["generic", "zeros_and_nonfinite", "uniform_fallback"])
@pytest.mark.parametrize("n,N,k,c", [(16, 64, 1.0, 1.0), (37, 111, 2.0, 0.1), (50, 50, 0.5, 3.0)])
def test_expected_counts_are_n_times_probability(kind, n, N, k, c):
    rng = np.random.default_rng(n + N)
    w = ad.weights(_residuals(kind, N, rng), k, c)
    cdf = np.cumsum(w)
    E = imp.expected_counts(cdf, n)
    np.testing.assert_allclose(E, n * ad.probabilities(w), rtol=0, atol=1e-12 * n)
    assert abs(E.sum() - n) < 1e-12 * n
    om = imp.importance_weights(w)
    assert np.all(om <= (1.0 + np.float32(c)) / np.float32(c) * (1 + 1e-15))
    if kind == "uniform_fallback":
        assert np.all(w == 1.0) and np.all(om == 1.0)


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
@pytest.mark.parametrize("k,c", [(1.0, 1.0), (2.0, 0.05)])
def test_expected_weighted_loss_is_the_pool_uniform_loss(golden_dir, variant, k, c):
    """E_u0 of the importance-weighted batch loss and gradient = the pool's uniform loss and gradient: the batch enters
    as per-candidate weights E[c_i] * om_i with the pool-based loss weights."""
    N, n = 96, 24
    (x, y, z, R), m1, m2 = _points(golden_dir, N, seed=7)
    theta = _theta(golden_dir)
    pool = cf.loss_and_grad(variant, theta, x, y, z, R, m1, m2)
    w = ad.weights(pool["res"].astype(np.float32), k, c)
    cdf = np.cumsum(w)
    E = imp.expected_counts(cdf, n)
    om = imp.importance_weights(w, cdf[-1])
    lw = imp.importance_loss_weights(n, N, m1.sum(), m2.sum())
    est = imp.loss_and_grad(variant, theta, x, y, z, R, m1, m2, *lw, point_weights=E * om)
    assert abs(est["Ltot"] - pool["Ltot"]) <= 1e-12 * pool["Ltot"]
    assert _rel(est["grad"], pool["grad"]) < 1e-12
    # one batch at a given u0 is the same sum with its integer counts (the estimate the device step computes)
    idx = ad.select(cdf, n, ad.u0(N, 0, 1))
    cnt = np.bincount(idx, minlength=N)
    one = imp.loss_and_grad(variant, theta, x[idx], y[idx], z[idx], R[idx], m1[idx], m2[idx], *lw, point_weights=om[idx])
    ref = imp.loss_and_grad(variant, theta, x, y, z, R, m1, m2, *lw, point_weights=cnt * om)
    assert abs(one["Ltot"] - ref["Ltot"]) <= 1e-12 * ref["Ltot"]


def test_importance_loss_weights_and_empty_pool_sets():
    np.testing.assert_array_equal(imp.importance_loss_weights(10, 40, 8, 5), [0.1, 40.0 / 80.0, 40.0 / 50.0])
    w = imp.importance_loss_weights(10, 40, 0, 5)
    assert np.isinf(w[1]) and np.isfinite(w[2])


def test_argument_refusals(golden_dir):
    (x, y, z, R), m1, m2 = _points(golden_dir, 8)
    with pytest.raises(ValueError):
        imp.loss_and_grad("poc", _theta(golden_dir), x, y, z, R, m1, m2, point_weights=np.ones(7))
