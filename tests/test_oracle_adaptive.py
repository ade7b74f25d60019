"""The numpy restatement of residual-adaptive selection (oracle/adaptive.py) on the CPU: the count bounds of systematic
resampling, the uniform fall-backs, non-finite residuals, and u0 on the Philox known-answer path."""
import numpy as np
import pytest

from oracle import adaptive as ad
from oracle import philox


@pytest.mark.parametrize("n,N,k,c,seed", [(1000, 4000, 1.0, 1.0, 0), (4096, 4096, 2.0, 0.0, 1), (777, 5000, 1.0, 0.1, 2),
                                          (1 << 14, 1 << 16, 0.5, 1.0, 3)])
def test_selection_counts_within_floor_and_ceil(n, N, k, c, seed):
    rng = np.random.default_rng(seed)
    res = (rng.standard_normal(N) * np.exp(rng.uniform(-20, 2, N))).astype(np.float32)
    w = ad.weights(res, k, c)
    cdf = np.cumsum(w)
    for u in (0.0, ad.u0(N, seed, 7), 1.0 - 2.0 ** -32):
        idx = ad.select(cdf, n, u)
        assert idx.shape == (n,) and idx.min() >= 0 and idx.max() < N
        assert np.all(np.diff(idx) >= 0)  # systematic resampling walks the pool in order
        cnt = np.bincount(idx, minlength=N)
        lo, hi = ad.count_bounds(ad.probabilities(np.diff(cdf, prepend=0.0)), n, slack=1e-9)
        assert np.all(cnt >= lo) and np.all(cnt <= hi)
        if c == 0.0:
            assert np.all(cnt[w == 0.0] == 0)


def test_k_zero_and_zero_residuals_are_uniform():
    rng = np.random.default_rng(5)
    res = rng.standard_normal(1000).astype(np.float32)
    w0 = ad.weights(res, 0.0, 1.0)
    assert np.all(w0 == w0[0])
    wz = ad.weights(np.zeros(1000, np.float32), 1.0, 1.0)
    assert np.all(wz == 1.0)
    cnt = np.bincount(ad.select(np.cumsum(wz), 250, 0.5), minlength=1000)
    assert set(np.unique(cnt)) <= {0, 1} and cnt.sum() == 250


def test_non_finite_residuals_get_weight_c():
    res = np.array([1.0, np.nan, 2.0, np.inf, -np.inf, -3.0], np.float32)
    w = ad.weights(res, 1.0, 0.25)
    assert np.all(w[[1, 3, 4]] == np.float64(np.float32(0.25)))
    Q = 6.0
    np.testing.assert_array_equal(w[[0, 2, 5]], np.array([1.0, 2.0, 3.0]) * 6.0 / Q + 0.25)
    assert np.all(ad.weights(np.full(4, np.nan, np.float32), 1.0, 0.25) == 1.0)  # Q = 0: uniform


def test_u0_on_philox_known_answers():
    # Random123 known-answer vectors of Philox4x32-10: counter 0 / key 0 and counter 2^32-1 everywhere
    assert ad.u0(0, 0, 0) == 0x6627E8D5 * 2.0 ** -32
    m = (1 << 64) - 1
    assert ad.u0(m, m, m) == 0x408F276D * 2.0 ** -32
    # the point just past a pool of N in the pool's own stream: the same counter the sampler would give point N
    N, seed, batch = 12345, 0xDEADBEEF12345678, (5 << 32) + 3
    r = philox.philox4x32_10(N, 0, batch & 0xFFFFFFFF, batch >> 32, seed & 0xFFFFFFFF, seed >> 32)
    assert ad.u0(N, seed, batch) == float(r[0]) * 2.0 ** -32
    assert 0.0 <= ad.u0(N, seed, batch) < 1.0
