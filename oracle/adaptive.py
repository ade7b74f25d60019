"""Residual-adaptive selection of pinn_sample_adaptive restated in numpy float64 (TEST INFRASTRUCTURE ONLY).

RAD (Wu, Zhu, Tan, Kartha & Lu, CMAME 403, 2023) with systematic resampling, as include/pinn_b200.h states it:
weights w_i = |res_i|^k * N / Q + c (Q = sum |res_j|^k over finite residuals; w = 1 when Q is 0 or not finite),
u0 = word 0 of Philox4x32-10 at counter {N, batch} times 2^-32, and output j = the first i with
cdf[i] > (j + u0) / n * cdf[N-1].
"""
import numpy as np

from .philox import philox4x32_10


def weights(res, k, c):
    """float32 residuals -> float64 weights w (the device's k and c are float32)"""
    r = np.asarray(res, np.float32).astype(np.float64)
    k, c = float(np.float32(k)), float(np.float32(c))
    fin = np.isfinite(r)
    q = np.zeros_like(r)
    with np.errstate(over="ignore"):  # |res|^k past the float64 range is inf, as on the device
        q[fin] = np.abs(r[fin]) ** k
    Q = q.sum()
    if not (Q > 0.0 and np.isfinite(Q)):
        return np.ones_like(r)
    return q * float(r.size) / Q + c


def u0(pool, seed, batch):
    """Word 0 of Philox4x32-10 at counter {pool_lo, pool_hi, batch_lo, batch_hi}, key = seed, times 2^-32"""
    w = philox4x32_10(pool & 0xFFFFFFFF, (pool >> 32) & 0xFFFFFFFF, batch & 0xFFFFFFFF, (batch >> 32) & 0xFFFFFFFF,
                      seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)[0]
    return float(np.uint32(w)) * 2.0 ** -32


def select(cdf, n, u):
    """Systematic resampling over a non-decreasing float64 cdf: the pool index of every output j in [0, n)"""
    cdf = np.asarray(cdf, np.float64)
    t = (np.arange(n, dtype=np.float64) + u) / np.float64(n) * cdf[-1]
    return np.minimum(np.searchsorted(cdf, t, side="right"), cdf.size - 1)


def probabilities(w):
    """P_i = w_i / sum w"""
    w = np.asarray(w, np.float64)
    return w / w.sum()


def count_bounds(P, n, slack=0.0):
    """floor(n P_i - slack), ceil(n P_i + slack): the counts systematic resampling can give candidate i"""
    nP = n * np.asarray(P, np.float64)
    return np.floor(nP - slack), np.ceil(nP + slack)
