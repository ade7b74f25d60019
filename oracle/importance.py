"""Importance-weighted adaptive batches restated on the CPU in float64 (TEST INFRASTRUCTURE ONLY).

* ``loss_and_grad``           - closed_form.loss_and_grad with a per-point weight om: every per-point term of the sums
                                (res^2, m1 psi^2, m2 psi^2, E) and so of the gradient takes om, while the default set
                                sizes stay counts of points (pinn_loss_fwd_bwd_weighted).  The hand-written reverse sweep
                                of closed_form, with the seeds scaled by om.
* ``autograd_loss_and_grad``  - the same weighted loss by nested autograd (ref_autograd's fields), which the closed form
                                is checked against.
* ``importance_weights``, ``importance_loss_weights`` - om_i = T / (N w_i) = 1 / (N P_i) and the loss weights {1/n,
                                N/(n |set1 of the pool|), N/(n |set2 of the pool|)} of pinn_sample_adaptive_importance.
* ``expected_counts``         - E over u0 of the counts of systematic resampling (oracle/adaptive.py:select), exactly.

Systematic resampling takes candidate i c_i(u0) times with E_u0[c_i] = n P_i, so the expectation of the weighted batch
loss is the pool's uniform loss {1/N, 1/|set1|, 1/|set2|}.
"""
import numpy as np
import torch

from . import closed_form as cf
from . import layout
from . import ref_autograd as ra
from .adaptive import select


def loss_and_grad(variant, theta, x, y, z, R, m1, m2, w_pde=None, w_bc1=None, w_bc2=None, point_weights=None):
    """closed_form.loss_and_grad with per-point weights (None: all 1, the unweighted loss)."""
    P = layout.unpack_poc(theta)
    x, y, z, R = [np.asarray(v, np.float64).reshape(-1) for v in (x, y, z, R)]
    m1 = np.asarray(m1, np.float64).reshape(-1)
    m2 = np.asarray(m2, np.float64).reshape(-1)
    n = x.size
    om = np.ones(n) if point_weights is None else np.asarray(point_weights, np.float64).reshape(-1)
    if om.size != n:
        raise ValueError("point_weights must have one entry per point")
    w_pde = 1.0 / n if w_pde is None else w_pde
    w_bc1 = 1.0 / m1.sum() if w_bc1 is None else w_bc1
    w_bc2 = 1.0 / m2.sum() if w_bc2 is None else w_bc2
    nev, sN, cL, cV, cE = cf.VARIANTS[variant]
    f = cf._forward(variant, P, x, y, z, R)
    res, psi, gate, E, N, DN, q = f["res"], f["psi"], f["gate"], f["E"], f["N"], f["DN"], f["q"]
    sums = dict(res2=(om * res * res).sum(), psi2_1=(om * m1 * psi * psi).sum(), psi2_2=(om * m2 * psi * psi).sum(),
                E=(om * E).sum())
    Lpde = w_pde * sums["res2"]
    Lbc = w_bc1 * sums["psi2_1"] + w_bc2 * sums["psi2_2"]
    # seeds: closed_form's, each point's scaled by its weight
    rbar = 2 * w_pde * res * om
    pbar = 2 * (w_bc1 * m1 + w_bc2 * m2) * psi * om
    lamN = rbar * gate * (cV * q + cE * E) + pbar * gate
    lamD = rbar * cL * gate
    gbar = rbar * (cL * DN + cV * q * N + cE * E * N) + pbar * N
    Ebar = rbar * cE * psi
    gA = cf.mlp_bwd(P, f["stA"], sN * lamN, sN * lamD)
    if nev == 2:
        gB = cf.mlp_bwd(P, f["stB"], sN * lamN, sN * lamD)
        gA = [a + b for a, b in zip(gA, gB)]
    grads = gA + [np.array([lamN.sum()])] + cf.enet_bwd(P, R, f["stE"], Ebar) + cf.gate_bwd(P, R, f["stG"], gbar)
    return dict(Ltot=Lpde + Lbc, Lpde=Lpde, Lbc=Lbc, E=E, grad=layout.pack_poc(grads), sums=sums,
                psi=psi, res=res, lap=f["lap"])


def autograd_loss_and_grad(variant, theta, x, y, z, R, m1, m2, om, w_pde, w_bc1, w_bc2):
    """The weighted training loss by nested autograd (float64):
    Ltot = w_pde sum om res^2 + w_bc1 sum om m1 psi^2 + w_bc2 sum om m2 psi^2 -> (Ltot, Lpde, Lbc, sum om E, dLtot/dtheta).
    x, y, z, R: (n, 1) float64 tensors; m1, m2, om: (n,) float64 tensors (set membership 0/1 and the per-point weights)."""
    theta = theta.detach().clone().requires_grad_(True)
    if variant == "poc":
        psi, _, _, res, E = ra.poc_fields(theta, x, y, z, R)
    else:
        psi, _, res, E = ra.trainpy_fields(theta, x, y, z, R)
    psi, res, E = psi[:, 0], res[:, 0], E[:, 0]
    Lpde = w_pde * (om * res ** 2).sum()
    Lbc = w_bc1 * (om * m1 * psi ** 2).sum() + w_bc2 * (om * m2 * psi ** 2).sum()
    Ltot = Lpde + Lbc
    Ltot.backward()
    return Ltot.detach(), Lpde.detach(), Lbc.detach(), (om * E).sum().detach(), theta.grad.detach()


def importance_weights(w, total=None):
    """om_i = T / (N w_i) (T = sum w unless given, e.g. the device's cdf[N-1])"""
    w = np.asarray(w, np.float64)
    T = w.sum() if total is None else float(total)
    return T / (float(w.size) * w)


def importance_loss_weights(n, N, count1, count2):
    """{1/n, N/(n |set1|), N/(n |set2|)} of the pool's set sizes, as the device forms them (an empty set: inf)"""
    with np.errstate(divide="ignore"):
        return np.array([1.0 / n, np.float64(N) / (np.float64(n) * np.float64(count1)),
                         np.float64(N) / (np.float64(n) * np.float64(count2))])


def expected_counts(cdf, n):
    """E over u0 ~ U[0, 1) of c_i(u0) = #{j : select(cdf, n, u0)[j] = i}, exactly: c(u0) only changes where some
    t_j = (j + u0) / n * T crosses a cdf entry, i.e. at u0 = frac(cdf[i] n / T); between two such breakpoints it is
    constant, so the integral is the sum of c at each piece's midpoint times the piece's length."""
    cdf = np.asarray(cdf, np.float64)
    T = cdf[-1]
    b = np.mod(cdf * n / T, 1.0)
    b = np.unique(np.concatenate([[0.0, 1.0], b[(b > 0.0) & (b < 1.0)]]))
    E = np.zeros(cdf.size)
    for lo, hi in zip(b[:-1], b[1:]):
        if hi > lo:
            E += (hi - lo) * np.bincount(select(cdf, n, 0.5 * (lo + hi)), minlength=cdf.size)
    return E
