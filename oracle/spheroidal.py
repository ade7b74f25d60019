"""Prolate-spheroidal quadrature oracle (TEST INFRASTRUCTURE ONLY): float64 restatement of pinn_spheroidal_reduce.

With the nuclei at x = +R (r1) and x = -R (r2), mu = (r1 + r2)/(2R), nu = (r2 - r1)/(2R) and s = R (mu - 1) >= 0:

    x = R mu nu,   rho = R sqrt((mu^2 - 1)(1 - nu^2)),   dV = r1 r2 ds dnu dphi,   r1 r2 = (R + s)^2 - (R nu)^2

Every wavefunction of the model depends on (x, y, z) through r1 and r2 only, so the phi integral is 2 pi and the factor
r1 r2 of dV cancels the 1/r singularities of H psi: tensor Gauss-Legendre in (s, nu) converges exponentially.  The
domain is the spheroid r1 + r2 <= 2 (R + panels[-1]).
"""
import numpy as np
from scipy.special import roots_legendre

from . import closed_form


def nodes(n_s=16, n_nu=24, panels=(0, 2, 6, 18)):
    """(s, ws, nu, wnu): n_s Gauss-Legendre nodes on every panel [panels[i], panels[i+1]] of s, n_nu on nu in [-1, 1]."""
    t, wt = roots_legendre(n_s)
    s, ws = [], []
    for a, b in zip(panels[:-1], panels[1:]):
        h = 0.5 * (b - a)
        s.append(a + h * (t + 1.0))
        ws.append(h * wt)
    nu, wnu = roots_legendre(n_nu)
    return np.concatenate(s), np.concatenate(ws), np.asarray(nu, np.float64), np.asarray(wnu, np.float64)


def points(R, s, nu):
    """Cartesian points (x, y, z) and weights factor r1 r2 of the (s, nu) tensor grid at one R, s-major."""
    S, NU = np.meshgrid(s, nu, indexing="ij")
    S, NU = S.ravel(), NU.ravel()
    mu = 1.0 + S / R
    x = R * mu * NU
    y = np.sqrt(S * (2.0 * R + S) * (1.0 - NU * NU))
    return x, y, np.zeros_like(x), (R + S) ** 2 - (R * NU) ** 2


def sums(variant, theta, R, n_s=16, n_nu=24, panels=(0, 2, 6, 18)):
    """{psiHpsi, psi2, lcaoHlcao, lcao2, E_net} as arrays over R (float64 throughout)."""
    s, ws, nu, wnu = nodes(n_s, n_nu, panels)
    W2 = 2.0 * np.pi * np.outer(ws, wnu).ravel()
    R = np.atleast_1d(np.asarray(R, np.float64))
    out = {k: np.zeros(R.size) for k in ("psiHpsi", "psi2", "lcaoHlcao", "lcao2", "E_net")}
    for k, Rk in enumerate(R):
        x, y, z, r1r2 = points(Rk, s, nu)
        f = closed_form.fields(variant, theta, x, y, z, np.full(x.size, Rk))
        w = W2 * r1r2
        r1 = np.sqrt((x - Rk) ** 2 + y * y)
        r2 = np.sqrt((x + Rk) ** 2 + y * y)
        f1, f2 = np.exp(-r1), np.exp(-r2)
        lc = f1 + f2
        hl = -0.5 * lc - f1 / r2 - f2 / r1   # H e^-r1 = -1/2 e^-r1 - e^-r1 / r2: the 1/r1 terms cancel
        out["psiHpsi"][k] = w @ (f["psi"] * f["hpsi"])
        out["psi2"][k] = w @ (f["psi"] ** 2)
        out["lcaoHlcao"][k] = w @ (lc * hl)
        out["lcao2"][k] = w @ (lc * lc)
        out["E_net"][k] = f["E"][0]
    return out


def lcao_energy(R):
    """<lcao|H|lcao>/<lcao|lcao> of lcao = e^-r1 + e^-r2 in closed form (electronic energy, no 1/(2R) term):
    D = 2R, overlap S, Coulomb J and exchange K integrals of the 1s orbitals, E = -1/2 - (J + K)/(1 + S)."""
    D = 2.0 * np.asarray(R, np.float64)
    S = np.exp(-D) * (1.0 + D + D * D / 3.0)
    J = 1.0 / D - np.exp(-2.0 * D) * (1.0 + 1.0 / D)
    K = np.exp(-D) * (1.0 + D)
    return -0.5 - (J + K) / (1.0 + S)
