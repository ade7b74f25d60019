"""Analysis callers of the hot path in inference mode (SURVEY.md 8f-3, 8f-4), on the device:

    simpson_weights          <->  scipy.integrate.simps as nested by integra3d            poc/main.py:179-186
    grid_sums                <->  grid build + parametricPsi + hamiltonian + integra3d     poc/main.py:438-494, 646-676
    energy_from_psi          <->  energy_from_psi(Ri, params)                               poc/main.py:438-464
    energy_from_psi_LCAO     <->  energy_from_psi_LCAO(Ri, params)                          poc/main.py:467-492
    dEdR_int                 <->  dEdR_int(Ri, params) (Hellmann-Feynman)                   poc/main.py:646-676
    calculate_E_R            <->  calculate_E_R(params)                                     poc/main.py:495-517
    spheroidal_sums          <->  the E_int / Elcao sums of calculate_E_R, converged (prolate-spheroidal Gauss-Legendre)
    rayleigh_curve           <->  E_int, Elcao, E_net of calculate_E_R for a whole R sweep in one launch
    enet_curve / returnGate  <->  E-net on an R grid, -dE/dR, d2E/dR2, gate                 energy.py:21-33; poc/main.py:164-176, 1324-1332

The grid is never materialised: the kernel generates the points from the three linspaces and accumulates the
Simpson-weighted sums (pinn_grid_reduce); 10^8 points cost the same memory as 10^3.  That grid cannot resolve the cusps
of psi at the nuclei (E_int is off by ~3e-3 at n_test = 80); spheroidal_sums / rayleigh_curve integrate in
prolate-spheroidal coordinates instead, where the volume element cancels the 1/r terms and ~1000 nodes per R reach
float32 accuracy (pinn_spheroidal_reduce, INTEGRATION.md).
"""
import ctypes

import numpy as np
import torch

from ._lib import Handle, PinnError
from .params import check_supported_model

_DEFAULTS = {"xL": -18, "xR": 18, "yL": -18, "yR": 18, "zL": -18, "zR": 18, "RxL": 0.2, "RxR": 4, "n_test": 80}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def simpson_weights(n, h, rule="avg"):
    """1-D weights w with  integral ~ w @ f  on n equally spaced samples.
    rule 'avg': scipy <= 1.10 `simps` (even='avg'), what the reference called; 'simpson': scipy >= 1.11 `simpson`."""
    def odd(m):
        w = np.zeros(m)
        w[0] = w[-1] = 1.0
        w[1:-1:2] = 4.0
        w[2:-1:2] = 2.0
        return w * h / 3.0
    if n < 3:
        raise ValueError("Simpson needs at least 3 samples")
    if n % 2 == 1:
        return odd(n)
    if rule == "avg":
        a = np.zeros(n); a[:-1] += odd(n - 1); a[-2:] += 0.5 * h
        b = np.zeros(n); b[1:] += odd(n - 1); b[:2] += 0.5 * h
        return 0.5 * (a + b)
    if rule == "simpson":
        w = np.zeros(n); w[:-1] += odd(n - 1); w[-3:] += h * np.array([-1.0 / 12.0, 2.0 / 3.0, 5.0 / 12.0])
        return w
    raise ValueError("rule must be 'avg' or 'simpson'")


def _theta32(theta, dev):
    return torch.as_tensor(np.asarray(theta, np.float64)).to(device=dev, dtype=torch.float32).contiguous()


def grid_sums(theta, Ri, params=None, variant="poc", n=None, rule="avg", device=None):
    """The five quadrature sums + E_net at R = Ri on the n_test^3 grid -> dict.  n: int or (nx, ny, nz)."""
    if not torch.cuda.is_available():
        raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
    pr = dict(_DEFAULTS)
    pr.update(params or {})
    check_supported_model(pr)
    n = pr["n_test"] if n is None else n
    nx, ny, nz = (n, n, n) if np.isscalar(n) else n
    h = Handle.get(torch.cuda.current_device() if device is None else device)
    dev = torch.device("cuda", h.device)
    variant = {"poc": 0, "trainpy": 1}.get(variant, variant)
    lim = (ctypes.c_double * 6)(pr["xL"], pr["xR"], pr["yL"], pr["yR"], pr["zL"], pr["zR"])
    # integra3d integrates the LAST tensor axis with the x samples and the first with z (poc/main.py:185); the axes of
    # the reference's grids are identical, so the product rule below is the same number
    w = [torch.as_tensor(simpson_weights(m, (hi - lo) / (m - 1), rule)).to(dev)
         for m, lo, hi in ((nx, pr["xL"], pr["xR"]), (ny, pr["yL"], pr["yR"]), (nz, pr["zL"], pr["zR"]))]
    out = torch.empty(8, dtype=torch.float64, device=dev)
    th = _theta32(theta, dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    rc = h.L.pinn_grid_reduce(h.h, variant, _ptr(th), nx, ny, nz, lim, float(Ri), _ptr(w[0]), _ptr(w[1]), _ptr(w[2]),
                              _ptr(out), ctypes.c_void_p(stream))
    h.check(rc, "pinn_grid_reduce")
    o = out.cpu().numpy()
    return {"psiHpsi": o[0], "psi2": o[1], "lcaoHlcao": o[2], "lcao2": o[3], "dVdR_psi2": o[4], "E_net": o[5]}


def energy_from_psi(theta, Ri, params=None, **kw):
    """(E_integral, E_net) = (<psi|H|psi>/<psi|psi>, E-net(Ri))  poc/main.py:438-464"""
    s = grid_sums(theta, Ri, params, **kw)
    return s["psiHpsi"] / s["psi2"], s["E_net"]


def energy_from_psi_LCAO(theta, Ri, params=None, **kw):
    """<lcao|H|lcao>/<lcao|lcao>  poc/main.py:467-492"""
    s = grid_sums(theta, Ri, params, **kw)
    return s["lcaoHlcao"] / s["lcao2"]


def dEdR_int(theta, Ri, params=None, **kw):
    """Hellmann-Feynman force integral with the nuclear term: <psi|dV/dR|psi>/<psi|psi> - 1/(2 Ri^2)  poc/main.py:646-676"""
    s = grid_sums(theta, Ri, params, **kw)
    return s["dVdR_psi2"] / s["psi2"] - 1.0 / (2.0 * Ri ** 2)


def calculate_E_R(theta, params=None, **kw):
    """energyDictionary of calculate_E_R (poc/main.py:495-517): R = RxL .. RxR step 0.1 -> E_int, Elcao, E_net (+ dEdR)."""
    pr = dict(_DEFAULTS)
    pr.update(params or {})
    Rs = np.round(np.arange(pr["RxL"], pr["RxR"] + .1, .1), 2)
    d = {"R": Rs, "E_int": np.zeros(len(Rs)), "Elcao": np.zeros(len(Rs)), "E_net": np.zeros(len(Rs)),
         "dEdR_HF": np.zeros(len(Rs))}
    for i, Ri in enumerate(Rs):
        s = grid_sums(theta, float(Ri), pr, **kw)
        d["E_int"][i] = s["psiHpsi"] / s["psi2"]
        d["Elcao"][i] = s["lcaoHlcao"] / s["lcao2"]
        d["E_net"][i] = s["E_net"]
        d["dEdR_HF"][i] = s["dVdR_psi2"] / s["psi2"] - 1.0 / (2.0 * Ri ** 2)
    return d


def spheroidal_nodes(n_s=16, n_nu=24, panels=(0, 2, 6, 18)):
    """(s, ws, nu, wnu), float64: Gauss-Legendre with n_s nodes on every panel [panels[i], panels[i+1]] of
    s = (r1 + r2)/2 - R and n_nu nodes on nu = (r2 - r1)/(2R) in [-1, 1].  The domain is the spheroid
    r1 + r2 <= 2 (R + panels[-1]); the same nodes serve every R."""
    panels = np.asarray(panels, np.float64)
    if n_s < 1 or n_nu < 1 or panels.size < 2 or panels[0] < 0 or np.any(np.diff(panels) <= 0):
        raise ValueError("need n_s, n_nu >= 1 and increasing panel edges starting at s >= 0")
    t, wt = np.polynomial.legendre.leggauss(int(n_s))
    half = 0.5 * np.diff(panels)
    s = (panels[:-1, None] + half[:, None] * (t[None, :] + 1.0)).ravel()
    ws = (half[:, None] * wt[None, :]).ravel()
    nu, wnu = np.polynomial.legendre.leggauss(int(n_nu))
    return s, ws, nu, wnu


def spheroidal_sums(theta, R, variant="poc", n_s=16, n_nu=24, panels=(0, 2, 6, 18), params=None, device=None):
    """psiHpsi, psi2, lcaoHlcao, lcao2 (the sums of grid_sums) and E_net at every R, on the spheroidal node set of
    spheroidal_nodes -> dict of float64 arrays over R.  One launch (+ one finishing reduction) for the whole sweep, one
    host synchronisation.  The Hellmann-Feynman sum is not formed: its integrand is not smooth in these coordinates."""
    if not torch.cuda.is_available():
        raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
    check_supported_model(params or {})
    Rh = np.asarray(R, np.float64).ravel()
    if Rh.size == 0 or not np.all(Rh > 0) or not np.all(np.isfinite(Rh)):
        raise ValueError("R must be a non-empty list of finite values > 0")
    h = Handle.get(torch.cuda.current_device() if device is None else device)
    dev = torch.device("cuda", h.device)
    variant = {"poc": 0, "trainpy": 1}.get(variant, variant)
    s, ws, nu, wnu = [torch.as_tensor(a).to(dev) for a in spheroidal_nodes(n_s, n_nu, panels)]
    Rd = torch.as_tensor(Rh).to(dev)
    out = torch.empty((Rh.size, 8), dtype=torch.float64, device=dev)
    th = _theta32(theta, dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    rc = h.L.pinn_spheroidal_reduce(h.h, variant, _ptr(th), Rh.size, _ptr(Rd), s.numel(), _ptr(s), _ptr(ws), nu.numel(),
                                    _ptr(nu), _ptr(wnu), _ptr(out), ctypes.c_void_p(stream))
    h.check(rc, "pinn_spheroidal_reduce")
    o = out.cpu().numpy()
    return {"psiHpsi": o[:, 0], "psi2": o[:, 1], "lcaoHlcao": o[:, 2], "lcao2": o[:, 3], "E_net": o[:, 5]}


def rayleigh_curve(theta, R=None, params=None, **kw):
    """E_int = <psi|H|psi>/<psi|psi>, Elcao and E_net over an R sweep, converged (spheroidal_sums) -> dict of arrays.
    R defaults to the R list of calculate_E_R (RxL .. RxR step 0.1)."""
    pr = dict(_DEFAULTS)
    pr.update(params or {})
    if R is None:
        R = np.round(np.arange(pr["RxL"], pr["RxR"] + .1, .1), 2)
    R = np.asarray(R, np.float64).ravel()
    s = spheroidal_sums(theta, R, params=pr, **kw)
    return {"R": R, "E_int": s["psiHpsi"] / s["psi2"], "Elcao": s["lcaoHlcao"] / s["lcao2"], "E_net": s["E_net"]}


def enet_curve(theta, R, device=None):
    """E(R), dE/dR, d2E/dR2 of the E-net and the gate g(R) at the given R values (float64) -> dict of numpy arrays."""
    if not torch.cuda.is_available():
        raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
    h = Handle.get(torch.cuda.current_device() if device is None else device)
    dev = torch.device("cuda", h.device)
    Rd = torch.as_tensor(np.asarray(R, np.float64).ravel()).to(dev)
    n = Rd.numel()
    outs = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(4)]
    th = _theta32(theta, dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    rc = h.L.pinn_enet_curve(h.h, _ptr(th), _ptr(Rd), n, *[_ptr(o) for o in outs], ctypes.c_void_p(stream))
    h.check(rc, "pinn_enet_curve")
    E, dE, d2E, g = [o.cpu().numpy() for o in outs]
    return {"R": np.asarray(R, np.float64).ravel(), "E": E, "dE": dE, "d2E": d2E, "gate": g}


def energy_curve(theta, Rlo=0.2, Rhi=4.0, n=1000):
    """energy.py:21-33: R grid and the total energy E(R) + 1/(2R) it plots."""
    R = np.linspace(Rlo, Rhi, n)
    c = enet_curve(theta, R)
    return R, c["E"] + 1.0 / (2.0 * R)


def returnGate(theta, params=None, n=None):
    """returnGate() poc/main.py:164-176 -> (R, gate) as (n,1) arrays."""
    pr = dict(_DEFAULTS)
    pr.update(params or {})
    n = n or pr.get("n_train", 100000)
    R = np.linspace(pr["RxL"], pr["RxR"], n)
    c = enet_curve(theta, R)
    return R.reshape(-1, 1), c["gate"].reshape(-1, 1)
