"""GPU tests of the prolate-spheroidal quadrature (pinn_spheroidal_reduce, analysis.spheroidal_sums / rayleigh_curve):
parity with the float64 oracle and with the per-point inference summed on the host, the LCAO closed form, the
variational bound, determinism across sweeps, and argument checking."""
import ctypes
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import spheroidal as osph

pytestmark = pytest.mark.gpu

R39 = np.round(np.arange(0.2, 4.0 + .1, .1), 2)   # the R list of calculate_E_R (poc/main.py:495-517)
SUMS = ("psiHpsi", "psi2", "lcaoHlcao", "lcao2")


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ck(golden_dir):
    return np.load(os.path.join(golden_dir, "checkpoints.npz"))


@pytest.fixture(scope="module")
def init_theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]   # train.py's init rule, seed 12345


@pytest.fixture(scope="module")
def exact(golden_dir):
    ex = np.load(os.path.join(golden_dir, "poc_paper_run_seed0.npz"))
    assert np.allclose(ex["R"], R39)
    return ex["E_exact"]


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
@pytest.mark.parametrize("weights", ["fineTune", "init"])
def test_sums_match_the_float64_oracle(variant, weights, ck, init_theta):
    th32 = (ck["ionHsym_fineTune"] if weights == "fineTune" else init_theta).astype(np.float32)
    R = np.array([0.2, 0.7, 2.0, 4.0])
    got = pk.analysis.spheroidal_sums(th32, R, variant=variant)
    ref = osph.sums(variant, th32.astype(np.float64), R)
    for k in SUMS:
        assert np.all(np.abs(got[k] - ref[k]) <= 2e-5 * np.abs(ref[k])), (k, got[k], ref[k])
    assert np.abs(got["E_net"] - ref["E_net"]).max() < 1e-6


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
def test_sums_equal_the_per_point_fields_summed_on_the_host(variant, ck, init_theta):
    """The points of the documented formulas, built on the host in float64 and passed to `fields`, are the kernel's
    points: the quadrature of the per-point psi and H psi with the same weights is the kernel's sums, and E_net is the
    per-point E.  13 x 21 nodes per panel -> 39 * 21 = 819 per R: 7 super-tiles per R, the last one ragged."""
    th32 = (ck["ionHsym_fineTune"] if variant == "poc" else init_theta).astype(np.float32)
    R = np.array([0.35, 1.3, 3.1])
    s, ws, nu, wnu = pk.analysis.spheroidal_nodes(13, 21)
    got = pk.analysis.spheroidal_sums(th32, R, variant=variant, n_s=13, n_nu=21)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    S, NU = (a.ravel() for a in np.meshgrid(s, nu, indexing="ij"))
    WS, WNU = (a.ravel() for a in np.meshgrid(ws, wnu, indexing="ij"))
    for k, Rk in enumerate(R):
        x = Rk * (1.0 + S / Rk) * NU
        y = np.sqrt(S * (2.0 * Rk + S) * (1.0 - NU * NU))
        w = 2.0 * np.pi * WS * WNU * ((Rk + S) ** 2 - (Rk * NU) ** 2)
        f = pk.fields(variant, t(x), t(y), t(np.zeros_like(x)), t(np.full(x.size, Rk)), torch.from_numpy(th32).to(dev()))
        psi, hpsi = (f[q].cpu().numpy() for q in ("psi", "hpsi"))
        # (the kernel forms the products in float32, as here, and accumulates the weighted products in float64)
        ref = {"psiHpsi": w @ (psi * hpsi).astype(np.float64), "psi2": w @ (psi * psi).astype(np.float64)}
        for q in ref:
            assert abs(got[q][k] - ref[q]) <= 1e-9 * abs(ref[q]), (q, Rk, got[q][k], ref[q])
        assert got["E_net"][k] == float(f["E"].cpu().numpy()[0])


def test_lcao_column_matches_the_closed_form_at_1000_R(ck):
    R = np.linspace(0.2, 4.0, 1000)
    d = pk.analysis.rayleigh_curve(ck["ionHsym_fineTune"], R)
    err = np.abs(d["Elcao"] - osph.lcao_energy(R)).max()
    print("spheroidal Elcao vs closed form, 1000 R in [0.2, 4]: max error %.2e" % err)
    assert err < 1e-7                                      # measured 2.7e-8 on a B200 (float32 points, float64 sums)


def test_trained_energy_is_variational_and_converged(ck, exact):
    th = ck["ionHsym_fineTune"]
    d = pk.analysis.rayleigh_curve(th)
    assert np.array_equal(d["R"], R39)
    print("E_int - E_exact over the 39 R: min %.2e max %.2e" % ((d["E_int"] - exact).min(), (d["E_int"] - exact).max()))
    assert np.all(d["E_int"] > exact - 5e-5)              # the table has 4 decimals
    fine = pk.analysis.rayleigh_curve(th, n_s=32, n_nu=48)
    dE = np.abs(fine["E_int"] - d["E_int"]).max()
    print("E_int, 16x24 -> 32x48 nodes per panel: max change %.2e" % dE)
    assert dE < 1e-6


def _raw(h, variant, th, R, nodes, out, stream):
    s, ws, nu, wnu = nodes
    p = lambda a: ctypes.c_void_p(a.data_ptr()) if a is not None else None
    return h.L.pinn_spheroidal_reduce(h.h, variant, p(th), R.numel() if R is not None else 1, p(R),
                                      s.numel(), p(s), p(ws), nu.numel(), p(nu), p(wnu), p(out), ctypes.c_void_p(stream))


def test_sweep_rows_are_the_bits_of_single_R_calls(ck):
    th = ck["ionHsym_fineTune"]
    a = pk.analysis.spheroidal_sums(th, R39)
    b = pk.analysis.spheroidal_sums(th, R39)
    for k in SUMS + ("E_net",):
        assert np.array_equal(a[k], b[k]), k
    for i, Rk in enumerate(R39):
        one = pk.analysis.spheroidal_sums(th, [Rk])
        for k in SUMS + ("E_net",):
            assert one[k][0] == a[k][i], (k, Rk)
    # the raw rows: slot 4 (Hellmann-Feynman) is not formed, slots 6 and 7 are zero
    h = pk.Handle.get(0)
    nodes = [torch.as_tensor(v).to(dev()) for v in pk.analysis.spheroidal_nodes()]
    th32 = torch.as_tensor(th.astype(np.float32)).to(dev())
    Rd = torch.as_tensor(R39).to(dev())
    out = torch.full((R39.size, 8), 7.0, dtype=torch.float64, device=dev())
    h.check(_raw(h, 0, th32, Rd, nodes, out, torch.cuda.current_stream().cuda_stream), "pinn_spheroidal_reduce")
    o = out.cpu().numpy()
    assert np.all(o[:, [4, 6, 7]] == 0.0) and np.array_equal(o[:, 0], a["psiHpsi"])


def test_argument_errors_launch_nothing_and_R_le_0_gives_nan_rows(ck):
    h = pk.Handle.get(0)
    st = torch.cuda.current_stream().cuda_stream
    nodes = [torch.as_tensor(v).to(dev()) for v in pk.analysis.spheroidal_nodes(4, 5)]
    th32 = torch.as_tensor(ck["ionHsym_fineTune"].astype(np.float32)).to(dev())
    Rd = torch.tensor([1.0, 2.0], dtype=torch.float64, device=dev())
    out = torch.empty((2, 8), dtype=torch.float64, device=dev())
    s, ws, nu, wnu = nodes
    L, vp = h.L, lambda a: ctypes.c_void_p(a.data_ptr())
    bad = [
        (None, Rd, nodes, out, 0), (th32, None, nodes, out, 0), (th32, Rd, [None, ws, nu, wnu], out, 0),
        (th32, Rd, [s, None, nu, wnu], out, 0), (th32, Rd, [s, ws, None, wnu], out, 0),
        (th32, Rd, [s, ws, nu, None], out, 0), (th32, Rd, nodes, None, 0), (th32, Rd, nodes, out, 2), (th32, Rd, nodes, out, -1),
    ]
    before = h.launch_count()
    for th_, R_, nd, o_, var in bad:
        s_, ws_, nu_, wnu_ = nd
        p = lambda a: vp(a) if a is not None else None
        rc = L.pinn_spheroidal_reduce(h.h, var, p(th_), 2, p(R_), 4 * 3, p(s_), p(ws_), 5, p(nu_), p(wnu_), p(o_),
                                      ctypes.c_void_p(st))
        with pytest.raises(pk.PinnError):
            h.check(rc, "pinn_spheroidal_reduce")
    for nR, ns, nnu in ((0, 12, 5), (2, 0, 5), (2, 12, 0), (-1, 12, 5), (200000, 12000, 24)):
        rc = L.pinn_spheroidal_reduce(h.h, 0, vp(th32), nR, vp(Rd), ns, vp(s), vp(ws), nnu, vp(nu), vp(wnu), vp(out),
                                      ctypes.c_void_p(st))
        with pytest.raises(pk.PinnError):
            h.check(rc, "pinn_spheroidal_reduce")
    assert h.launch_count() == before
    with pytest.raises(ValueError):
        pk.analysis.spheroidal_sums(ck["ionHsym_fineTune"], [1.0, 0.0])
    # the handle is fine; R <= 0 on the device gives NaN rows, the other rows are the numbers of a clean call
    Rbad = torch.tensor([1.0, 0.0, -0.5, 2.0], dtype=torch.float64, device=dev())
    out4 = torch.empty((4, 8), dtype=torch.float64, device=dev())
    h.check(_raw(h, 0, th32, Rbad, nodes, out4, st), "pinn_spheroidal_reduce")
    assert h.launch_count() == before + 2
    o = out4.cpu().numpy()
    assert np.all(np.isnan(o[1])) and np.all(np.isnan(o[2]))
    good = pk.analysis.spheroidal_sums(ck["ionHsym_fineTune"], [1.0, 2.0], n_s=4, n_nu=5)
    assert np.array_equal(o[[0, 3], 0], good["psiHpsi"]) and np.array_equal(o[[0, 3], 5], good["E_net"])
