"""The prolate-spheroidal quadrature oracle (oracle/spheroidal.py) on the CPU: exact integrals, the LCAO closed form,
convergence in the node count, and the variational bound against the exact energies."""
import os

import numpy as np

from oracle import spheroidal as sph

R39 = np.round(np.arange(0.2, 4.0 + .1, .1), 2)   # the R list of calculate_E_R (poc/main.py:495-517)


def test_integral_of_exp_minus_2r1_is_pi():
    s, ws, nu, wnu = sph.nodes()
    for R in (0.2, 1.0, 4.0):
        x, y, z, r1r2 = sph.points(R, s, nu)
        w = 2.0 * np.pi * np.outer(ws, wnu).ravel() * r1r2
        r1 = np.sqrt((x - R) ** 2 + y * y + z * z)
        assert abs(w @ np.exp(-2.0 * r1) - np.pi) < 1e-12, R


def test_lcao_quotient_equals_its_closed_form():
    assert abs(sph.lcao_energy(1.0) - (-1.0537714953)) < 1e-10
    d = sph.sums("poc", np.zeros(1521), R39)   # (the LCAO sums do not depend on theta)
    assert np.abs(d["lcaoHlcao"] / d["lcao2"] - sph.lcao_energy(R39)).max() < 1e-12


def test_trained_model_energy_is_converged_and_above_the_exact_one(golden_dir):
    th = np.load(os.path.join(golden_dir, "checkpoints.npz"))["ionHsym_fineTune"]
    a = sph.sums("poc", th, R39)
    b = sph.sums("poc", th, R39, n_s=32, n_nu=48)
    Ea, Eb = a["psiHpsi"] / a["psi2"], b["psiHpsi"] / b["psi2"]
    assert np.abs(Ea - Eb).max() < 1e-9
    ex = np.load(os.path.join(golden_dir, "poc_paper_run_seed0.npz"))
    assert np.allclose(ex["R"], R39)
    # variational bound; the exact table has 4 decimals
    assert np.all(Ea > ex["E_exact"] - 5e-5), (Ea - ex["E_exact"]).min()
