"""The fused training step at saturated sigmoids, and the dense-grid kernel past 2^31 points.

The other parity tests run three weight vectors (train.py's init and the two shipped checkpoints), whose sigmoid
pre-activations stay within about [-11.5, 5.3].  Here every sigmoid layer in turn is driven into u in [8, 12] and into
[-12, -8] - there 1 - sigma(u) is e^-u, between 6e-6 and 3e-4 - and the step is compared with the float64 oracle at the
bars of test_gpu_parity.py, per tensor and per gradient entry: Adam takes a full-size step on every entry, so a small
entry has to be as accurate as a large one.

Regimes are built from train.py's init vector by shifting one layer's biases (and shrinking a unit's weights where its
input range would not fit in the band) so that every unit's pre-activation lies in the band for ANY point: the inputs of
a layer are bounded (exp(-r) and sigmoids in [0, 1], R in the union of the two samplers' ranges [0.2, 4]), not only the
points sampled here (oracle/regimes.py).  The CPU test checks the bands with the float64 oracle on the points the GPU tests use.
"""
import ctypes
import os
import time

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf
from oracle import layout
from oracle import pointwise as pw
from oracle import ref_autograd as ra
from oracle.regimes import BAND, LAYERS, REGIMES, unit_signs, regime_theta

OFFS = layout.offsets() + [1521]
N = 4096 + 37                     # the last 128-point super-tile is ragged
SEED = 7


def sample(variant):
    g = torch.Generator().manual_seed(SEED + variant)
    x, y, z, R, i1, i2 = ra.sample_box(N, "poc" if variant == 0 else "trainpy", g)
    a32 = [v.numpy().ravel().astype(np.float32) for v in (x, y, z, R)]
    m1, m2 = np.zeros(N), np.zeros(N)
    m1[i1.numpy()] = 1
    m2[i2.numpy()] = 1
    return a32, m1, m2


def preactivations(theta, variant, a32):
    """Every sigmoid pre-activation (points x units) per layer, in float64; the poc form evaluates the base MLP twice,
    the second time with the two orbitals swapped."""
    P = layout.unpack_poc(np.asarray(theta, np.float64))
    x, y, z, R = [a.astype(np.float64) for a in a32]
    g = cf.geometry(x, y, z, R)
    ins = [(g["f1"], g["f2"])] + ([(g["f2"], g["f1"])] if variant == 0 else [])
    u1 = [np.stack(ab, 1) @ P[0].T + P[1] for ab in ins]
    u2 = [cf._sig(u) @ P[2].T + P[3] for u in u1]
    e1 = R[:, None] * P[6].reshape(-1) + P[7]
    return {"base_L1": np.concatenate(u1), "base_L2": np.concatenate(u2), "enet_L1": e1,
            "enet_L2": cf._sig(e1) @ P[8].T + P[9], "gate_L1": R[:, None] * P[12].reshape(-1) + P[13]}


@pytest.fixture(scope="module")
def init_theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]   # train.py's init rule, seed 12345


# ---------------------------------------------------------------------------------------------
# CPU: the regimes reach their bands
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("regime", sorted(REGIMES))
def test_regime_reaches_its_band(regime, variant, init_theta):
    th = regime_theta(init_theta, regime)
    u = preactivations(th, variant, sample(variant)[0])
    for layer, sign in REGIMES[regime].items():
        s = unit_signs(layer, sign)
        us = u[layer] * s                                      # folded onto the positive side
        assert us.min() >= BAND[0] and us.max() <= BAND[1], (layer, us.min(), us.max())
    for layer in set(LAYERS) - set(REGIMES[regime]):           # the other layers stay where the init put them
        assert np.abs(u[layer]).max() < BAND[0], layer


# ---------------------------------------------------------------------------------------------
# GPU: loss, gradient and fields in every regime
# ---------------------------------------------------------------------------------------------
def dev():
    return torch.device("cuda:0")


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def entry_rel(a, b):
    """Largest relative error over the entries with |b| >= 1e-2 max|b|."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    big = np.abs(b) >= 1e-2 * np.abs(b).max()
    return float((np.abs(a - b)[big] / np.abs(b)[big]).max()) if big.any() else 0.0


def run_gpu(variant, a32, th32, m1, m2, grad_mask=0xFFFF):
    w = torch.tensor([1.0 / N, 1.0 / m1.sum(), 1.0 / m2.sum()], dtype=torch.float64, device=dev())
    sums, dth, E = pk.loss_and_grad_raw(variant, *[t(a) for a in a32], t(th32), t((m1 + 2 * m2).astype(np.uint8)), w,
                                        grad_mask, want_E=True)
    torch.cuda.synchronize()
    return sums.cpu().numpy(), dth.cpu().numpy(), E.cpu().numpy()


def grad_errors(dth, ref, tensors=range(16)):
    return {layout.POC_TENSORS[i][0]: (rel(dth[OFFS[i]:OFFS[i + 1]], ref[OFFS[i]:OFFS[i + 1]]),
                                       entry_rel(dth[OFFS[i]:OFFS[i + 1]], ref[OFFS[i]:OFFS[i + 1]])) for i in tensors}


def report(tag, errs):
    worst_t = max(errs, key=lambda k: errs[k][0])
    worst_e = max(errs, key=lambda k: errs[k][1])
    print("\n%s: tensor %.2e (%s), entry %.2e (%s)" % (tag, errs[worst_t][0], worst_t, errs[worst_e][1], worst_e))
    for k, (et, ee) in errs.items():
        if et >= 1e-5 or ee >= 1e-4:
            print("    %-18s tensor %.2e  entry %.2e" % (k, et, ee))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("regime", ["init"] + sorted(REGIMES))
def test_step_and_fields_at_saturated_sigmoids(regime, variant, init_theta):
    th32 = init_theta.astype(np.float32) if regime == "init" else regime_theta(init_theta, regime)
    a32, m1, m2 = sample(variant)
    name = "poc" if variant == 0 else "trainpy"
    a64 = [a.astype(np.float64) for a in a32]
    ref = cf.loss_and_grad(name, th32.astype(np.float64), *a64, m1, m2)
    sums, dth, E = run_gpu(variant, a32, th32, m1, m2)
    errs = grad_errors(dth, ref["grad"])
    report("%s %s" % (regime, name), errs)
    out = pk.fields(variant, *[t(a) for a in a32], t(th32))
    torch.cuda.synchronize()
    f = cf.fields(name, th32.astype(np.float64), *a64)
    ferr = {k: rel(out[k].cpu().numpy(), f[k]) for k in ("psi", "lap", "res", "hpsi", "E")}
    lerr = {"Ltot": abs(sums[0] - ref["Ltot"]) / ref["Ltot"], "Lpde": abs(sums[1] - ref["Lpde"]) / ref["Lpde"],
            "Lbc": abs(sums[2] - ref["Lbc"]) / ref["Lbc"], "sumE": abs(sums[3] - ref["sums"]["E"]) / abs(ref["sums"]["E"]),
            "E": rel(E, ref["E"])}
    print("    losses " + " ".join("%s %.1e" % kv for kv in lerr.items()) + " | fields " +
          " ".join("%s %.1e" % kv for kv in ferr.items()))
    bad = {k: v for k, v in {**lerr, **ferr}.items() if not v < 1e-5}
    bad.update({k: v for k, v in errs.items() if not (v[0] < 1e-5 and v[1] < 1e-4)})
    assert not bad, bad
    pw.check("fields %s %s" % (regime, name), {k: out[k].cpu().numpy() for k in pw.OUTPUTS}, f,
             pw.magnitudes(name, th32.astype(np.float64), *a64), pw.C_KERNEL, a64)


@pytest.mark.gpu
def test_fine_tune_mask_at_saturated_enet(init_theta):
    """freezeBase + freezeDecayUnit with the E-net's second layer on the positive side: E-net gradients only, each as
    accurate as without the mask."""
    th32 = regime_theta(init_theta, "enet_L2_pos")
    a32, m1, m2 = sample(0)
    ref = cf.loss_and_grad("poc", th32.astype(np.float64), *[a.astype(np.float64) for a in a32], m1, m2)
    sums, dth, _ = run_gpu(0, a32, th32, m1, m2, grad_mask=pk.FINE_TUNE_GRAD_MASK)
    assert abs(sums[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    assert np.all(dth[:OFFS[6]] == 0) and np.all(dth[OFFS[12]:] == 0)
    errs = grad_errors(dth, ref["grad"], range(6, 12))
    report("enet_L2_pos poc, fine-tune mask", errs)
    assert all(et < 1e-5 and ee < 1e-4 for et, ee in errs.values()), errs


# ---------------------------------------------------------------------------------------------
# GPU: the dense-grid kernel past 2^31 points
# ---------------------------------------------------------------------------------------------
def _grid_reduce(nx, ny, nz, lim, R, wx, wy, wz, th):
    h = pk.Handle.get(0)
    out = torch.empty(8, dtype=torch.float64, device=dev())
    p = lambda a: ctypes.c_void_p(a.data_ptr())
    rc = h.L.pinn_grid_reduce(h.h, 0, p(th), nx, ny, nz, (ctypes.c_double * 6)(*lim), R, p(wx), p(wy), p(wz), p(out),
                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    h.check(rc, "pinn_grid_reduce")
    return out.cpu().numpy()


@pytest.mark.gpu
def test_grid_reduce_past_2_31_points(init_theta):
    """1320 x 1291 x 1283 = 2.19e9 points: indices from 2^31 on take the 64-bit branch of the index mapping, and index
    2^31 falls inside plane 1296.  Only the 30 planes 1290..1319 carry weight; they straddle x = 0 with the nuclei
    (R = 0.15) between two planes.  The same 30 planes as a grid of their own (same x positions bit for bit: dx = 1/64
    and the offsets are exact in binary) stay on the 32-bit branch, evaluate the same float32 terms, and must give the
    same sums up to the order of the double accumulation.  Distinct ny and nz catch a swapped iy / iz."""
    nx, ny, nz, x_lo, planes = 1320, 1291, 1283, 1290, 30
    assert (x_lo + planes) * ny * nz > 2 ** 31 > x_lo * ny * nz and nx == x_lo + planes
    assert 1296 * ny * nz <= 2 ** 31 < 1297 * ny * nz
    d = dev()
    th = t(init_theta.astype(np.float32))
    x0 = -1305 / 64                                          # x = (ix - 1305) / 64: planes 1290..1319 cover [-15, 14] / 64
    lim_all = (x0, x0 + (nx - 1) / 64, -18.0, 18.0, -17.0, 19.0)
    lim_slab = (x0 + x_lo / 64, x0 + (nx - 1) / 64) + lim_all[2:]
    assert (lim_all[1] - lim_all[0]) / (nx - 1) == 1 / 64 == (lim_slab[1] - lim_slab[0]) / (planes - 1)
    k = np.arange(max(ny, nz), dtype=np.float64)
    wy = t((36 / (ny - 1)) * (1.0 + 0.5 * np.cos(0.37 * k[:ny])))
    wz = t((36 / (nz - 1)) * (1.0 + 0.3 * np.sin(0.11 * k[:nz]) + 0.1 * (k[:nz] % 3)))
    wx_all = torch.zeros(nx, dtype=torch.float64, device=d)
    wx_all[x_lo:] = 1.0
    wx_slab = torch.ones(planes, dtype=torch.float64, device=d)
    ref = _grid_reduce(planes, ny, nz, lim_slab, 0.15, wx_slab, wy, wz, th)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = _grid_reduce(nx, ny, nz, lim_all, 0.15, wx_all, wy, wz, th)
    dt = time.perf_counter() - t0
    print("\npinn_grid_reduce, %d x %d x %d = %.3g points: %.3f s wall (%.3g points/s)" % (nx, ny, nz, nx * ny * nz, dt,
                                                                                        nx * ny * nz / dt))
    print("    sums " + " ".join("%.15e" % v for v in got[:5]) + "\n    slab " + " ".join("%.15e" % v for v in ref[:5]))
    assert np.all(np.isfinite(ref[:6])) and np.all(ref[[1, 3]] > 0)
    for i in range(5):
        assert abs(got[i] - ref[i]) <= 1e-12 * abs(ref[i]), (i, got[i], ref[i])
    assert got[5] == ref[5]
