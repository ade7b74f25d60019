"""pinn_fields point by point: every output within C u M of the float64 oracle (oracle/pointwise.py) at the edges of the
domain, the same bits whichever outputs are requested, at every launch shape and at 6.7e7 points, and the adaptive
pool's residual the same bits as pinn_fields past 2^22 candidates.  Each case runs both forms at trained and init
weights."""
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf
from oracle import pointwise as pw
from oracle import ref_autograd as ra
from pinn_for_quantum_wavefunction_surfaces_b200.ops import _F32, _F64, _ptr

pytestmark = pytest.mark.gpu
C = pw.C_KERNEL
NAMES = ("poc", "trainpy")
BLOCK = (1 << 16) + 37


@pytest.fixture(scope="module")
def thetas(golden_dir):
    ck = np.load(os.path.join(golden_dir, "checkpoints.npz"))
    init = np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]  # train.py's init rule, seed 12345
    return {"trained": ck["ionHsym"].astype(np.float32), "init": init.astype(np.float32)}


def fields_into(variant, cols, theta, outs):
    """pinn_fields on caller-owned columns: `outs` maps the requested outputs to float32 device tensors."""
    h = pk.Handle.get(0)
    code = _F64 if cols[0].dtype == torch.float64 else _F32
    th = torch.as_tensor(theta, dtype=torch.float32).cuda()
    h.check(h.L.pinn_fields(h.h, NAMES.index(variant), cols[0].numel(), *[_ptr(c) for c in cols], code, _ptr(th),
                            *[_ptr(outs.get(k)) for k in ("psi", "lap", "hpsi", "res", "E")],
                            torch.cuda.current_stream().cuda_stream), "pinn_fields")
    return outs


def run(variant, a, theta, want=pw.OUTPUTS):
    cols = [torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in a]
    outs = {k: torch.full((a[0].size,), float("nan"), device="cuda") for k in want}
    fields_into(variant, cols, theta, outs)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in outs.items()}


def check_vs_oracle(tag, variant, a, theta):
    a64 = [np.asarray(v, np.float64) for v in a]
    th64 = theta.astype(np.float64)
    pw.check(tag, run(variant, a, theta), cf.fields(variant, th64, *a64), pw.magnitudes(variant, th64, *a64), C,
             coords=a64)


# ---------------------------------------------------------------------------------------------
# edge points
# ---------------------------------------------------------------------------------------------
def edge_points(R):
    """Points 0.005 from each nucleus along several directions, on the molecular axis between and outside the nuclei,
    on the mid-plane x = 0, and on the faces and corners of the +-18 sampling box and of a +-20 box (r ~ 35)."""
    pts = []
    dirs = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, 0, -1], [1, 1, 1], [-1, 2, 0]], np.float64)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    for xn in (R, -R):
        pts += [np.array([xn, 0.0, 0.0]) + 0.005 * d for d in dirs]
    pts += [[R * f, 0.0, 0.0] for f in (-0.9, -0.5, -0.1, 0.0, 0.3, 0.7, 0.95)]
    pts += [[s * (R + d), 0.0, 0.0] for s in (1, -1) for d in (0.01, 0.5, 2.0, 10.0, 17.0)]
    pts += [[0.0, y, z] for y in (0.0, 0.01, 1.0, 7.5, -18.0) for z in (0.0, 0.3, -5.0, 18.0)]
    for L in (18.0, 20.0):
        pts += [[s * L, 0.0, 0.0] for s in (1, -1)] + [[0.0, s * L, 0.0] for s in (1, -1)] + [[0.0, 0.0, L]]
        pts += [[sx * L, sy * L, sz * L] for sx in (1, -1) for sy in (1, -1) for sz in (1, -1)]
        pts += [[L, L, 0.0], [-L, 0.0, L]]
    p = np.array(pts, np.float64)
    return [p[:, 0], p[:, 1], p[:, 2], np.full(len(p), R)]


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("which", ["trained", "init"])
@pytest.mark.parametrize("variant", NAMES)
def test_edge_points_within_the_bound(variant, which, dtype, thetas):
    # R = 0.2 and 4 bound the training range; 0.05, 6 and 10 lie outside it, which callers of fields can pass
    a = [np.concatenate(c) for c in zip(*[edge_points(R) for R in (0.2, 4.0, 0.05, 6.0, 10.0)])]
    a = [v.astype(np.float32) for v in a] if dtype == "f32" else a
    check_vs_oracle("edges %s %s %s" % (variant, which, dtype), variant, a, thetas[which])


# ---------------------------------------------------------------------------------------------
# output subsets, launch shapes, views
# ---------------------------------------------------------------------------------------------
def sample(variant, n, seed):
    x, y, z, R, _, _ = ra.sample_box(n, variant, torch.Generator().manual_seed(seed))
    return [v.numpy().ravel().astype(np.float32) for v in (x, y, z, R)]


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("which", ["trained", "init"])
@pytest.mark.parametrize("variant", NAMES)
def test_every_output_subset_gives_the_same_bits(variant, which, thetas):
    a = sample(variant, 3000, 21)
    full = run(variant, a, thetas[which])
    for want in [(k,) for k in pw.OUTPUTS] + [("res",), ("psi", "res"), ("lap", "hpsi", "E")]:
        got = run(variant, a, thetas[which], want)
        for k in want:
            assert np.array_equal(bits(got[k]), bits(full[k])), (want, k)


@pytest.mark.parametrize("which", ["trained", "init"])
@pytest.mark.parametrize("variant", NAMES)
def test_launch_shapes_and_views_give_the_block_s_bits(variant, which, thetas):
    nb = 2 * 148 * 128 + 5
    a = sample(variant, nb, 22)
    block = run(variant, a, thetas[which])
    check_vs_oracle("block %s %s" % (variant, which), variant, a, thetas[which])
    for n in (1, 31, 127, 128, 129, 148 * 128 - 1, 148 * 128, 148 * 128 + 1, nb):
        got = run(variant, [v[:n] for v in a], thetas[which])
        for k in pw.OUTPUTS:
            assert np.array_equal(bits(got[k]), bits(block[k][:n])), (n, k)
    for off in (1, 3):  # columns that start 4 and 12 bytes into an allocation
        n = 5000
        cols = []
        for v in a:
            base = torch.zeros(n + 8, dtype=torch.float32, device="cuda")
            base[off:off + n] = torch.from_numpy(v[:n]).cuda()
            cols.append(base[off:off + n])
        obase = {k: torch.full((n + 8,), float("nan"), device="cuda") for k in pw.OUTPUTS}
        fields_into(variant, cols, thetas[which], {k: v[off:off + n] for k, v in obase.items()})
        torch.cuda.synchronize()
        for k in pw.OUTPUTS:
            o = obase[k].cpu().numpy()
            assert np.array_equal(bits(o[off:off + n]), bits(block[k][:n])), (off, k)
            assert np.isnan(o[:off]).all() and np.isnan(o[off + n:]).all(), (off, k)


# ---------------------------------------------------------------------------------------------
# scale: K copies of one checked block
# ---------------------------------------------------------------------------------------------
def copies_equal_block(variant, a, theta, K, dtype):
    """fields over K copies of the block a plus its first 101 points again, outputs filled with NaN first: every copy
    equals the block bit for bit, compared on the device 64 copies at a time."""
    B = a[0].size
    n = K * B + 101
    cols = []
    for v in a:
        b = torch.from_numpy(np.asarray(v, dtype)).cuda()
        cols.append(torch.cat([b.repeat(K), b[:101]]))
    outs = {k: torch.full((n,), float("nan"), device="cuda") for k in pw.OUTPUTS}
    fields_into(variant, cols, theta, outs)
    block = fields_into(variant, [c[:B].clone() for c in cols], theta,
                        {k: torch.full((B,), float("nan"), device="cuda") for k in pw.OUTPUTS})
    for k in pw.OUTPUTS:
        o, ref = outs[k].view(torch.int32), block[k].view(torch.int32)
        for k0 in range(0, K, 64):
            k1 = min(K, k0 + 64)
            assert torch.equal(o[k0 * B:k1 * B].view(k1 - k0, B), ref.expand(k1 - k0, B)), (k, k0)
        assert torch.equal(o[K * B:], ref[:101]), k
    del outs, cols
    torch.cuda.empty_cache()
    return {k: v.cpu().numpy() for k, v in block.items()}


@pytest.mark.parametrize("which", ["trained", "init"])
@pytest.mark.parametrize("variant", NAMES)
def test_copies_of_a_checked_block_at_6_7e7_points(variant, which, thetas):
    a = sample(variant, BLOCK, 23)
    th = thetas[which]
    block = copies_equal_block(variant, a, th, 1024, np.float32)
    a64 = [v.astype(np.float64) for v in a]
    th64 = th.astype(np.float64)
    pw.check("scale block %s %s" % (variant, which), block, cf.fields(variant, th64, *a64),
             pw.magnitudes(variant, th64, *a64), C, coords=a64)
    # float64 coordinates: x -/+ R formed in float64 (the block's points moved off the float32 grid)
    rng = np.random.default_rng(5)
    a64 = [v + rng.uniform(-1e-7, 1e-7, v.size) * np.abs(v) for v in a64]
    block = copies_equal_block(variant, a64, th, 64, np.float64)
    pw.check("scale block f64 %s %s" % (variant, which), block, cf.fields(variant, th64, *a64),
             pw.magnitudes(variant, th64, *a64), C, coords=a64)


@pytest.mark.parametrize("which", ["trained", "init"])
@pytest.mark.parametrize("variant", NAMES)
def test_adaptive_pool_residual_past_2_22_is_the_fields_residual(variant, which, thetas):
    n = (1 << 20) + 5
    out = pk.sample_adaptive(variant, thetas[which], n, pool_factor=4, seed=9, batch=2)
    assert out["res"].numel() > 1 << 22
    f = pk.fields(variant, *[out["pool"][k] for k in "xyzR"], torch.from_numpy(thetas[which]).cuda(), want=("res",))
    assert torch.equal(out["res"].view(torch.int32), f["res"].view(torch.int32))
