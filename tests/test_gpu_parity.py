"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
(libpinn_b200.so via ctypes) and is compared with the float64 CPU oracle / golden reference outputs.

Tolerances (BASELINE.json north_star): psi, laplacian, residual: 1e-5 norm-relative
(max|a-b| / max|b|); loss: 1e-5 relative.  Parameter gradients: 1e-5 norm-relative per tensor at
generic (random-init) weights.  At the shipped *trained* weights the gradient is a cancelling sum
(|res| ~ 1e-3 of its terms, psi at the boundary ~2e-5 from O(0.1) terms), so ANY float32 evaluation
is limited there: torch's own float32 autograd reaches 1.4e-4 (measured, DESIGN.md).  The network sees (0, 0) at every
boundary point, so the error there is one fixed rounding pattern, not an average; the kernel is deterministic and
measures 3e-5 ... 4e-5 on these fixtures (DESIGN.md section 4); the bars below are 3x that.
"""
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf
from oracle import layout
from oracle import pointwise as pw
from oracle import ref_autograd as ra

pytestmark = pytest.mark.gpu

OFFS = layout.offsets() + [1521]


def dev():
    return torch.device("cuda:0")


TRAINED_GRAD_BAR = 1.2e-4   # gradient at the shipped trained weights: measured 3.7e-5 (module docstring) x 3
TRAINED_LBC_BAR = 1.5e-4    # Lbc ~ 9e-10 = psi^2 of a 2e-5 cancellation of O(0.1) terms: measured 4e-5 x 3


def test_one_engine_no_dispatch():
    """The library carries the tcgen05 engine only: asking for the FFMA engine is refused and changes nothing."""
    h = pk.Handle.get(0)
    assert h.get_engine() == "tcgen05"
    with pytest.raises(pk.PinnError):
        h.set_engine("ffma")
    assert h.get_engine() == "tcgen05"


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def masks(n, i1, i2):
    m1 = np.zeros(n)
    m2 = np.zeros(n)
    m1[np.asarray(i1)] = 1
    m2[np.asarray(i2)] = 1
    return m1, m2


def run_gpu(variant, a32, th32, m1, m2, weights="explicit", grad_mask=0xFFFF, dtype=np.float32, use_mask=True):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    n = a32[0].size
    mask = t((m1 + 2 * m2).astype(np.uint8)) if use_mask else None
    w = None
    if weights == "explicit":
        w = torch.tensor([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()], dtype=torch.float64, device=dev())
    sums, dth, E = pk.loss_and_grad_raw(variant, *[t(a.astype(dtype)) for a in a32], t(th32), mask, w, grad_mask,
                                        want_E=True)
    torch.cuda.synchronize()
    return sums.cpu().numpy(), dth.cpu().numpy(), E.cpu().numpy()


def sample(variant, n, seed):
    g = torch.Generator().manual_seed(seed)
    x, y, z, R, i1, i2 = ra.sample_box(n, "poc" if variant == 0 else "trainpy", g)
    a32 = [v.numpy().ravel().astype(np.float32) for v in (x, y, z, R)]
    m1, m2 = masks(n, i1.numpy(), i2.numpy())
    return a32, m1, m2


def oracle(variant, th32, a32, m1, m2, **kw):
    return cf.loss_and_grad("poc" if variant == 0 else "trainpy", th32.astype(np.float64),
                            *[a.astype(np.float64) for a in a32], m1, m2, **kw)


@pytest.fixture(scope="module")
def ck(golden_dir):
    return np.load(os.path.join(golden_dir, "checkpoints.npz"))


@pytest.fixture(scope="module")
def init_theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]  # train.py's init rule, seed 12345


def check_tensors(dth, ref, tol):
    for i, (nm, _) in enumerate(layout.POC_TENSORS):
        a, b = dth[OFFS[i]:OFFS[i + 1]], ref[OFFS[i]:OFFS[i + 1]]
        assert rel(a, b) < tol, (nm, rel(a, b))


# ---------------------------------------------------------------------------------------------
def test_golden_reference_outputs_poc(golden_dir, ck):
    """CUDA path vs outputs of the REAL reference (NN_ion.LossFunctions + backward, fp64) on its own points."""
    g = np.load(os.path.join(golden_dir, "poc_seed0_n4096.npz"))
    n = g["x"].size
    m1, m2 = masks(n, g["i1"], g["i2"])
    a64 = [g[k] for k in "xyzR"]
    for tag in ("ionHsym", "ionHsym_fineTune"):
        th32 = ck[tag].astype(np.float32)
        sums, dth, E = run_gpu(0, a64, th32, m1, m2, dtype=np.float64)  # float64 coordinates, as the reference holds them
        ref = g[tag + "_loss"]
        assert abs(sums[0] - ref[0]) / ref[0] < 1e-5
        assert abs(sums[1] - ref[1]) / ref[1] < 1e-5
        # Lbc ~ 9e-10: psi^2 of a 2e-5 cancellation of O(0.1) terms, fp32-limited
        assert abs(sums[2] - ref[2]) / ref[2] < TRAINED_LBC_BAR
        assert rel(E, g[tag + "_E"]) < 1e-5
        assert rel(dth, g[tag + "_grad"]) < TRAINED_GRAD_BAR
        t = lambda a: torch.from_numpy(a).to(dev())
        f = pk.fields("poc", *[t(a) for a in a64], t(th32))
        torch.cuda.synchronize()
        assert rel(f["psi"].cpu().numpy(), g[tag + "_psi"]) < 1e-5
        assert rel(f["lap"].cpu().numpy(), g[tag + "_lap"]) < 1e-5
        assert rel(f["hpsi"].cpu().numpy(), g[tag + "_hpsi"]) < 1e-5
        assert rel(f["E"].cpu().numpy(), g[tag + "_E"]) < 1e-5
        keys = ("psi", "lap", "hpsi", "E")
        pw.check("golden poc " + tag, {k: f[k].cpu().numpy() for k in keys}, {k: g[tag + "_" + k] for k in keys},
                 pw.magnitudes("poc", ck[tag], *a64, rounded_weights=True), pw.C_KERNEL, a64)


def test_golden_reference_outputs_trainpy(golden_dir):
    """CUDA path vs outputs of the reference's own train.py lines 41-57 (+ backward) at its init weights."""
    g = np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))
    n = g["x"].size
    m1, m2 = masks(n, g["i1"], g["i2"])
    sums, dth, E = run_gpu(1, [g[k] for k in "xyzR"], g["theta"].astype(np.float32), m1, m2, dtype=np.float64)
    for k in range(3):
        assert abs(sums[k] - g["loss"][k]) / g["loss"][k] < 1e-5
    assert rel(E, g["e"]) < 1e-5
    check_tensors(dth, g["grad"], 1e-5)
    t = lambda a: torch.from_numpy(a).to(dev())
    f = pk.fields("trainpy", *[t(g[k]) for k in "xyzR"], t(g["theta"]))
    assert rel(f["psi"].cpu().numpy(), g["psi"]) < 1e-5
    assert rel(f["res"].cpu().numpy(), g["res"]) < 1e-5
    a64 = [g[k] for k in "xyzR"]
    pw.check("golden trainpy", {k: f[k].cpu().numpy() for k in ("psi", "res")}, {k: g[k].reshape(-1) for k in ("psi", "res")},
             pw.magnitudes("trainpy", g["theta"], *a64, rounded_weights=True), pw.C_KERNEL, a64)


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000, 20000])
def test_loss_and_grad_vs_oracle_ragged_sizes(variant, n, init_theta):
    a32, m1, m2 = sample(variant, max(n, 64), 100 + n)
    a32, m1, m2 = [a[:n] for a in a32], m1[:n], m2[:n]
    m1[0] = 1  # keep both boundary sets non-empty
    m2[0] = 1
    th32 = init_theta.astype(np.float32)
    ref = oracle(variant, th32, a32, m1, m2)
    sums, dth, E = run_gpu(variant, a32, th32, m1, m2)
    assert abs(sums[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    assert abs(sums[1] - ref["Lpde"]) / ref["Lpde"] < 1e-5
    assert abs(sums[2] - ref["Lbc"]) / ref["Lbc"] < 1e-5
    assert abs(sums[3] - ref["sums"]["E"]) < 1e-5 * abs(ref["sums"]["E"])
    assert rel(E, ref["E"]) < 1e-5
    assert abs(sums[7] - ref["E"][-1]) < 1e-5
    check_tensors(dth, ref["grad"], 1e-5)


def test_trained_weights_vs_oracle(ck):
    a32, m1, m2 = sample(0, 8192, 3)
    th32 = ck["ionHsym"].astype(np.float32)
    ref = oracle(0, th32, a32, m1, m2)
    sums, dth, E = run_gpu(0, a32, th32, m1, m2)
    assert abs(sums[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    assert abs(sums[1] - ref["Lpde"]) / ref["Lpde"] < 1e-5
    assert rel(dth, ref["grad"]) < TRAINED_GRAD_BAR  # fp32 cancellation limit, see module docstring
    # E-net and gate gradients do not pass through the cancelling output layer: tight
    for i in range(6, 16):
        assert rel(dth[OFFS[i]:OFFS[i + 1]], ref["grad"][OFFS[i]:OFFS[i + 1]]) < 2e-5


@pytest.mark.parametrize("variant", [0, 1])
def test_fields_vs_oracle(variant, ck, init_theta):
    for th in (ck["ionHsym"], init_theta):
        a32, _, _ = sample(variant, 30000, 11)
        th32 = th.astype(np.float32)
        f = cf.fields("poc" if variant == 0 else "trainpy", th32.astype(np.float64), *[a.astype(np.float64) for a in a32])
        t = lambda a: torch.from_numpy(a).to(dev())
        out = pk.fields(variant, *[t(a) for a in a32], t(th32))
        torch.cuda.synchronize()
        got = {k: out[k].cpu().numpy() for k in pw.OUTPUTS}
        for k in pw.OUTPUTS:
            assert rel(got[k], f[k]) < 1e-5, (k, rel(got[k], f[k]))
        a64 = [a.astype(np.float64) for a in a32]
        name = "poc" if variant == 0 else "trainpy"
        pw.check("fields %s" % name, got, f, pw.magnitudes(name, th32.astype(np.float64), *a64), pw.C_KERNEL, a64)


def test_points_at_the_clamp_distance(init_theta):
    """x[r<cutOff]=cutOff (poc/main.py:147-149): points 0.005 from a nucleus, 1/r = 200."""
    n = 64
    R = np.linspace(0.2, 4.0, n).astype(np.float32)
    x = (R + np.float32(0.005)).astype(np.float32)
    x[n // 2:] = -(R[n // 2:] + np.float32(0.005))
    y = np.zeros(n, np.float32)
    z = np.zeros(n, np.float32)
    m1 = np.zeros(n); m2 = np.zeros(n); m1[0] = m2[1] = 1
    th32 = init_theta.astype(np.float32)
    # coordinates in float64 so that x-R keeps its digits (the kernel forms the difference in double)
    a64 = [v.astype(np.float64) for v in (x, y, z, R)]
    ref = cf.loss_and_grad("poc", th32.astype(np.float64), *a64, m1, m2)
    sums, dth, E = run_gpu(0, a64, th32, m1, m2, dtype=np.float64)
    assert abs(sums[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    check_tensors(dth, ref["grad"], 2e-5)


def test_f64_and_f32_inputs_agree(init_theta):
    a32, m1, m2 = sample(0, 5000, 21)
    th32 = init_theta.astype(np.float32)
    s32, g32, _ = run_gpu(0, a32, th32, m1, m2, dtype=np.float32)
    s64, g64, _ = run_gpu(0, a32, th32, m1, m2, dtype=np.float64)
    assert abs(s32[0] - s64[0]) / s64[0] < 1e-6 and rel(g32, g64) < 1e-5


def test_in_kernel_sets_and_counted_weights_match_explicit_mask(init_theta):
    """mask=NULL: sets from r>=17.5 in the kernel; weights=NULL: 1/n, 1/count from the count kernel."""
    a32, m1, m2 = sample(0, 10000, 31)
    # recompute the sets in float32 exactly as the kernel does, away from the threshold
    th32 = init_theta.astype(np.float32)
    s_a, g_a, _ = run_gpu(0, a32, th32, m1, m2, weights="explicit", use_mask=True)
    s_b, g_b, _ = run_gpu(0, a32, th32, m1, m2, weights=None, use_mask=False)
    assert abs(s_a[0] - s_b[0]) / s_a[0] < 1e-6 and rel(g_b, g_a) < 1e-5


def test_fine_tune_grad_mask(ck):
    """freezeBase + freezeDecayUnit (poc/main.py:305-319): only the E-net tensors get gradients."""
    a32, m1, m2 = sample(0, 4096, 41)
    th32 = ck["ionHsym_fineTune"].astype(np.float32)
    ref = oracle(0, th32, a32, m1, m2)
    sums, dth, _ = run_gpu(0, a32, th32, m1, m2, grad_mask=pk.FINE_TUNE_GRAD_MASK)
    assert abs(sums[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    assert np.all(dth[:OFFS[6]] == 0) and np.all(dth[OFFS[12]:] == 0)
    assert rel(dth[OFFS[6]:OFFS[12]], ref["grad"][OFFS[6]:OFFS[12]]) < 2e-5


def test_deterministic_and_shard_additive_at_full_size(init_theta):
    """2^18 points (BASELINE config 3): run-to-run bit-identical; two shards with global weights add up to
    the whole (the data-parallel contract); a permutation of the points changes nothing beyond round-off."""
    n = 1 << 18
    a32, m1, m2 = sample(0, n, 51)
    th32 = init_theta.astype(np.float32)
    s1, g1, _ = run_gpu(0, a32, th32, m1, m2)
    s2, g2, _ = run_gpu(0, a32, th32, m1, m2)
    assert np.array_equal(s1, s2) and np.array_equal(g1, g2)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    w = torch.tensor([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()], dtype=torch.float64, device=dev())
    tot_s, tot_g = 0.0, 0.0
    for sl in (slice(0, 100003), slice(100003, n)):
        mk = t((m1[sl] + 2 * m2[sl]).astype(np.uint8))
        s, g, _ = pk.loss_and_grad_raw(0, *[t(a[sl]) for a in a32], t(th32), mk, w)
        tot_s = tot_s + s.cpu().numpy()[:7]
        tot_g = tot_g + g.cpu().numpy()
    assert np.allclose(tot_s, s1[:7], rtol=1e-6)
    assert rel(tot_g, g1) < 1e-5
    perm = np.random.default_rng(0).permutation(n)
    s3, g3, _ = run_gpu(0, [a[perm] for a in a32], th32, m1[perm], m2[perm])
    assert abs(s3[0] - s1[0]) / s1[0] < 1e-6 and rel(g3, g1) < 1e-5
    # and the loss agrees with the float64 oracle on a CPU-sized subsample scaled by the same weights
    sub = slice(0, 20000)
    ref = oracle(0, th32, [a[sub] for a in a32], m1[sub], m2[sub], w_pde=1.0 / n, w_bc1=1.0 / m1.sum(),
                 w_bc2=1.0 / m2.sum())
    mk = t((m1[sub] + 2 * m2[sub]).astype(np.uint8))
    s, g, _ = pk.loss_and_grad_raw(0, *[t(a[sub]) for a in a32], t(th32), mk, w)
    assert abs(s.cpu().numpy()[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    check_tensors(g.cpu().numpy(), ref["grad"], 1e-5)


class TinyIon(torch.nn.Module):
    """Same 16 parameters / names / init as the reference's NN_ion (poc/main.py:223-245); test-local."""

    def __init__(self):
        super().__init__()
        L = torch.nn.Linear
        self.Lin_H1, self.Lin_H2, self.Lin_out = L(2, 16), L(16, 16), L(16, 1)
        self.Lin_E1, self.Lin_E2, self.Lin_Eout = L(1, 32), L(32, 32), L(32, 1)
        torch.nn.init.constant_(self.Lin_Eout.bias[0], -1)
        self.netDecayL, self.netDecay = L(1, 10), L(10, 1)


@pytest.mark.parametrize("where", ["cuda", "cpu"])
def test_autograd_function_drives_adam_like_the_reference_loop(where):
    """3 Adam steps (poc/main.py:394-404) with the fused LossFunctions vs the float64 autograd oracle.
    `cpu` exercises the host-buffer entry (pinn_loss_fwd_bwd_host) the unmodified CPU reference loop would use."""
    torch.manual_seed(5)
    dt = torch.float64
    m_ref = TinyIon().to(dt)
    m_gpu = TinyIon().to(dt)
    m_gpu.load_state_dict(m_ref.state_dict())
    if where == "cuda":
        m_gpu = m_gpu.to(dev())
    pk.patch_nn_ion(TinyIon)
    o_ref = torch.optim.Adam(m_ref.parameters(), lr=8e-3)
    o_gpu = torch.optim.Adam(m_gpu.parameters(), lr=8e-3)
    g = torch.Generator().manual_seed(9)
    for step in range(3):
        x, y, z, R, i1, i2 = ra.sample_box(3000, "poc", g)
        x, y, z, R = [v.float().double() for v in (x, y, z, R)]
        b1 = (i1, torch.zeros_like(i1))  # torch.where tuples on an (n,1) tensor (poc/main.py:392-393)
        b2 = (i2, torch.zeros_like(i2))
        o_ref.zero_grad()
        theta = torch.cat([p.detach().reshape(-1) for p in m_ref.parameters()])
        Lt, Lp, Lb, E, gr = ra.loss_and_grad("poc", theta, x, y, z, R, i1, i2)
        for p, gpart in zip(m_ref.parameters(), [torch.tensor(a) for a in layout.unpack_poc(gr.numpy())]):
            p.grad = gpart.reshape(p.shape).clone()
        o_ref.step()
        o_gpu.zero_grad()
        mv = (lambda v: v.to(dev())) if where == "cuda" else (lambda v: v)
        Ltot, LossPDE, Lbc, Eo = m_gpu.LossFunctions(mv(x), mv(y), mv(z), mv(R), {"BCcutoff": 17.5}, b1, b2)
        assert Ltot.dtype == dt and Eo.shape == (3000, 1)
        assert abs(Ltot.item() - Lt.item()) / Lt.item() < 1e-5
        assert abs(Lbc.item() - Lb.item()) / Lb.item() < 1e-5
        assert abs(Eo[-1].item() - E[-1].item()) < 1e-5
        Ltot.backward()
        o_gpu.step()
    for a, b in zip(m_gpu.parameters(), m_ref.parameters()):
        assert torch.allclose(a.detach().cpu(), b.detach(), atol=2e-5), (a.detach().cpu() - b.detach()).abs().max()


def test_trainpy_function_cpu_tensors(init_theta):
    """PinnLossTrainPy.apply with train.py-shaped CPU float64 tensors (in,out layout, gate before E-net)."""
    tp = [torch.tensor(a, requires_grad=True) for a in layout.to_trainpy(init_theta)]
    a32, m1, m2 = sample(1, 2500, 61)
    x, y, z, R = [torch.tensor(a.astype(np.float64)).reshape(-1, 1) for a in a32]
    i1, i2 = torch.tensor(np.nonzero(m1)[0]), torch.tensor(np.nonzero(m2)[0])
    Ltot, Lpde, Lbc, e = pk.loss_trainpy(x, y, z, R, i1, i2, *tp)
    Ltot.backward()
    ref = oracle(1, init_theta, a32, m1, m2)
    assert abs(Ltot.item() - ref["Ltot"]) / ref["Ltot"] < 1e-5
    assert abs(torch.mean(e).item() - ref["E"].mean()) < 1e-5
    got = layout.from_trainpy([p.grad.numpy() for p in tp])
    check_tensors(got, ref["grad"], 1e-5)
    assert tp[0].grad.shape == (2, 16) and tp[2].grad.shape == (16, 16)


@pytest.mark.parametrize("order", ["poc", "trainpy"])
@pytest.mark.parametrize("pdt", [torch.float64, torch.float32])
def test_tensor_pointer_entry_equals_packed_entry(init_theta, order, pdt):
    """pinn_loss_fwd_bwd_tensors (the kernel gathers the caller's 16 tensors through their pointers, takes the weights by
    value, writes E in the parameter dtype and the gradient in the parameter layout) == pinn_loss_fwd_bwd on the packed
    float32 vector: the same bits."""
    import ctypes
    variant = 0 if order == "poc" else 1
    n = 5000
    a32, m1, m2 = sample(variant, n, 17)
    d = dev()
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(d)
    th = init_theta if pdt == torch.float64 else init_theta.astype(np.float32).astype(np.float64)
    parts = layout.unpack_poc(th) if order == "poc" else layout.to_trainpy(th)
    params = [torch.tensor(np.ascontiguousarray(a), dtype=pdt, device=d) for a in parts]
    mk = t((m1 + 2 * m2).astype(np.uint8))
    w = [1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()]
    cols = [t(a) for a in a32]
    s0, g0, E0 = pk.loss_and_grad_raw(variant, *cols, t(th.astype(np.float32)), mk, torch.tensor(w, dtype=torch.float64, device=d),
                                      want_E=True)
    h = pk.Handle.get(0)
    out = torch.empty(8 + 1521, dtype=torch.float64, device=d)
    E1 = torch.empty(n, dtype=pdt, device=d)
    ptrs = (ctypes.c_void_p * 16)(*[p.data_ptr() for p in params])
    code = {torch.float32: 0, torch.float64: 1}
    rc = h.L.pinn_loss_fwd_bwd_tensors(h.h, variant, n, *[c.data_ptr() for c in cols], 0, mk.data_ptr(), ptrs, code[pdt], variant,
                                       (ctypes.c_double * 3)(*w), 0xFFFF, 17.5, out.data_ptr(), out.data_ptr() + 64, E1.data_ptr(),
                                       code[pdt], torch.cuda.current_stream().cuda_stream)
    h.check(rc, "pinn_loss_fwd_bwd_tensors")
    torch.cuda.synchronize()
    assert torch.equal(out[:8], s0) and torch.equal(E1.float(), E0)
    g1 = out[8:].cpu().numpy()
    if order == "trainpy":   # canonical tensor order, each tensor in (in,out) layout -> back to (out,in)
        back = []
        for i, (nm, shp) in enumerate(layout.POC_TENSORS):
            blk = g1[OFFS[i]:OFFS[i + 1]]
            back.append(blk.reshape(shp[::-1]).T.ravel() if len(shp) == 2 else blk)
        g1 = np.concatenate(back)
    assert np.array_equal(g1, g0.cpu().numpy())


def test_mask_from_index_sets_and_its_cache():
    n = 10007
    rng = np.random.default_rng(5)
    i1 = torch.tensor(np.sort(rng.choice(n, 4000, replace=False)), device=dev())
    i2 = torch.tensor(np.sort(rng.choice(n, 5000, replace=False)), device=dev())
    ref, c1, c2 = pk.indices_to_mask(n, (i1, torch.zeros_like(i1)), i2, dev())
    h = pk.Handle.get(0)
    st = torch.cuda.current_stream().cuda_stream
    got = pk.ops._mask_cache.get(h, n, i1, i2, dev(), st)[:n]
    assert torch.equal(got, ref) and (c1, c2) == (4000, 5000)
    again = pk.ops._mask_cache.get(h, n, i1, i2, dev(), st)
    assert again.data_ptr() == got.data_ptr()                       # unchanged index tensors: reused
    i1[5:] = torch.flip(i1[5:], [0])                                 # an in-place edit bumps the tensor's version
    fresh = pk.ops._mask_cache.get(h, n, i1, i2, dev(), st)
    assert fresh.data_ptr() != got.data_ptr()
    assert torch.equal(fresh[:n], pk.indices_to_mask(n, i1, i2, dev())[0])
    empty = torch.empty(0, dtype=torch.long, device=dev())
    m = pk.ops._mask_cache.get(h, 5, empty, torch.tensor([4], device=dev()), dev(), st)[:5]
    assert m.tolist() == [0, 0, 0, 0, 2]


def test_trainpy_function_cuda_tensors(init_theta):
    """PinnLossTrainPy.apply on CUDA float64 tensors: the direct-pointer path with train.py's order and (in,out) layout."""
    tp = [torch.tensor(a, device=dev(), requires_grad=True) for a in layout.to_trainpy(init_theta)]
    a32, m1, m2 = sample(1, 2500, 61)
    x, y, z, R = [torch.tensor(a.astype(np.float64), device=dev()).reshape(-1, 1) for a in a32]
    i1, i2 = torch.tensor(np.nonzero(m1)[0], device=dev()), torch.tensor(np.nonzero(m2)[0], device=dev())
    Ltot, Lpde, Lbc, e = pk.loss_trainpy(x, y, z, R, i1, i2, *tp)
    (3.0 * Ltot).backward()
    ref = oracle(1, init_theta, a32, m1, m2)
    assert Ltot.dtype == torch.float64 and e.dtype == torch.float64 and e.shape == (2500, 1)
    assert abs(Ltot.item() - ref["Ltot"]) / ref["Ltot"] < 1e-5
    assert abs(torch.mean(e).item() - ref["E"].mean()) < 1e-5
    got = layout.from_trainpy([p.grad.cpu().numpy() / 3.0 for p in tp])
    check_tensors(got, ref["grad"], 1e-5)
    assert tp[0].grad.shape == (2, 16) and tp[2].grad.shape == (16, 16)
    # a frozen tensor gets no gradient and does not disturb the others
    tp2 = [p.detach().clone().requires_grad_(k not in (0, 2)) for k, p in enumerate(tp)]
    L2 = pk.loss_trainpy(x, y, z, R, i1, i2, *tp2)[0]
    L2.backward()
    assert tp2[0].grad is None and tp2[2].grad is None and torch.allclose(tp2[1].grad * 3.0, tp[1].grad, rtol=1e-12)


def test_calls_on_different_streams_of_one_handle_do_not_share_scratch(init_theta):
    """Every stream that calls in gets its own workspace (per-CTA partial rows, set counters): evaluations enqueued on two
    streams at once - they do overlap on the device - return what they return alone."""
    d = dev()
    th = torch.from_numpy(init_theta.astype(np.float32)).to(d)
    jobs = []
    for k, n in enumerate((1 << 17, 50000, 1 << 16, 77777)):
        a32, m1, m2 = sample(0, n, 200 + k)
        jobs.append([torch.from_numpy(a).to(d) for a in a32])
    alone = []
    for cols in jobs:
        s, g, _ = pk.loss_and_grad_raw(0, *cols, th)          # weights = None: the set-count kernels use the workspace too
        alone.append((s.clone(), g.clone()))
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in jobs]
    for rep in range(5):
        res = []
        for cols, st in zip(jobs, streams):
            with torch.cuda.stream(st):
                res.append(pk.loss_and_grad_raw(0, *cols, th))
        torch.cuda.synchronize()
        for (s, g, _), (s0, g0) in zip(res, alone):
            assert torch.equal(s[:7], s0[:7]) and torch.equal(g, g0)


def test_roofline_measurement_helpers(init_theta):
    """bench.py's denominators are measured by the library in the run: the FFMA rate of the device and the SM clock the
    step kernel and the FFMA loop actually ran at (block 0 times itself)."""
    h = pk.Handle.get(0)
    flops, ms, mhz = h.measure_fp32_peak()
    assert 55e12 < flops < 76e12 and 0.4 < ms < 0.8 and 1500 < mhz < 2100      # 148 SMs x 128 lanes x 2 x 1.965 GHz = 74.4e12
    a32, m1, m2 = sample(0, 1 << 16, 5)
    d = dev()
    pk.loss_and_grad_raw(0, *[torch.from_numpy(a).to(d) for a in a32], torch.from_numpy(init_theta.astype(np.float32)).to(d))
    assert 1200 < h.step_kernel_clock(torch.cuda.current_stream().cuda_stream) < 2100


def test_empty_boundary_set_gives_nan_like_the_reference(init_theta):
    """mean over an empty selection is NaN in the reference (poc/main.py:349-350); same here."""
    tp = [torch.tensor(a, requires_grad=True) for a in layout.to_trainpy(init_theta)]
    x = torch.zeros(64, 1, dtype=torch.float64) + 0.3
    R = torch.ones(64, 1, dtype=torch.float64)
    Ltot, Lpde, Lbc, e = pk.loss_trainpy(x, x, x, R, torch.tensor([], dtype=torch.long), torch.tensor([1]), *tp)
    assert torch.isnan(Ltot) and torch.isnan(Lbc) and torch.isfinite(Lpde)


def test_argument_errors_do_not_crash(init_theta):
    h = pk.Handle.get(0)
    with pytest.raises(pk.PinnError):
        h.check(h.L.pinn_loss_fwd_bwd(h.h, 7, 10, None, None, None, None, 0, None, None, None, 0xFFFF, 17.5, None,
                                      None, None, None), "bad variant")
    with pytest.raises(pk.PinnError):
        h.check(h.L.pinn_fields(h.h, 0, 0, None, None, None, None, 0, None, None, None, None, None, None, None), "n=0")
    assert h.launch_count() >= 0


# ---------------------------------------------------------------------------------------------
# pointer alignment and host-memory paths of the coordinate stage (cp.async one super-tile ahead)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("off", [1, 2, 3])
def test_unaligned_views_of_coordinates_mask_and_theta(init_theta, off):
    """x,y,z,R only 4-byte aligned, the mask at an odd byte address (the kernel fetches the aligned word around each
    mask byte), theta off the 16-byte boundary the TMA bulk copy wants (plain-load fallback): same bits as aligned."""
    n = 3000 + off
    a32, m1, m2 = sample(0, n, 71)
    th32 = init_theta.astype(np.float32)
    d = dev()
    w = torch.tensor([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()], dtype=torch.float64, device=d)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(d)
    mk = (m1 + 2 * m2).astype(np.uint8)
    s0, g0, _ = pk.loss_and_grad_raw(0, *[t(a) for a in a32], t(th32), t(mk), w)

    def shifted(a, k):
        buf = torch.zeros(a.size + 8, dtype=torch.from_numpy(a[:1]).dtype, device=d)
        buf[k:k + a.size] = t(a)
        v = buf[k:k + a.size]
        assert v.data_ptr() % 16 != 0 or a.dtype == np.uint8
        return v

    s1, g1, _ = pk.loss_and_grad_raw(0, *[shifted(a, off) for a in a32], shifted(th32, off), shifted(mk, off), w)
    assert torch.equal(s0[:7], s1[:7]) and torch.equal(g0, g1)
    ref = oracle(0, th32, a32, m1, m2)
    assert abs(s1.cpu().numpy()[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_entry_pinned_in_place_equals_staged_pageable(init_theta, dtype):
    """pinn_loss_fwd_bwd_host: page-locked inputs are read by the kernel in place over PCIe, pageable ones are staged
    (one copy below 8 rounds of super-tiles, 4 overlapped chunks above): same results, explicit mask and derived sets,
    float32 and float64 coordinates."""
    import ctypes
    h = pk.Handle.get(0)
    for n in (5000, 200000):
        a32, m1, m2 = sample(0, n, 81)
        cols = [torch.from_numpy(a.astype(dtype)) for a in a32]
        mk = torch.from_numpy((m1 + 2 * m2).astype(np.uint8))
        th64 = init_theta.astype(np.float32).astype(np.float64)
        wv = np.array([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()])
        P = lambda a: ctypes.c_void_p(a.ctypes.data)
        TP = lambda x: ctypes.c_void_p(x.data_ptr())
        res = {}
        for mode in ("pageable", "pinned"):
            c = [x.pin_memory() for x in cols] if mode == "pinned" else cols
            m = mk.pin_memory() if mode == "pinned" else mk
            for use_mask in (True, False):
                sums, dth = np.zeros(8), np.zeros(1521)
                rc = h.L.pinn_loss_fwd_bwd_host(h.h, 0, n, TP(c[0]), TP(c[1]), TP(c[2]), TP(c[3]), 1 if dtype == np.float64 else 0,
                                                TP(m) if use_mask else None, P(th64), P(wv), 0xFFFF, 17.5, P(sums), P(dth), None)
                h.check(rc, "pinn_loss_fwd_bwd_host")
                res[(mode, use_mask)] = (sums.copy(), dth.copy())
        for use_mask in (True, False):
            sa, ga = res[("pageable", use_mask)]
            sb, gb = res[("pinned", use_mask)]
            if n < 100000:   # one launch either way: identical bits; chunked staging only changes the summation order
                assert np.array_equal(sa[:7], sb[:7]) and np.array_equal(ga, gb)
            else:
                assert np.allclose(sa[:7], sb[:7], rtol=2e-6) and rel(ga, gb) < 1e-5
        assert abs(res[("pinned", True)][0][0] - res[("pinned", False)][0][0]) / res[("pinned", True)][0][0] < 1e-6
        if n <= 5000:
            ref = oracle(0, init_theta.astype(np.float32), a32, m1, m2)
            assert abs(res[("pinned", True)][0][0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
            check_tensors(res[("pinned", True)][1], ref["grad"], 1e-5)


def test_prepared_host_step_equals_the_plain_host_call(init_theta):
    """ops.HostStep (arguments bound once) against the float64 oracle and against loss_trainpy on the same CPU tensors."""
    a32, m1, m2 = sample(1, 3000, 91)
    cols = [torch.from_numpy(a.astype(np.float64)).pin_memory() for a in a32]
    mk = torch.from_numpy((m1 + 2 * m2).astype(np.uint8)).pin_memory()
    step = pk.HostStep("trainpy", *cols, mask=mk)
    th64 = np.ascontiguousarray(init_theta.astype(np.float32).astype(np.float64))
    w = np.array([1.0 / 3000, 1.0 / m1.sum(), 1.0 / m2.sum()])
    ref = oracle(1, init_theta.astype(np.float32), a32, m1, m2)
    for _ in range(3):   # the output arrays are reused
        sums, dth = step(th64, w)
        assert abs(sums[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
        check_tensors(dth, ref["grad"], 1e-5)
    s2, d2 = pk.HostStep("trainpy", *cols)(th64)     # sets and weights derived on the device
    assert abs(s2[0] - ref["Ltot"]) / ref["Ltot"] < 1e-5
    t = pk.Handle.get(0).host_timing()
    assert t["total"] > 0 and abs(t["enqueue"] + t["wait"] + t["copy_out"] - t["total"]) < 1.0


def test_bench_dumps_what_its_last_timed_step_computed(tmp_path):
    """bench.py --dump-outputs: loss.npy, dtheta.npy and sums.npy are, bit for bit, the evaluation of the batch the last
    of the --steps timed steps used (the timed region starts on batch 0 whatever the spin-up took), so that two builds run
    with the same arguments can be compared output for output."""
    import json
    import subprocess
    import sys
    import bench    # the repository root is on sys.path (tests/conftest.py)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from pinn_for_quantum_wavefunction_surfaces_b200 import dp
    n, steps = 4096, 7
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                        "--points", str(n), "--no-extras", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    loss, sums, dth = (np.load(tmp_path / (k + ".npy")) for k in ("loss", "sums", "dtheta"))
    assert loss.dtype == sums.dtype == dth.dtype == np.float64
    assert loss.shape == (3,) and sums.shape == (8,) and dth.shape == (1521,) and np.array_equal(loss, sums[:3])
    b = bench.synth_batch(n, (steps - 1) % bench.N_BATCHES)
    r1 = torch.sqrt((b[0] - b[3]) ** 2 + b[1] ** 2 + b[2] ** 2)
    r2 = torch.sqrt((b[0] + b[3]) ** 2 + b[1] ** 2 + b[2] ** 2)
    w = dp.global_weights(n, int((r1 >= 17.5).sum()), int((r2 >= 17.5).sum()), device=dev())
    theta = torch.from_numpy(bench.load_theta().astype(np.float32)).to(dev())
    s, g, _ = pk.loss_and_grad_raw(0, *[b[k].contiguous().to(dev()) for k in range(4)], theta, None, w)
    assert np.array_equal(sums, s.cpu().numpy()) and np.array_equal(dth, g.cpu().numpy())
