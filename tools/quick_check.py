"""Ad-hoc GPU check: parity per tensor at random-init and trained weights + raw kernel timing."""
import os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf, layout, ref_autograd as ra

dev = torch.device("cuda:0")
gd = os.path.join(ROOT, "tests", "golden")
names = [n for n, _ in layout.POC_TENSORS]
offs = layout.offsets() + [1521]

def case(variant, theta, n, seed):
    g = torch.Generator().manual_seed(seed)
    x, y, z, R, i1, i2 = ra.sample_box(n, "poc" if variant == 0 else "trainpy", g)
    a32 = [t.numpy().ravel().astype(np.float32) for t in (x, y, z, R)]
    th32 = theta.astype(np.float32)
    m1 = np.zeros(n); m1[i1.numpy()] = 1
    m2 = np.zeros(n); m2[i2.numpy()] = 1
    ref = cf.loss_and_grad("poc" if variant == 0 else "trainpy", th32.astype(np.float64), *[a.astype(np.float64) for a in a32], m1, m2)
    t = lambda a: torch.from_numpy(a).to(dev)
    mask = t((m1 + 2 * m2).astype(np.uint8))
    w = torch.tensor([1.0 / n, 1.0 / m1.sum(), 1.0 / m2.sum()], dtype=torch.float64, device=dev)
    sums, dth, E = pk.loss_and_grad_raw(variant, *[t(a) for a in a32], t(th32), mask, w, want_E=True)
    torch.cuda.synchronize()
    sums, dth = sums.cpu().numpy(), dth.cpu().numpy()
    print("variant %d n %d: Ltot %.8e ref %.8e rel %.2e | Lpde rel %.2e Lbc rel %.2e" % (
        variant, n, sums[0], ref["Ltot"], abs(sums[0] - ref["Ltot"]) / ref["Ltot"],
        abs(sums[1] - ref["Lpde"]) / ref["Lpde"], abs(sums[2] - ref["Lbc"]) / ref["Lbc"]))
    gmax = np.abs(ref["grad"]).max()
    for i, nm in enumerate(names):
        a, b = dth[offs[i]:offs[i + 1]], ref["grad"][offs[i]:offs[i + 1]]
        print("   %-18s max|ref| %.3e  err/max|ref_tensor| %.2e  err/max|grad| %.2e" % (
            nm, np.abs(b).max(), np.abs(a - b).max() / max(np.abs(b).max(), 1e-300), np.abs(a - b).max() / gmax))

ck = np.load(os.path.join(gd, "checkpoints.npz"))
rng = np.random.default_rng(1)
tp = np.load(os.path.join(gd, "trainpy_n2048.npz"))
case(0, tp["theta"], 4096, 1)      # random-init weights (train.py init rule), poc form
case(1, tp["theta"], 5000, 2)      # train.py form, ragged n
case(0, ck["ionHsym"], 4096, 3)    # trained weights

# raw timing, 2^18 points
for variant in (0, 1):
    n = 1 << 18
    g = torch.Generator().manual_seed(5)
    x, y, z, R, i1, i2 = ra.sample_box(n, "poc", g)
    xs = [t_.ravel().float().to(dev) for t_ in (x, y, z, R)]
    th = torch.from_numpy(ck["ionHsym"].astype(np.float32)).to(dev)
    sums = torch.empty(8, dtype=torch.float64, device=dev); dth = torch.empty(1521, dtype=torch.float64, device=dev)
    for _ in range(3):
        pk.loss_and_grad_raw(variant, *xs, th, None, None, sums=sums, dtheta=dth)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        pk.loss_and_grad_raw(variant, *xs, th, None, None, sums=sums, dtheta=dth)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    print("variant %d: n=2^18 step %.3f ms -> %.3e points/s" % (variant, ms, n / ms * 1e3))
