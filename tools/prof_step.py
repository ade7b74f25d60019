"""Tiny driver for ncu: a few training-step launches on one 2^18-point batch.
   python tools/prof_step.py [variant 0|1] [launches] [finetune 0|1]"""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import ref_autograd as ra

variant = int(sys.argv[1]) if len(sys.argv) > 1 else 0
launches = int(sys.argv[2]) if len(sys.argv) > 2 else 4
finetune = int(sys.argv[3]) if len(sys.argv) > 3 else 0
dev = torch.device("cuda:0")
n = 1 << 18
g = torch.Generator().manual_seed(5)
x, y, z, R, i1, i2 = ra.sample_box(n, "poc" if variant == 0 else "trainpy", g)
xs = [t.ravel().float().to(dev) for t in (x, y, z, R)]
ck = np.load(os.path.join(ROOT, "tests", "golden", "checkpoints.npz"))
th = torch.from_numpy(ck["ionHsym"].astype(np.float32)).to(dev)
w = torch.tensor([1.0 / n, 2.0 / n, 2.0 / n], dtype=torch.float64, device=dev)
sums = torch.empty(8, dtype=torch.float64, device=dev)
dth = torch.empty(1521, dtype=torch.float64, device=dev)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for i in range(launches):
    if i == launches - 1:
        e0.record()
    pk.loss_and_grad_raw(variant, *xs, th, None, w, pk.FINE_TUNE_GRAD_MASK if finetune else 0xFFFF, sums=sums, dtheta=dth)
e1.record()
torch.cuda.synchronize()
print("variant %d: last step %.4f ms, Ltot %.6e" % (variant, e0.elapsed_time(e1), float(sums[0])))
