"""Where does a super-tile's time go?  Runs the training step with a -DPINN_TIMELINE build of the library (clock64 stamps at
phase boundaries of tile 3 of CTA 0) and prints the per-warp phase durations.
   build (CPU box):  python tools/timeline.py build
   run (GPU box):    PINN_B200_LIBRARY=tools/dbg/libpinn_b200_tl.so python tools/timeline.py [variant]"""
import ctypes, glob, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tools", "dbg", "libpinn_b200_tl.so")
if len(sys.argv) > 1 and sys.argv[1] == "build":
    csrc = os.path.join(ROOT, "pinn_for_quantum_wavefunction_surfaces_b200", "csrc")
    srcs = sorted(glob.glob(os.path.join(csrc, "*.cu")))
    subprocess.run(["nvcc", "-O3", "-std=c++17", "-lineinfo", "-DPINN_TIMELINE", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-Xcompiler", "-fPIC", "-shared", "-o", OUT] + srcs + ["-lcudart"], check=True, cwd=csrc)
    print("built", OUT)
    sys.exit(0)
os.environ.setdefault("PINN_B200_LIBRARY", OUT)
sys.path.insert(0, ROOT)
import numpy as np, torch
import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import ref_autograd as ra
variant = int(sys.argv[1]) if len(sys.argv) > 1 else 0
dev = torch.device("cuda:0")
h = pk.Handle.get(0)
n = 1 << 18
g = torch.Generator().manual_seed(5)
x, y, z, R, i1, i2 = ra.sample_box(n, "poc", g)
xs = [t.ravel().float().to(dev) for t in (x, y, z, R)]
th = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "checkpoints.npz"))["ionHsym"].astype(np.float32)).to(dev)
w = torch.tensor([1.0 / n, 2.0 / n, 2.0 / n], dtype=torch.float64, device=dev)
warm = int(sys.argv[2]) if len(sys.argv) > 2 else 3   # many launches first = clocks ramped up like in a long run
for _ in range(warm):
    pk.loss_and_grad_raw(variant, *xs, th, None, w)
torch.cuda.synchronize()
buf = (ctypes.c_longlong * (16 * 32))()
rc = h.L.pinn_debug_timeline(buf)
assert rc == 0, rc
tl = np.array(buf[:]).reshape(16, 32)
names = {0: "tile start", 1: "fwd L1 + st done", 2: "fwd role barrier", 4: "H stash written", 3: "fwd MMA done", 5: "fwd L2 done", 6: "group barrier",
         7: "bwd L2 + st done", 8: "bwd role barrier", 9: "dW mma.sync done", 10: "colsums done", 11: "bwd MMA done",
         12: "bwd L1 done", 15: "tile end"}
nw = 12 if variant == 0 else 8
t0 = tl[:nw, 0].min()
order = [0, 1, 2, 4, 3, 5, 6, 7, 8, 9, 10, 11, 12, 15]
print("warp role grp | " + " | ".join("%s" % names[k] for k in order))
for wv in range(nw):
    role, grp = wv >> 2, wv & 3
    row = tl[wv]
    print("%4d %4d %3d | " % (wv, role, grp) + " ".join("%6d" % (row[k] - t0 if row[k] else -1) for k in order))
print("tile length (warp 0): %d cycles" % (tl[0, 15] - tl[0, 0]))

kb = (ctypes.c_longlong * 48)()
assert h.L.pinn_debug_timeline_kernel(kb) == 0
k = np.array(kb[:])
print("CTA 0, warp 0: setup %d cycles | first tiles %s | steady tile %d | epilogue (fold) %d cycles | kernel body %d cycles = %.1f us" % (
    k[1] - k[0], " ".join(str(int(k[3 + i] - k[2 + i])) for i in range(6)), k[10] - k[9], k[41] - k[40], k[41] - k[0], (k[41] - k[0]) / 1965.0))

cb = (ctypes.c_longlong * 512)()
assert h.L.pinn_debug_timeline_cta(cb) == 0
c = np.array(cb[:]).reshape(256, 2)[:148]
t0 = c[:, 0].min()
print("CTA entry: first 0, median +%.2f us, last +%.2f us | CTA exit: first +%.2f us, median +%.2f us, last +%.2f us (globaltimer)" % (
    (np.median(c[:, 0]) - t0) / 1e3, (c[:, 0].max() - t0) / 1e3, (c[:, 1].min() - t0) / 1e3, (np.median(c[:, 1]) - t0) / 1e3, (c[:, 1].max() - t0) / 1e3))
# event-timed duration of the same launch, for the part outside the CTAs
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
hh = pk.Handle.get(0); hh.profile_begin()
for _ in range(20):
    pk.loss_and_grad_raw(variant, *xs, th, None, w)
torch.cuda.synchronize()
ms, cnt = hh.profile_collect()
print("event-timed step kernel: %.2f us (instrumented build)" % (ms / cnt * 1e3))
print("effective SM clock of that launch: %.0f MHz (CTA 0: %d cycles in %.2f us)" % (
    (k[41] - k[0]) / ((c[0, 1] - c[0, 0]) / 1e3), k[41] - k[0], (c[0, 1] - c[0, 0]) / 1e3))
