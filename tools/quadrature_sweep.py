"""Time the two ways of getting E_int(R) for the paper's E(R) table, with the fine-tuned checkpoint:

  cartesian_80      analysis.calculate_E_R at n_test = 80 (39 R, one 512 000-point Simpson grid per R, the reference's
                    resolution)
  spheroidal_39     one analysis.rayleigh_curve call at the same 39 R (1 152 Gauss-Legendre nodes per R, one launch)
  spheroidal_1000   one rayleigh_curve call at 1000 R in [0.2, 4]

Each is warmed up once and then timed `--reps` times with CUDA events around the call, which ends in a host
synchronisation (the results are copied to the host); the median is reported.  Prints one JSON line that carries the
device name and its power limit, and the largest difference between the two E_int columns.

    python tools/quadrature_sweep.py [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pinn_for_quantum_wavefunction_surfaces_b200 as pk  # noqa: E402


def power_limit_w(index):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def timed(fn, reps):
    fn()
    ms, out = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("quadrature_sweep.py needs a CUDA device")
    th = np.load(os.path.join(ROOT, "tests", "golden", "checkpoints.npz"))["ionHsym_fineTune"]
    R1000 = np.linspace(0.2, 4.0, 1000)
    t_cart, cart = timed(lambda: pk.analysis.calculate_E_R(th, {"n_test": 80}), args.reps)
    t_39, sph = timed(lambda: pk.analysis.rayleigh_curve(th), args.reps)
    t_1000, _ = timed(lambda: pk.analysis.rayleigh_curve(th, R1000), args.reps)
    dev = torch.cuda.current_device()
    res = {
        "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev), "reps": args.reps,
        "cartesian_80_39R_ms": t_cart, "spheroidal_39R_ms": t_39, "spheroidal_1000R_ms": t_1000,
        "points_per_R": {"cartesian_80": 80 ** 3, "spheroidal": int(np.prod([len(v) for v in pk.analysis.spheroidal_nodes()[::2]]))},
        "E_int_cartesian80_minus_spheroidal": {"R": [float(r) for r in sph["R"]],
                                               "diff": [float(d) for d in cart["E_int"] - sph["E_int"]]},
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
