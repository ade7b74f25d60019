"""Cost and use of the held-out validation loss (pinn_loss_eval, Trainer.set_validation).

Reports, as one JSON file (--out, default validation_loss.json in the working directory) with the device's name and
power limit read in the same run:
  * ms per pinn_loss_eval call at 2^18, 2^20 and 2^22 sampler points, against loss_and_grad_raw (the training kernel and
    its reduction) on the same points, device events over --reps calls after a warm-up;
  * ms per trainer step at 100 000 points without validation and with validation=dict(n=2^20, every=100), device events
    on the trainer's stream, alternated twice;
  * the held-out Ltot curves (2^20 points, seed 999, every 100 steps, from a step-0 evaluation) of the paper schedule's
    first stage (5000 steps at 8e-3 from init_poc(0), seed 0), uniform against residual-adaptive batches (pool 4, k 1,
    c 1), and the best-on-validation record of each."""
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

AD = dict(pool_factor=4, k=1.0, c=1.0)
N_TRAIN = 100000
VAL = dict(n=1 << 20, seed=999, every=100)


def power_limit_w(index):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def timed(fn, reps):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def eval_cost(reps):
    th = torch.from_numpy(pk.init_poc(0).astype(np.float32)).cuda()
    out = {}
    for lg in (18, 20, 22):
        b = pk.sample(1 << lg, 5, 0)
        cols = [b[k] for k in "xyzR"]
        sums, dth = torch.empty(8, dtype=torch.float64, device="cuda"), torch.empty(pk.N_THETA, dtype=torch.float64, device="cuda")
        ev = lambda: pk.loss_eval(0, *cols, th, mask=b["mask"], weights=b["weights"], sums=sums)
        tr = lambda: pk.loss_and_grad_raw(0, *cols, th, b["mask"], b["weights"], sums=sums, dtheta=dth)
        r = {"loss_eval_ms": [], "loss_and_grad_raw_ms": []}
        for _ in range(2):  # alternated, twice
            r["loss_eval_ms"].append(timed(ev, reps))
            r["loss_and_grad_raw_ms"].append(timed(tr, reps))
        out["2^%d" % lg] = r
    return out


def ms_per_step(validation, steps):
    tr = pk.Trainer("poc", N_TRAIN, pk.init_poc(0), seed=0, lr=8e-3, validation=validation)
    tr.run(200)
    tr.read()
    ts = torch.cuda.ExternalStream(tr.h.L.pinn_trainer_stream(tr.t), device=torch.device("cuda:0"))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ts)
    tr.run(steps)
    e1.record(ts)
    tr.read()
    tr.close()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="validation_loss.json")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--timing-steps", type=int, default=3000)
    args = ap.parse_args()
    rep = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(0), "n_train": N_TRAIN, "validation": VAL,
           "adaptive": AD, "schedule": "poc paper stage 1: 5000 steps lr 8e-3 seed 0 from init_poc(0)"}
    rep["eval_ms"] = eval_cost(args.reps)
    for _ in range(2):  # alternated, twice
        for name, v in (("without", None), ("with", VAL)):
            rep.setdefault("ms_per_step_" + name + "_validation", []).append(ms_per_step(v, args.timing_steps))
    for name, a in (("uniform", None), ("adaptive", AD)):
        last, saved, loss = pk.train_poc(pk.init_poc(0), {"n_train": N_TRAIN, "epochs": 5000, "lr": 8e-3}, seed=0, adaptive=a,
                                         validation=VAL)
        v = loss["validation"]
        rep[name] = {"rows": v["rows"].tolist(), "best_val_loss": v["best_val_loss"], "best_val_step": v["best_val_step"],
                     "last_val_Ltot": float(v["rows"][-1, 1]), "min_Ltot_own_batches": float(loss["Ltot"].min())}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps({k: v for k, v in rep.items() if k not in ("uniform", "adaptive")}))
    for name in ("uniform", "adaptive"):
        r = rep[name]
        print("%-8s held-out Ltot: step 0 %.3e, step 5000 %.3e, best %.3e at step %d" % (
            name, r["rows"][0][1], r["last_val_Ltot"], r["best_val_loss"], r["best_val_step"]))


if __name__ == "__main__":
    main()
