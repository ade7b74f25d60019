"""Cost and effect of importance-weighted adaptive batches (pinn_loss_fwd_bwd_weighted, Trainer importance mode).

Reports, as one JSON file (--out, default importance_sampling.json in the working directory) with the device's name and
power limit read in the same run:
  * ms per training evaluation (the C entries pinn_loss_fwd_bwd and pinn_loss_fwd_bwd_weighted: step kernel + reduction)
    at 10^5 and 2^18 points of an importance draw, unweighted against weighted, device events over --reps calls,
    alternated --rounds times (the C entries, because loss_and_grad_raw's check of the weights' values reads them back);
  * ms per trainer step at 10^5 points, adaptive against adaptive + importance (pool 4, k 1, c 1), alternated twice;
  * the poc paper schedule (5000 steps lr 8e-3 from init_poc(seed), training seed `seed`, then 2000 fine-tune steps lr 5e-4
    on the E-net, seed 1000 + seed; 10^5 points) for every seed of --seeds and each arm uniform / adaptive / adaptive +
    importance: the held-out Ltot, Lpde, Lbc (validation=dict(n=2^20, seed=999, every=100): last row of each stage) and
    max|E_net - E_exact|, max|E_int - E_exact| over R >= 1 (rayleigh_curve) of the model each stage saved; then the
    median, minimum and maximum per arm."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pinn_for_quantum_wavefunction_surfaces_b200 as pk  # noqa: E402

N_TRAIN = 100000
VAL = dict(n=1 << 20, seed=999, every=100)
ARMS = {"uniform": None, "adaptive": dict(pool_factor=4, k=1.0, c=1.0),
        "importance": dict(pool_factor=4, k=1.0, c=1.0, importance=True)}


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


def step_cost(reps, rounds):
    th = torch.from_numpy(pk.init_poc(0).astype(np.float32)).cuda()
    out = {}
    for n in (100000, 1 << 18):
        b = pk.sample_adaptive("poc", th, n, seed=5, batch=0, importance=True, **ARMS["adaptive"])
        cols = [b[k] for k in "xyzR"]
        sums, dth = torch.empty(8, dtype=torch.float64, device="cuda"), torch.empty(pk.N_THETA, dtype=torch.float64, device="cuda")
        h = pk.Handle.get(0)
        P = lambda t: ctypes.c_void_p(t.data_ptr())
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        head = [h.h, 0, n] + [P(c) for c in cols] + [0, P(b["mask"]), P(th), P(b["weights"])]
        tail = [0xFFFF, 17.5, P(sums), P(dth), None, st]
        plain = lambda: h.check(h.L.pinn_loss_fwd_bwd(*head, *tail), "pinn_loss_fwd_bwd")
        weighted = lambda: h.check(h.L.pinn_loss_fwd_bwd_weighted(*head, P(b["point_weights"]), *tail),
                                   "pinn_loss_fwd_bwd_weighted")
        r = {"unweighted_ms": [], "weighted_ms": []}
        for _ in range(rounds):
            r["unweighted_ms"].append(timed(plain, reps))
            r["weighted_ms"].append(timed(weighted, reps))
        r["weighted_over_unweighted"] = float(np.median(r["weighted_ms"]) / np.median(r["unweighted_ms"]))
        out[str(n)] = r
    return out


def ms_per_step(adaptive, steps):
    tr = pk.Trainer("poc", N_TRAIN, pk.init_poc(0), seed=0, lr=8e-3, adaptive=adaptive)
    tr.run(50, use_graph=True)
    tr.read()
    ts = torch.cuda.ExternalStream(tr.h.L.pinn_trainer_stream(tr.t), device=torch.device("cuda:0"))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ts)
    tr.run(steps, use_graph=True)
    e1.record(ts)
    tr.read()
    tr.close()
    return e0.elapsed_time(e1) / steps


def run_arm(seed, adaptive, Rt, Eex):
    t0 = time.time()
    last1, saved1, loss1 = pk.train_poc(pk.init_poc(seed), {"n_train": N_TRAIN, "epochs": 5000, "lr": 8e-3}, seed=seed,
                                        adaptive=adaptive, validation=VAL)
    s1 = saved1 if saved1 is not None else last1
    last2, saved2, loss2 = pk.train_poc(s1, {"n_train": N_TRAIN, "epochs": 2000, "lr": 5e-4}, freezeUnits=True,
                                        seed=1000 + seed, adaptive=adaptive, validation=VAL)
    s2 = saved2 if saved2 is not None else last2
    r = {"seconds": time.time() - t0}
    ge1 = Rt >= 1.0 - 1e-9
    for stage, th, loss in (("stage1", s1, loss1), ("stage2", s2, loss2)):
        row = loss["validation"]["rows"][-1]
        E_net = pk.analysis.enet_curve(th, Rt)["E"]
        E_int = pk.analysis.rayleigh_curve(th, R=Rt)["E_int"]
        r[stage] = {"held_out_Ltot": float(row[1]), "held_out_Lpde": float(row[2]), "held_out_Lbc": float(row[3]),
                    "max_abs_E_net_minus_exact_R_ge_1": float(np.abs(E_net - Eex)[ge1].max()),
                    "max_abs_E_int_minus_exact_R_ge_1": float(np.abs(E_int - Eex)[ge1].max())}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="importance_sampling.json")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--timing-steps", type=int, default=1000)
    ap.add_argument("--seeds", type=int, nargs="+", default=[0, 1, 2, 3, 4])
    args = ap.parse_args()
    ref = np.load(os.path.join(ROOT, "tests", "golden", "poc_paper_run_seed0.npz"))
    Rt, Eex = ref["R"], ref["E_exact"]
    rep = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(0), "n_train": N_TRAIN,
           "validation": VAL, "arms": ARMS,
           "schedule": "poc paper: 5000 steps lr 8e-3 from init_poc(seed), seed; 2000 fine-tune steps lr 5e-4, seed 1000 + seed"}
    rep["evaluation_ms"] = step_cost(args.reps, args.rounds)
    for _ in range(2):  # alternated, twice
        for name in ("adaptive", "importance"):
            rep.setdefault("trainer_ms_per_step_" + name, []).append(ms_per_step(ARMS[name], args.timing_steps))
    runs = {name: {} for name in ARMS}
    for seed in args.seeds:
        for name, a in ARMS.items():
            runs[name][seed] = run_arm(seed, a, Rt, Eex)
            print("seed %d %-10s %s" % (seed, name, json.dumps(runs[name][seed]["stage2"])), flush=True)
    rep["runs"] = runs
    summary = {}
    for name in ARMS:
        summary[name] = {}
        for stage in ("stage1", "stage2"):
            for key in runs[name][args.seeds[0]][stage]:
                v = np.array([runs[name][s][stage][key] for s in args.seeds])
                summary[name][stage + "." + key] = {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}
    rep["summary"] = summary
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps({k: v for k, v in rep.items() if k not in ("runs", "summary")}))
    for name in ARMS:
        print(name)
        for k, v in summary[name].items():
            print("  %-45s median %.3e  [%.3e, %.3e]" % (k, v["median"], v["min"], v["max"]))


if __name__ == "__main__":
    main()
