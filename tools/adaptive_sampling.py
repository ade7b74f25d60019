"""Uniform against residual-adaptive collocation (RAD: pool 4, k 1, c 1) on the paper schedule: 5000 steps at 8e-3, then
2000 fine-tune steps at 5e-4 on the E-net from the saved model, 100 000 points, from init_poc(0), the same seeds for both.

Reports, as one JSON file (--out, default adaptive_sampling.json in the working directory) with the device's name and
power limit:
  * ms per optimizer step (device events on the trainer's stream) for uniform and for adaptive steps at 100 000 points,
    and the kernels of one adaptive draw (the pool's sampler, its residual, the four selection kernels) from
    torch.profiler, each averaged over the profiled draws;
  * the held-out Lpde of every saved model on one fixed uniform batch of 2^20 points (seed 999, batch 0);
  * E_net (the E-net) and E_int (rayleigh_curve) against E_exact at the 39 R of tests/golden/poc_paper_run_seed0.npz.
The adaptive run's Ltot history is over adaptive batches and is not comparable with the uniform run's; the held-out Lpde is."""
import argparse
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

AD = dict(pool_factor=4, k=1.0, c=1.0)
N_TRAIN = 100000


def power_limit_w(index):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def ms_per_step(adaptive, steps):
    """device-event time per step of a Trainer at N_TRAIN points, every step resampling (sc_sampling 1)"""
    tr = pk.Trainer("poc", N_TRAIN, pk.init_poc(0), seed=0, lr=8e-3, adaptive=adaptive)
    tr.run(20)
    tr.read()
    ts = torch.cuda.ExternalStream(tr.h.L.pinn_trainer_stream(tr.t), device=torch.device("cuda:0"))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ts)
    tr.run(steps)
    e1.record(ts)
    tr.read()
    tr.close()
    return e0.elapsed_time(e1) / steps


def draw_kernels(theta, reps):
    """per-kernel device time of one adaptive draw at N_TRAIN points (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    th = torch.from_numpy(np.asarray(theta, np.float32)).cuda()
    for _ in range(3):
        pk.sample_adaptive("poc", th, N_TRAIN, **AD)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for b in range(reps):
            pk.sample_adaptive("poc", th, N_TRAIN, batch=b, **AD)
        torch.cuda.synchronize()
    us = {}
    for ev in prof.key_averages():
        name = ev.key
        tag = ("pool_sampler" if "sample_kernel" in name else "pool_residual" if "pinn_step_tc_kernel" in name else
               name.split("(")[0].split("::")[-1] if "rad_" in name else None)
        if tag:
            total = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            us[tag] = us.get(tag, 0.0) + total / reps
    return {k: v * 1e-3 for k, v in us.items()}  # ms per draw


def held_out_lpde(theta, batch):
    th = torch.from_numpy(np.asarray(theta, np.float32)).cuda()
    sums, _, _ = pk.loss_and_grad_raw(0, batch["x"], batch["y"], batch["z"], batch["R"], th, batch["mask"], batch["weights"])
    return float(sums[1].item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="adaptive_sampling.json")
    ap.add_argument("--timing-steps", type=int, default=500)
    args = ap.parse_args()
    ref = np.load(os.path.join(ROOT, "tests", "golden", "poc_paper_run_seed0.npz"))
    Rt, Eex = ref["R"], ref["E_exact"]
    theta0 = pk.init_poc(0)
    held = pk.sample(1 << 20, 999, 0)
    rep = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(0), "n_train": N_TRAIN,
           "adaptive": AD, "schedule": "poc paper: 5000 steps lr 8e-3 seed 0, then 2000 fine-tune steps lr 5e-4 seed 1000"}
    # timing
    for _ in range(2):  # alternated, twice
        for name, a in (("uniform", None), ("adaptive", AD)):
            rep.setdefault("ms_per_step_" + name, []).append(ms_per_step(a, args.timing_steps))
    rep["adaptive_draw_kernels_ms"] = draw_kernels(ref["theta_stage1_saved"], 20)
    # the schedule, both arms
    for name, a in (("uniform", None), ("adaptive", AD)):
        t0 = time.time()
        last1, saved1, loss1 = pk.train_poc(theta0, {"n_train": N_TRAIN, "epochs": 5000, "lr": 8e-3}, seed=0, adaptive=a)
        t1 = time.time()
        s1 = saved1 if saved1 is not None else last1
        last2, saved2, loss2 = pk.train_poc(s1, {"n_train": N_TRAIN, "epochs": 2000, "lr": 5e-4}, freezeUnits=True,
                                            seed=1000, adaptive=a)
        t2 = time.time()
        s2 = saved2 if saved2 is not None else last2
        arm = {"seconds_stage1": t1 - t0, "seconds_stage2": t2 - t1, "stage1_saved": saved1 is not None,
               "stage2_saved": saved2 is not None, "min_Ltot_own_batches": [float(loss1["Ltot"].min()), float(loss2["Ltot"].min())]}
        for stage, th in (("stage1", s1), ("stage2", s2)):
            E_net = pk.analysis.enet_curve(th, Rt)["E"]
            E_int = pk.analysis.rayleigh_curve(th, R=Rt)["E_int"]
            arm[stage] = {"held_out_Lpde": held_out_lpde(th, held),
                          "max_abs_E_net_minus_exact": float(np.abs(E_net - Eex).max()),
                          "max_abs_E_net_minus_exact_R_ge_1": float(np.abs(E_net - Eex)[Rt >= 1.0 - 1e-9].max()),
                          "max_abs_E_int_minus_exact": float(np.abs(E_int - Eex).max()),
                          "max_abs_E_int_minus_exact_R_ge_1": float(np.abs(E_int - Eex)[Rt >= 1.0 - 1e-9].max()),
                          "E_net": E_net.tolist(), "E_int": E_int.tolist()}
        rep[name] = arm
    rep["R"], rep["E_exact"] = Rt.tolist(), Eex.tolist()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rep, f, indent=1)
    short = {k: v for k, v in rep.items() if k not in ("R", "E_exact", "uniform", "adaptive")}
    print(json.dumps(short))
    for name in ("uniform", "adaptive"):
        for stage in ("stage1", "stage2"):
            s = rep[name][stage]
            print("%-8s %s: held-out Lpde %.3e | max|E_net-exact| %.2e (R>=1 %.2e) | max|E_int-exact| %.2e (R>=1 %.2e)"
                  % (name, stage, s["held_out_Lpde"], s["max_abs_E_net_minus_exact"], s["max_abs_E_net_minus_exact_R_ge_1"],
                     s["max_abs_E_int_minus_exact"], s["max_abs_E_int_minus_exact_R_ge_1"]))


if __name__ == "__main__":
    main()
