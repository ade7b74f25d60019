"""The device L-BFGS (Trainer.run_lbfgs) against device Adam on the paper's E-net fine-tune (freezeUnits), one fixed batch.

Reports, as one JSON file (--out, default lbfgs_finetune.json in the working directory) with the device's name and power
limit:
  * ms per evaluation (device events on the trainer's stream) of Adam (step kernel, reduction + Adam) and of L-BFGS
    (step kernel, reduction, L-BFGS kernel) at 10^5 and 2^18 points, in the plain and the graph form: fixed-step calls at
    lr 1e-6 that use every slot and hold few curvature pairs, and strong-Wolfe calls with a full history of 20 (the
    fine-tune's setting), with the L-BFGS kernel's mean time inside them;
  * the L-BFGS kernel alone (torch.profiler) at history 10, 20 and 100 with the history full, driven by the stand-alone
    entries on a device-side quadratic, and at the first iteration (empty history);
  * the fine-tune from the re-run's stage-1 model (tests/golden/poc_paper_run_seed0.npz) on one batch of 100 000 points:
    2000 Adam steps at lr 5e-4 against L-BFGS (strong Wolfe, history 20, at most 400 evaluations): batch and held-out
    Ltot, max|E_net - E_exact| over R >= 1, and |E_net - E_int| at R = 1, 2, 3 (analysis.rayleigh_curve)."""
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

MASK = pk.FINE_TUNE_GRAD_MASK


def power_limit_w(index):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def _timed(tr, fn):
    ts = torch.cuda.ExternalStream(tr.h.L.pinn_trainer_stream(tr.t), device=torch.device("cuda:0"))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ts)
    out = fn()
    e1.record(ts)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def eval_times(n, theta, reps):
    """ms per evaluation: Adam steps and fixed-step L-BFGS calls (every slot evaluated) on one batch of n points"""
    s = pk.sample(n, seed=5, batch=0)
    w = s["weights"].cpu().numpy()
    out = {}
    for use_graph in (False, True):
        tag = "graph" if use_graph else "plain"
        tr = pk.Trainer("poc", n, theta, lr=5e-4, grad_mask=MASK)
        tr.set_batch(s["x"], s["y"], s["z"], s["R"], s["mask"], w)
        tr.run(20, resample=False, use_graph=use_graph)
        tr.read()
        ms, _ = _timed(tr, lambda: tr.run(reps * 25, resample=False, use_graph=use_graph))
        out["adam_" + tag] = ms / (reps * 25)
        kw = dict(max_iter=25, max_eval=25, history_size=20, tolerance_grad=0, tolerance_change=0, lr=1e-6)
        tr.run_lbfgs(use_graph=use_graph, **kw)
        tot, evals = 0.0, 0
        for _ in range(reps):
            ms, (st, _) = _timed(tr, lambda: tr.run_lbfgs(use_graph=use_graph, **kw))
            tot += ms
            evals += st["evals"]
        out["lbfgs_" + tag] = tot / evals
        tr.close()
        # the fine-tune's setting (strong Wolfe, history 20): a first call fills the history, the second is timed, a third
        # gives the L-BFGS kernel's mean time inside such a call (torch.profiler; about 35 us with 20 pairs held)
        kw = dict(max_iter=100, max_eval=100, history_size=20, tolerance_grad=0, tolerance_change=0,
                  line_search_fn="strong_wolfe")
        tr = pk.Trainer("poc", n, theta, grad_mask=MASK)
        tr.set_batch(s["x"], s["y"], s["z"], s["R"], s["mask"], w)
        tr.run_lbfgs(use_graph=use_graph, **kw)
        ms, (st, _) = _timed(tr, lambda: tr.run_lbfgs(use_graph=use_graph, **kw))
        out["lbfgs_strong_wolfe_h20_" + tag] = ms / max(st["evals"], 1)
        out["lbfgs_strong_wolfe_h20_evals_" + tag] = st["evals"]
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
            tr.run_lbfgs(use_graph=use_graph, **kw)
            torch.cuda.synchronize()
        out["lbfgs_strong_wolfe_h20_kernel_us_" + tag] = _kernel_mean_us(prof, 0)
        tr.close()
    return out


def lbfgs_kernel_us(history, reps=20):
    """mean device time of one L-BFGS kernel launch with `history` pairs held, and at the first iteration"""
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    diag = torch.rand(pk.N_THETA, dtype=torch.float64, device=dev, generator=g) + 1.0
    center = torch.randn(pk.N_THETA, dtype=torch.float64, device=dev, generator=g)
    st = pk.LBFGSState(np.zeros(pk.N_THETA), history_size=history)
    sums = torch.zeros(8, dtype=torch.float64, device=dev)
    grad = torch.zeros(pk.N_THETA, dtype=torch.float64, device=dev)

    def evaluate():
        r = st.theta - center
        sums[0:1] = 0.5 * (diag * r * r).sum(0, keepdim=True)
        grad.copy_(diag * r)

    def advance(k):
        for _ in range(k):
            evaluate()
            pk.lbfgs_advance(st, sums, grad)

    kw = dict(max_iter=history + reps + 10, lr=1e-3, tolerance_grad=0, tolerance_change=0)
    res = {}
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        pk.lbfgs_begin(st, **kw)
        advance(2)  # the first evaluation, then the first iteration (no history)
        torch.cuda.synchronize()
    res["first_two_evaluations"] = _kernel_mean_us(prof, 2)
    advance(history + 2)  # the history is full from here on
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        advance(reps)
        torch.cuda.synchronize()
    res["history_full"] = _kernel_mean_us(prof, reps)
    s = st.status()
    res["n_iter"] = s["n_iter"]
    return res


def _kernel_mean_us(prof, launches):
    tot, cnt = 0.0, 0
    for ev in prof.key_averages():
        if "lbfgs_kernel" in ev.key:
            tot += getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            cnt += ev.count
    return {"mean_us": tot / max(cnt, 1), "launches": cnt}


def ltot(theta, b):
    t32 = torch.from_numpy(np.asarray(theta, np.float32)).cuda()
    sums, _, _ = pk.loss_and_grad_raw(0, b["x"], b["y"], b["z"], b["R"], t32, b["mask"], b["weights"])
    return float(sums[0].item())


def energies(theta, Rt, Eex):
    E_net = pk.analysis.enet_curve(theta, Rt)["E"]
    rc = pk.analysis.rayleigh_curve(theta, R=np.array([1.0, 2.0, 3.0]))
    return {"max_abs_E_net_minus_exact_R_ge_1": float(np.abs(E_net - Eex)[Rt >= 1.0 - 1e-9].max()),
            "abs_E_net_minus_E_int_R123": np.abs(rc["E_net"] - rc["E_int"]).tolist(), "E_int_R123": rc["E_int"].tolist(),
            "E_net_R123": rc["E_net"].tolist()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="lbfgs_finetune.json")
    ap.add_argument("--reps", type=int, default=8)
    args = ap.parse_args()
    ref = np.load(os.path.join(ROOT, "tests", "golden", "poc_paper_run_seed0.npz"))
    Rt, Eex, th = ref["R"], ref["E_exact"], ref["theta_stage1_saved"].astype(np.float64)
    rep = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(0)}
    rep["ms_per_evaluation"] = {str(n): eval_times(n, th, args.reps) for n in (100000, 1 << 18)}
    rep["lbfgs_kernel_us"] = {str(h): lbfgs_kernel_us(h) for h in (10, 20, 100)}
    # the fine-tune comparison on one fixed batch
    n = 100000
    b = pk.sample(n, seed=2024, batch=0)
    held = pk.sample(n, seed=2025, batch=0)
    w = b["weights"].cpu().numpy()
    ta = pk.Trainer("poc", n, th, lr=5e-4, grad_mask=MASK)
    ta.set_batch(b["x"], b["y"], b["z"], b["R"], b["mask"], w)
    ta.run(2000, resample=False, use_graph=True)
    th_adam = ta.read()["theta"]
    ta.close()
    tl = pk.Trainer("poc", n, th, grad_mask=MASK)
    tl.set_batch(b["x"], b["y"], b["z"], b["R"], b["mask"], w)
    st, trace = tl.run_lbfgs(max_iter=400, max_eval=399, history_size=20, tolerance_grad=0, tolerance_change=0,
                             line_search_fn="strong_wolfe", use_graph=True)
    th_lb = tl.read()["theta"]
    tl.close()
    rep["finetune"] = {"n": n, "batch_seed": 2024, "held_out_seed": 2025}
    for name, t, evals in (("start", th, 0), ("adam_2000_lr5e-4", th_adam, 2000), ("lbfgs_strong_wolfe_h20", th_lb, st["evals"])):
        rep["finetune"][name] = {"evaluations": evals, "Ltot_batch": ltot(t, b), "Ltot_held_out": ltot(t, held),
                                 **energies(t, Rt, Eex)}
    rep["finetune"]["lbfgs_status"] = st
    rep["finetune"]["lbfgs_trace_Ltot"] = trace[:, 0].tolist()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rep, f, indent=1)
    short = {k: v for k, v in rep.items() if k != "finetune"}
    print(json.dumps(short, indent=1))
    for name in ("start", "adam_2000_lr5e-4", "lbfgs_strong_wolfe_h20"):
        s = rep["finetune"][name]
        print("%-24s evals %5d  Ltot batch %.4e  held-out %.4e  max|E_net-exact| R>=1 %.2e  |E_net-E_int| R=1,2,3 %s"
              % (name, s["evaluations"], s["Ltot_batch"], s["Ltot_held_out"], s["max_abs_E_net_minus_exact_R_ge_1"],
                 " ".join("%.2e" % v for v in s["abs_E_net_minus_E_int_R123"])))
    print("lbfgs:", st)


if __name__ == "__main__":
    main()
