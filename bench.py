#!/usr/bin/env python
"""Benchmark of the PINN residual-and-gradient hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--points P] [--dump-outputs DIR]

A step = one training evaluation (forward + Laplacian + loss + parameter gradients; for N>1 including the
sum of the 8 + 1521 float64 over the ranks, fused into the reduction kernel or, --allreduce nccl, as a
separate all-reduce) of the poc-form ionHsym model on one batch of P synthetic collocation points per GPU
(default 2^18 = BASELINE config 3; weak scaling: every GPU gets its own P points).
Prints ONE JSON line (rank 0): value (device-resident inputs), roofline (kernel events; FP32 peak measured in this run;
ncu figures of the committed capture when it belongs to this build), e2e (page-locked host inputs through HostStep /
pinn_loss_fwd_bwd_host), seam_e2e (the reference-style loop: patched LossFunctions -> backward -> torch Adam -> .cpu()),
config4_global_batch (2^22 points/step sharded over the ranks), value_steady (>= 1000 steps), at N>1 dp_parity (the fused
exchange against one GPU and against an NCCL all-reduce, on a common batch, before anything is timed), and at N=1
cpu_baseline, reference_autograd_on_gpu, dense_grid_inference, device_train_loop.  See DESIGN.md section 5.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_POINT = 27044.0          # canonical algorithmic FLOPs of one poc training step (SURVEY.md 8d)
FP32_PEAK_FALLBACK = 72.0e12      # round-1 measurement (profiles/r01_microbench_pipes.jsonl); the run measures its own
FP32_PEAK_NOMINAL = 148 * 128 * 2 * 1.965e9
N_BATCHES = 40                    # rotating input batches: 40 x 4 MiB = 168 MB > 126 MB L2


def synth_batch(n, seed, variant="poc"):
    """x,y,z ~ U(-18,18), R ~ U(0.2,4), clamp at 0.005 from the nuclei (poc/main.py:124-156)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(4, n, generator=g, dtype=torch.float32)
    x, y, z = (2 * u[0] - 1) * 18, (2 * u[1] - 1) * 18, (2 * u[2] - 1) * 18
    R = 0.2 + (4.0 - 0.2) * u[3]
    r1 = torch.sqrt((x - R) ** 2 + y ** 2 + z ** 2)
    r2 = torch.sqrt((x + R) ** 2 + y ** 2 + z ** 2)
    x = torch.where((r1 < 0.005) | (r2 < 0.005), torch.full_like(x, 0.005), x)
    return torch.stack([x, y, z, R]).contiguous()


def load_theta():
    return np.load(os.path.join(ROOT, "tests", "golden", "checkpoints.npz"))["ionHsym"]


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.05 and len(r) >= 7] or [r for _, r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(r[3 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "samples": len(rows), "power_w_max": max(float(r[2]) for r in rows)}


def host_threads():
    """All host cores this process may use.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which is why
    the thread count is set explicitly here instead of being left to the environment."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_points_per_s(theta, min_seconds, points=1 << 18):
    """The reference's own way of computing the step (nested autograd, float64, all host threads): oracle/ref_autograd.py
    on one full batch of `points` points, repeated for >= min_seconds."""
    import torch
    from oracle import ref_autograd as ra
    cores = host_threads()
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(1234)
    x, y, z, R, i1, i2 = ra.sample_box(points, "poc", g)
    th = torch.tensor(theta, dtype=torch.float64)
    ra.loss_and_grad("poc", th, x, y, z, R, i1, i2)  # warm-up
    times = []
    t_all = time.time()
    while time.time() - t_all < min_seconds or len(times) < 2:
        t0 = time.time()
        ra.loss_and_grad("poc", th, x, y, z, R, i1, i2)
        times.append(time.time() - t0)
    best = min(times)
    return points / best, cores, ("%d points (the full batch) x %d evaluations (best of), float64 nested autograd, %d threads"
                                  % (points, len(times), cores)), best


def ref_autograd_on_gpu(theta, dev, n=1 << 18):
    """BASELINE config 2: the reference's own algorithm (nested torch autograd, oracle/ref_autograd.py) executed by
    PyTorch on the same B200, float64 as shipped and float32, on one 2^18-point batch."""
    import torch
    from oracle import ref_autograd as ra
    g = torch.Generator().manual_seed(4321)
    x, y, z, R, i1, i2 = ra.sample_box(n, "poc", g)
    out = {}
    for name, dt in (("f64", torch.float64), ("f32", torch.float32)):
        a = [t.to(device=dev, dtype=dt) for t in (x, y, z, R)]
        j1, j2 = i1.to(dev), i2.to(dev)
        th = torch.tensor(theta, dtype=dt, device=dev)
        for _ in range(2):
            ra.loss_and_grad("poc", th, *a, j1, j2)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for _ in range(reps):
            ra.loss_and_grad("poc", th, *a, j1, j2)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = {"value": n / (ms * 1e-3), "unit": "points/s", "ms_per_step": ms}
    out["what"] = "torch eager nested autograd of the reference model on cuda:0, %d points, %d evaluations each" % (n, reps)
    return out


def dense_grid_inference(dev, n_axis=464):
    """BASELINE config 5: psi, H psi and the Simpson-weighted energy sums on a 464^3 = 1.0e8-point grid at one R
    (models/ionHsym_fineTune.pt weights), points generated in-kernel, only 5 sums leave each SM."""
    import torch
    import pinn_for_quantum_wavefunction_surfaces_b200 as pk
    th = np.load(os.path.join(ROOT, "tests", "golden", "checkpoints.npz"))["ionHsym_fineTune"]
    pk.analysis.grid_sums(th, 2.0, n=80, device=dev.index)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = pk.analysis.grid_sums(th, 2.0, n=n_axis, device=dev.index)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    pts = float(n_axis) ** 3
    # fixed-R inference: 6 656 FLOP/point (SURVEY.md 8d)
    return {"value": pts / (ms * 1e-3), "unit": "points/s", "ms": ms, "grid": "%d^3" % n_axis,
            "E_int": r["psiHpsi"] / r["psi2"], "flop_per_point": 6656.0, "tflops": 6656.0 * pts / (ms * 1e-3) / 1e12}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only): float64 nested
    autograd (oracle/ref_autograd.py, pinned to the real reference by tests/test_oracle.py) on the SAME workload as the
    GPU arm - one full batch of --points (2^18) points per step, --steps steps (about 0.4 s each on 16 cores), all host
    threads (set explicitly)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    theta = load_theta()
    import torch
    from oracle import ref_autograd as ra
    cores = host_threads()
    torch.set_num_threads(cores)
    ns = args.points
    g = torch.Generator().manual_seed(1234)
    x, y, z, R, i1, i2 = ra.sample_box(ns, "poc", g)
    th = torch.tensor(theta, dtype=torch.float64)
    ra.loss_and_grad("poc", th, x, y, z, R, i1, i2)
    W = max(0, min(args.warmup, 3) - 1)
    for _ in range(W):
        ra.loss_and_grad("poc", th, x, y, z, R, i1, i2)
    steps = max(1, args.steps)
    t0 = time.time()
    for _ in range(steps):
        r = ra.loss_and_grad("poc", th, x, y, z, R, i1, i2)
    dt = (time.time() - t0) / steps
    v = ns / dt
    if args.dump_outputs:
        E = r[3]
        if E.shape[0] > DUMP_MAX_POINTS:   # a fixed, seeded sample of the per-point energies keeps the dump small
            keep = np.sort(np.random.default_rng(0).choice(E.shape[0], DUMP_MAX_POINTS, replace=False))
            E = E[torch.from_numpy(keep)]
        dump_outputs(args.dump_outputs, loss=torch.stack(r[:3]), dtheta=r[4], E=E)
    sample = ("each step = one full batch of %d points; float64 nested autograd (oracle/ref_autograd.py), %d threads; "
              "%d steps timed" % (ns, cores, steps))
    emit({
        "impl": "reference", "metric": "collocation points/sec per training step (fwd+lap+bwd)", "value": v,
        "unit": "points/s", "n_gpus": args.gpus, "steps": steps, "warmup": W + 1, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "points_per_gpu": ns, "host_threads": cores},
        "cpu_baseline": {"value": v, "unit": "points/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def hbm_ceiling(bytes_per_launch, kernel_ms):
    """The contract's other denominator: the kernel against the measured HBM copy rate (MEASURED_PEAKS.json, burst figure for
    a kernel timed alone; the profiling recipe's 6650 GB/s "of fallback" when the file is absent).  27 kFLOP per 16 bytes puts this path
    three orders of magnitude on the compute side of the ridge, which is why `bound` is the FP32 pipe."""
    peak, src = 6650.0, "of fallback (B200_PROFILING.md)"
    pj = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pj):
        try:
            peak, src = float(json.load(open(pj))["hbm_gbs"]), "of measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    ach = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    return {"achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": src}


_RESULT_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries below us write there too (NCCL prints its version banner on
    communicator creation when NCCL_DEBUG is set in the environment), so file descriptor 1 is pointed at stderr for the
    whole run and the result line goes to a private duplicate of the original stdout."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    _RESULT_OUT.write(json.dumps(line) + "\n")
    _RESULT_OUT.flush()


DUMP_MAX_POINTS = 1 << 20          # --dump-outputs: per-point arrays beyond this many points are sampled (8 MB float64)


def dump_outputs(directory, **arrays):
    """--dump-outputs DIR: the arrays the timed path returned in its last step, one float64 DIR/<name>.npy each, so that
    two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.  Both arms
    write loss.npy (Ltot, Lpde, Lbc) and dtheta.npy under the same names."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a.detach().cpu().numpy().astype(np.float64))


def tensor_ceiling(flop_per_launch, kernel_ms):
    """SURVEY section 8(d)'s denominator for contractions moved to the tensor pipe: the measured dense tensor rate in TF32
    (= half the bf16 figure of MEASURED_PEAKS.json, burst, for a kernel timed alone; 1590 TFLOP/s bf16 "of fallback"
    without the file) divided by 3 for 3xTF32.  The numerator is the canonical FLOP count of the WHOLE step, of which about
    half (layer-2 mat-vecs of the MLP and the E-net, forward and reverse) runs on tcgen05; ncu's tensor-pipe utilisation
    (roofline.ncu_pipe_utilisation_pct.tensor) is the direct measurement."""
    bf16, src = 1590.0, "of fallback (B200_PROFILING.md)"
    pj = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pj):
        try:
            bf16, src = float(json.load(open(pj))["bf16_tflops"]), "of measured (MEASURED_PEAKS.json bf16_tflops / 2 / 3)"
        except (KeyError, ValueError):
            pass
    peak = bf16 / 2.0 / 3.0
    ach = flop_per_launch / (kernel_ms * 1e-3) / 1e12
    return {"achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": src}


def kernel_source_sha256():
    """Hash of the sources the step kernel is compiled from: ties the committed ncu figures (profiles/traffic.json) to a build."""
    import hashlib
    hsh = hashlib.sha256()
    csrc = os.path.join(ROOT, "pinn_for_quantum_wavefunction_surfaces_b200", "csrc")
    for f in ("pinn_step_tc.cu", "pinn_tc.cuh", "pinn_device.cuh", "pinn_common.cuh", "pinn_launch.h"):
        with open(os.path.join(csrc, f), "rb") as fh:
            hsh.update(fh.read())
    return hsh.hexdigest()


def committed_ncu_figures():
    """roofline.traffic / pipe utilisation come from ONE `ncu --set full` capture (a number taken under a profiler cannot be
    produced inside a timed run).  profiles/traffic.json records the hash of the kernel sources it was captured from; when
    the sources have changed since, the figures are withheld instead of silently describing another kernel."""
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(tf):
        return None, None, "no capture committed"
    tj = json.load(open(tf))
    now = kernel_source_sha256()
    if tj.get("kernel_source_sha256") != now:
        return None, None, ("stale: profiles/traffic.json was captured from kernel sources %s, this build is %s"
                            % (str(tj.get("kernel_source_sha256"))[:12], now[:12]))
    return tj.get("dram_bytes_per_launch"), tj.get("ncu_pipe_utilisation_pct"), "%s (kernel sources %s)" % (tj.get("source"), now[:12])


def dp_parity_check(pk, dp, dist, h, dev, rank, world, theta, n=1 << 18):
    """Correctness of the fused exchange where the driver can see it (N > 1), before anything is timed: every rank evaluates
    ITS SHARD of one common seeded batch through the fused exchange; the result must be bit-identical on all ranks, equal to
    the same shards summed by an NCCL all-reduce (same arithmetic, other transport: 1e-12) and equal to one GPU evaluating
    the whole batch alone (other tiling of the float32 partial sums: 1e-6).  Returns the dict for the JSON line."""
    import torch
    b = synth_batch(n, 777)                       # identical on every rank
    r1 = torch.sqrt((b[0] - b[3]) ** 2 + b[1] ** 2 + b[2] ** 2)
    r2 = torch.sqrt((b[0] + b[3]) ** 2 + b[1] ** 2 + b[2] ** 2)
    w = torch.tensor([1.0 / n, 1.0 / float((r1 >= 17.5).sum()), 1.0 / float((r2 >= 17.5).sum())], dtype=torch.float64, device=dev)
    per = n // world
    lo, hi = rank * per, (rank + 1) * per if rank < world - 1 else n
    sh = [b[k, lo:hi].contiguous().to(dev) for k in range(4)]
    full = [b[k].contiguous().to(dev) for k in range(4)]

    def evaluate(cols):
        out = torch.zeros(dp.N_OUT, dtype=torch.float64, device=dev)
        pk.loss_and_grad_raw(0, cols[0], cols[1], cols[2], cols[3], theta, None, w, sums=out[:8], dtheta=out[8:])
        return out
    fused = evaluate(sh)                          # exchange enabled: global sums on every rank
    torch.cuda.synchronize()
    gathered = [torch.empty_like(fused) for _ in range(world)]
    dist.all_gather(gathered, fused)
    bitwise = all(torch.equal(gathered[0].view(torch.int64), g.view(torch.int64)) for g in gathered[1:])
    h.dp_enable(False)
    local = evaluate(sh)
    dist.all_reduce(local)                        # the same shards through NCCL
    single = evaluate(full)                       # one GPU, whole batch (every rank does it; rank 0's is reported)
    torch.cuda.synchronize()
    dist.barrier()
    h.dp_enable(True)
    rel = lambda a, c: float((a - c).abs().max() / c.abs().max())
    res = {"points": n, "bitwise_equal_across_ranks": bool(bitwise),
           "rel_sums_vs_nccl_allreduce": rel(fused[:7], local[:7]), "rel_grad_vs_nccl_allreduce": rel(fused[8:], local[8:]),
           "rel_sums_vs_single_gpu": rel(fused[:7], single[:7]), "rel_grad_vs_single_gpu": rel(fused[8:], single[8:]),
           "bars": {"vs_nccl_allreduce": 1e-12, "vs_single_gpu": 1e-6}}
    res["ok"] = bool(bitwise and res["rel_sums_vs_nccl_allreduce"] < 1e-12 and res["rel_grad_vs_nccl_allreduce"] < 1e-12 and
                     res["rel_sums_vs_single_gpu"] < 1e-6 and res["rel_grad_vs_single_gpu"] < 1e-6)
    flag = torch.tensor([1 if res["ok"] else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res["ok_on_all_ranks"] = bool(int(flag.item()))
    return res


def seam_e2e(pk, dev, n, steps):
    """The drop-in boundary itself, timed: the reference's training-loop body (poc/main.py:394-411) - zero_grad,
    model.LossFunctions (patched: pk.patch_nn_ion), Ltot.backward(), torch.optim.Adam.step(), the four .cpu() reads of the
    history lines - on an nn.Module with NN_ion's parameter set (same names, shapes, order; float64 like the reference),
    batches of n points as (n,1) float64 tensors with torch.where index tuples.  Sampling is the reference's own code and
    is not part of the seam, so batches are drawn up front: 8 rotating batches (every step sees index tensors the mask cache
    does not hold = the resampling phase of the loop) and one frozen batch (the last 10 % of the reference's epochs)."""
    import torch
    import torch.nn as nn
    from pinn_for_quantum_wavefunction_surfaces_b200 import convert

    class IonParams(nn.Module):
        def __init__(self, theta):
            super().__init__()
            mk = lambda i, o: nn.Linear(i, o, dtype=torch.float64)
            self.Lin_H1, self.Lin_H2, self.Lin_out = mk(2, 16), mk(16, 16), mk(16, 1)
            self.Lin_E1, self.Lin_E2, self.Lin_Eout = mk(1, 32), mk(32, 32), mk(32, 1)
            self.netDecayL, self.netDecay = mk(1, 10), mk(10, 1)
            self.P, self.Ry, self.Rz = 1, 0, 0
            self.load_state_dict(convert.state_dict_from_theta(theta))
    assert [k for k, _ in IonParams(load_theta()).named_parameters()] == pk.POC_TENSOR_NAMES
    pk.patch_nn_ion(IonParams)
    params = {"BCcutoff": 17.5, "inversion_symmetry": 1, "Ry": 0, "Rz": 0}

    def batches(device, nb, pin=False):
        out = []
        for k in range(nb):
            b = synth_batch(n, 5000 + k).double()
            cols = [b[j].reshape(n, 1).contiguous() for j in range(4)]
            if pin:
                cols = [c.pin_memory() for c in cols]
            cols = [c.to(device) for c in cols] if device.type == "cuda" else cols
            r1 = torch.sqrt((cols[0] - cols[3]) ** 2 + cols[1] ** 2 + cols[2] ** 2)
            r2 = torch.sqrt((cols[0] + cols[3]) ** 2 + cols[1] ** 2 + cols[2] ** 2)
            out.append(cols + [torch.where(r1 >= 17.5), torch.where(r2 >= 17.5)])
        return out

    def loop(device, bs, K):
        model = IonParams(load_theta()).to(device)
        opt = torch.optim.Adam(model.parameters(), lr=1e-7, weight_decay=0)
        Ltot_h, Lpde_h, Lbc_h, E_h = (np.zeros([K + 5, 1]) for _ in range(4))   # the reference's history arrays (main.py:375-378)
        split = {"LossFunctions": 0.0, "backward": 0.0, "optimizer.step": 0.0, "history .cpu()": 0.0}
        pc = time.perf_counter
        for tt in range(K + 5):
            if tt == 5:                                  # 5 untimed steps first
                if device.type == "cuda":
                    torch.cuda.synchronize()
                split = {k: 0.0 for k in split}
                t_start = pc()
            x, y, z, R, b1, b2 = bs[tt % len(bs)]
            opt.zero_grad()
            t0 = pc()
            Ltot, LossPDE, Lbc, E = model.LossFunctions(x, y, z, R, params, b1, b2)
            t1 = pc()
            Ltot.backward(retain_graph=False)
            t2 = pc()
            opt.step()
            t3 = pc()
            Ltot_h[tt] = Ltot.cpu().data.numpy(); Lpde_h[tt] = LossPDE.cpu().data.numpy()     # main.py:408-411, literally
            Lbc_h[tt] = Lbc.cpu().data.numpy(); E_h[tt] = E[-1].cpu().data.numpy()
            t4 = pc()
            split["LossFunctions"] += t1 - t0; split["backward"] += t2 - t1
            split["optimizer.step"] += t3 - t2; split["history .cpu()"] += t4 - t3
        if device.type == "cuda":
            torch.cuda.synchronize()
        dt = (pc() - t_start) / K
        return {"value": n / dt, "unit": "points/s", "ms_per_step": dt * 1e3, "steps": K, "loss": float(Ltot_h[-1, 0]),
                "host_ms_per_step": {k: round(v / K * 1e3, 4) for k, v in split.items()}}
    def autograd_floor(device, K=200):
        """What PyTorch itself charges for ANY op with this signature: a torch.autograd.Function with the same 24 inputs and
        4 outputs that does nothing (one empty() in forward, one multiply and 16 views in backward), in the same loop."""
        model = IonParams(load_theta()).to(device)
        ps = tuple(model.parameters())
        sizes = [p.numel() for p in ps]

        class NoOp(torch.autograd.Function):
            @staticmethod
            def forward(ctx, variant, order, x, y, z, R, i1, i2, *params):
                out = torch.zeros(8 + 1521, dtype=torch.float64, device=x.device)
                E = torch.empty(x.shape[0], dtype=torch.float64, device=x.device).view(-1, 1)
                ctx.save_for_backward(out[8:])
                ctx.shapes = [p.shape for p in params]
                L, a, b2 = out[0], out[1], out[2]
                ctx.mark_non_differentiable(a, b2, E)
                return L, a, b2, E

            @staticmethod
            def backward(ctx, g, *_):
                (d,) = ctx.saved_tensors
                parts = (d * g).split(sizes)
                return (None,) * 8 + tuple(q if len(sh) == 1 else q.view(sh) for q, sh in zip(parts, ctx.shapes))
        x = torch.zeros(n, 1, dtype=torch.float64, device=device)
        tf = tb = 0.0
        pc = time.perf_counter
        for tt in range(K + 5):
            if tt == 5:
                tf = tb = 0.0
            for p in ps:
                p.grad = None
            t0 = pc()
            L = NoOp.apply(0, "poc", x, x, x, x, None, None, *ps)[0]
            t1 = pc()
            L.backward()
            t2 = pc()
            tf += t1 - t0; tb += t2 - t1
        if device.type == "cuda":
            torch.cuda.synchronize()
        return {"forward_ms": round(tf / K * 1e3, 4), "backward_ms": round(tb / K * 1e3, 4)}
    cpu = torch.device("cpu")
    n_small = n
    res = {"cuda_resident": loop(dev, batches(dev, 8), steps),
           "cuda_resident_frozen_batch": loop(dev, batches(dev, 1), steps),
           "cpu_resident_pageable": loop(cpu, batches(cpu, 8), max(5, steps // 4)),
           "cpu_resident_pinned": loop(cpu, batches(cpu, 8, pin=True), max(5, steps // 4)),
           "autograd_floor_cuda": autograd_floor(dev),
           "e2e_fraction_note": "per step the loop spends ~0.26 ms in torch.optim.Adam.step and ~0.1 ms in the four .cpu() reads on the "
                                "host - the reference's own lines - against 0.14 ms for a whole e2e step; autograd_floor_cuda is what a "
                                "torch.autograd.Function with the same 24 inputs costs when it does nothing; the seam is host-bound at "
                                "2^18 points and GPU-bound from ~2^21 points per step on (cuda_resident_4M_points)",
           "what": "reference loop body (poc/main.py:394-411) on the patched LossFunctions: zero_grad, LossFunctions, backward, "
                   "torch.optim.Adam.step, 4 history reads with .cpu(); float64 (n,1) tensors + torch.where index tuples; "
                   "host_ms_per_step splits the wall time by line (the .cpu() line absorbs the wait for the GPU)"}
    n = 1 << 22                      # BASELINE config 4's batch on one GPU: the host work hides behind the kernel
    res["cuda_resident_4M_points"] = loop(dev, batches(dev, 3), max(10, steps // 4))
    n = n_small
    return res


WORKLOAD = "ionHsym poc-form training step, 2^18 collocation points/step/GPU (BASELINE config 3)"


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=1 << 18, help="collocation points per GPU per step")
    ap.add_argument("--global-points", type=int, default=1 << 22,
                    help="BASELINE config 4: points per step of the WHOLE job, sharded over the ranks (extra key config4_global_batch)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling-legs-only", action="store_true",
                    help="N=1 run of a one-box scaling table: skip the legs that only run at N=1 (seam, reference autograd on the GPU, "
                         "grid quadrature, cpu_baseline) so that the line has exactly the legs the N>1 lines have")
    ap.add_argument("--no-extras", action="store_true",
                    help="only the headline timed regions (profiling runs): no e2e / seam / config-4 / training-loop legs")
    ap.add_argument("--allreduce", default="fused", choices=["fused", "nccl"],
                    help="N>1: sum over ranks fused into the reduction kernel over NVLink peer memory (pinn_dp_*), or a "
                         "separate NCCL all-reduce per step (the baseline it replaces)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them returned as DIR/<name>.npy (float64): "
                         "loss.npy (Ltot, Lpde, Lbc), dtheta.npy (1521) and sums.npy (the 8 sums of the C ABI); "
                         "--impl reference: loss.npy, dtheta.npy and E.npy (E per point, a fixed seeded sample of "
                         "%d points when the batch is larger)" % DUMP_MAX_POINTS)
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import pinn_for_quantum_wavefunction_surfaces_b200 as pk
    from pinn_for_quantum_wavefunction_surfaces_b200 import dp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # host buffers of this rank (page-locked batches of the e2e leg) are allocated on the NUMA node of its GPU
    numa_cpus = pk.bind_host_to_device_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.points
    W = max(args.warmup, 3)
    K = args.steps
    h = pk.Handle.get(local)
    fused = world > 1 and args.allreduce == "fused"
    if fused and not dp.attach_fused(h, strict=False):
        fused = False   # all ranks agreed: no peer mapping on this box -> the NCCL all-reduce path (reported in config)
        if rank == 0:
            print("bench: fused exchange unavailable, falling back to --allreduce nccl", file=sys.stderr)

    theta = torch.from_numpy(load_theta().astype(np.float32)).to(dev)
    parity = None
    if fused:
        parity = dp_parity_check(pk, dp, dist, h, dev, rank, world, theta)
        if not parity["ok_on_all_ranks"]:
            if rank == 0:
                emit({"metric": "collocation points/sec per training step (fwd+lap+bwd)", "value": None, "n_gpus": world,
                      "dp_parity": parity, "error": "data-parallel parity check failed; nothing was timed"})
            raise SystemExit(3)

    def make_batches(npts, nb, seed0):
        hb = [synth_batch(npts, seed0 + 1000 * rank + b).pin_memory() for b in range(nb)]
        db = [b.to(dev) for b in hb]
        # boundary sets are derived in-kernel (r >= 17.5); their global sizes for the 1/count weights come from a count
        # pass per batch done up front on the host (the sampler knows them in a real run), so that the only kernels this
        # process launches are the library's own
        ws = []
        for b in hb:
            r1 = torch.sqrt((b[0] - b[3]) ** 2 + b[1] ** 2 + b[2] ** 2)
            r2 = torch.sqrt((b[0] + b[3]) ** 2 + b[1] ** 2 + b[2] ** 2)
            ws.append(dp.global_weights(npts, int((r1 >= 17.5).sum()), int((r2 >= 17.5).sum()), device=dev))
        return hb, db, ws
    host_batches, dev_batches, wts = make_batches(n, N_BATCHES, 0)
    out = torch.zeros(dp.N_OUT, dtype=torch.float64, device=dev)

    def make_step(db, ws):
        nb = len(db)

        def step(i):
            b = db[i % nb]
            pk.loss_and_grad_raw(0, b[0], b[1], b[2], b[3], theta, None, ws[i % nb], sums=out[:8], dtheta=out[8:])
            if world > 1 and not fused:
                dist.all_reduce(out)
        return step
    step = make_step(dev_batches, wts)

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(stepfn, first, count):
        """`count` steps bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fence()
        e0.record()
        for i in range(count):
            stepfn(first + i)
        e1.record()
        fence()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for i in range(W):
        step(i)
    fence()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # the clock sampler needs ~0.15 s to deliver its first rows: the GPU keeps stepping meanwhile (more warm-up) instead of
    # idling, so that the timed region starts on a busy, clocked-up device straight after the fence
    # (the number of these steps must be the same on every rank - each one is an exchange - so it is agreed on first)
    t_spin = time.time()
    i_spin = W
    for _ in range(20):
        step(i_spin)
        i_spin += 1
    torch.cuda.synchronize()
    more = torch.tensor([int(0.25 / max(time.time() - t_spin, 1e-4)) * 20], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(more, op=dist.ReduceOp.MAX)
    for _ in range(min(int(more.item()), 20000)):
        step(i_spin)
        i_spin += 1
    torch.cuda.synchronize()
    # however long the spin-up took, the timed region starts on batch 0: its last step sees the same batch in every run
    i_spin = -(-i_spin // N_BATCHES) * N_BATCHES
    # Two back-to-back timed regions of the same K steps (clocks sampled over both): the first without any extra stream
    # operation gives `value`; the second brackets every step-kernel launch with CUDA events on the launching stream
    # (pinn_profile_begin/collect) and gives the kernel's average duration for the roofline.  (The event records sit
    # between the step kernel and its programmatic-dependent reduction kernel and cost a few microseconds per step, which
    # is why they are kept out of the first region.)
    launches0 = h.launch_count()
    t0 = time.time()
    ms = timed(step, i_spin, K)
    launches = h.launch_count() - launches0
    last = out.clone() if args.dump_outputs else None
    h.profile_begin()
    ms_profiled = timed(step, i_spin + K, K)
    kern_ms, kern_n = h.profile_collect()
    # the roofline's denominator, measured now on this device (clock samples of the same window)
    step_mhz = h.step_kernel_clock(torch.cuda.current_stream(dev).cuda_stream)   # CTA 0's own cycles / nanoseconds, last step
    fp32_peak, fp32_ms, fp32_mhz = h.measure_fp32_peak()
    steady = None
    if not args.no_extras:
        Ks = max(K, 1000)
        steady = {"value": float(n) * world * Ks / (timed(step, i_spin + 2 * K, Ks) * 1e-3), "unit": "points/s", "steps": Ks}
    t1 = time.time()
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    loss = float(out[0].item())
    line_extra = {}

    if not args.no_extras:
        # ---- end to end: host buffers through the C ABI (H2D of the batch, kernel, D2H of loss+gradient), every step
        th64 = np.ascontiguousarray(load_theta())
        wts_h = [np.ascontiguousarray(w.cpu().numpy()) for w in wts]   # the caller's sampler knows the set sizes
        # the public call of a host-resident caller: one prepared HostStep per (reused, pinned) batch buffer
        host_steps = [pk.HostStep("poc", b[0], b[1], b[2], b[3], device=local) for b in host_batches]

        def e2e_step(i):
            sums_h, dth_h = host_steps[i % N_BATCHES](th64, wts_h[i % N_BATCHES])
            if world > 1 and not fused:
                out[:8] = torch.from_numpy(sums_h).to(dev)
                out[8:] = torch.from_numpy(dth_h).to(dev)
                dist.all_reduce(out)

        Ke = max(3, min(K, 200))
        fence()
        for i in range(N_BATCHES + 3):   # one pass over every page-locked batch buffer first (the GPU's first touch of a
            e2e_step(i)                  # host page is slower), then the timed calls
        fence()
        te0 = time.time()
        for i in range(Ke):
            e2e_step(N_BATCHES + 3 + i)
        fence()
        te = (time.time() - te0) / Ke
        e2e_split = h.host_timing()   # of the last call
        h.profile_begin()             # the kernel's share, measured on a few more calls outside the timed loop
        for i in range(10):
            e2e_step(N_BATCHES + 3 + Ke + i)
        fence()
        e2e_kern_ms, e2e_kern_n = h.profile_collect()
        tte = torch.tensor([te], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tte, op=dist.ReduceOp.MAX)
        te = float(tte.item())
        line_extra["e2e"] = {
            "value": float(n) * world / te, "unit": "points/s", "h2d_bytes_per_step": int(16 * n + 1521 * 4),
            "d2h_bytes_per_step": int((8 + 1521) * 8), "ms_per_step": te * 1e3, "steps": Ke,
            "kernel_ms": e2e_kern_ms / max(e2e_kern_n, 1), "last_call_us": {k: round(v, 1) for k, v in e2e_split.items()},
            "api": "HostStep -> pinn_loss_fwd_bwd_host (pinned float32 host batches read in place by the kernel: bulk copies "
                   "(cp.async.bulk) of the next super-tile's columns over PCIe while the current one is computed; pageable "
                   "inputs are staged in up to 4 chunks)"}
        del host_steps
        # What the host link gives when all ranks pull their batches at once (plain cudaMemcpyAsync from the same page-locked
        # buffers, no kernel): the ceiling of the e2e path's scaling.  4.2 MB per step and GPU cross PCIe; on an HGX box
        # the GPUs share switch uplinks, so the aggregate stops growing long before 8 x the single-GPU rate.
        fence()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for rep in range(3):
            for hb, db in zip(host_batches, dev_batches):
                db.copy_(hb, non_blocking=True)
        c1.record()
        fence()
        gbs = torch.tensor([3 * N_BATCHES * 16.0 * n / (c0.elapsed_time(c1) * 1e-3) / 1e9], dtype=torch.float64, device=dev)
        gmin, gsum = gbs.clone(), gbs.clone()
        if world > 1:
            dist.all_reduce(gmin, op=dist.ReduceOp.MIN)
            dist.all_reduce(gsum, op=dist.ReduceOp.SUM)
        line_extra["e2e"]["host_link_probe"] = {
            "h2d_GBps_per_gpu_min": float(gmin.item()), "h2d_GBps_all_gpus": float(gsum.item()),
            "e2e_needs_GBps_per_gpu_at_device_rate": 16.0 * n / (ms / K * 1e-3) / 1e9,
            "what": "all ranks copy their page-locked batches host->device at once (cudaMemcpyAsync, no kernel)"}

        # ---- BASELINE config 4 as written: 2^22 points per step of the whole job, sharded over the ranks
        G = args.global_points
        n4 = G // world
        nb4 = max(4, -(-160_000_000 // (16 * n4)))      # rotating batches: > 126 MB L2 in total
        _, db4, w4 = make_batches(n4, nb4, 7000)
        # (make_batches -> dp.global_weights: the weights of a sharded batch are those of the GLOBAL batch)
        step4 = make_step(db4, w4)
        fence()                      # the ranks drew their batches on the host at different speeds: meet before exchanging
        for i in range(3):
            step4(i)
        K4 = max(3, min(K, 200))
        ms4 = timed(step4, 3, K4)
        line_extra["config4_global_batch"] = {
            "value": float(n4) * world * K4 / (ms4 * 1e-3), "unit": "points/s", "global_points": int(n4 * world),
            "points_per_gpu": int(n4), "ms_per_step": ms4 / K4, "steps": K4, "scaling": "strong",
            "inputs": "%d rotating batches of %.1f MB per GPU resident in HBM" % (nb4, 16 * n4 / 1e6),
            "what": "BASELINE config 4: 2^22 collocation points per step sharded over the ranks, one fused exchange per step"}
        del db4

        # ---- the whole training loop on the device (sampler -> loss/gradient -> Adam, CUDA-graph replay)
        if world == 1 or fused:
            tr = pk.Trainer("poc", n, load_theta(), seed=1, lr=1e-6, device=local)
            fence()
            Kl = max(10, min(K, 300))
            ts = torch.cuda.ExternalStream(tr.h.L.pinn_trainer_stream(tr.t), device=dev)
            res = {}
            for graph in (False, True):
                tr.run(20, use_graph=graph)
                tr.read()
                l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                l0.record(ts)
                tr.run(Kl, use_graph=graph)
                l1.record(ts)
                tr.read()
                lms = torch.tensor([l0.elapsed_time(l1)], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(lms, op=dist.ReduceOp.MAX)
                res[graph] = n * world * Kl / (float(lms.item()) * 1e-3)
            line_extra["device_train_loop"] = {
                "value": res[False], "unit": "points/s", "steps": Kl, "value_with_cuda_graph_replay": res[True],
                "what": "pinn_trainer: per step the fused loss/gradient kernel and one kernel with reduction%s + float64 Adam + "
                        "Philox sampler of the next batch, launched as programmatic dependents, no host sync"
                        % (" + set-size and gradient exchange over NVLink" if world > 1 else "")}
            tr.close()

        # ---- N = 1: the seam itself, and two more reference points (BASELINE configs 2 and 5)
        if world == 1 and not args.scaling_legs_only:
            line_extra["seam_e2e"] = seam_e2e(pk, dev, n, max(20, min(K, 100)))
            if not args.no_cpu_baseline:
                line_extra["reference_autograd_on_gpu"] = ref_autograd_on_gpu(load_theta(), dev)
                line_extra["dense_grid_inference"] = dense_grid_inference(dev)

    if rank == 0:
        total_points = float(n) * world
        value = total_points * K / (ms * 1e-3)
        kern_avg_ms = kern_ms / max(kern_n, 1)
        achieved = FLOP_PER_POINT * n / (kern_avg_ms * 1e-3)
        traffic, ncu_pipes, ncu_src = committed_ncu_figures()
        line = {
            "metric": "collocation points/sec per training step (fwd+lap+bwd)",
            "value": value, "unit": "points/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "ms_per_step_with_kernel_events": ms_profiled / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "points_per_gpu": n, "global_points": int(total_points), "weights": "models/ionHsym.pt (tests/golden/checkpoints.npz)",
                       "inputs": "%d rotating batches resident in HBM, %.0f MB > 126 MB L2" % (N_BATCHES, N_BATCHES * n * 16 / 1e6),
                       "warmup_note": "%d warm-up steps, then %d more untimed steps while the clock sampler starts (no idle gap in front of the timed region)" % (W, i_spin - W),
                       "host_numa_binding": ("rank 0 bound to CPUs %s-%s of its GPU's NUMA node" % (numa_cpus[0], numa_cpus[-1])) if numa_cpus else "none",
                       "parallelism": ("dp%d point sharding; sum of 1529 f64 over ranks %s" % (
                           world, "fused into the reduction kernel (NVLink peer stores + flags, pinn_dp_*)" if fused
                           else "by one NCCL all-reduce per step")) if world > 1 else "single GPU"},
            "roofline": {"bound": "fp32_ffma", "achieved": achieved / 1e12, "peak": fp32_peak / 1e12,
                         "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                         "frac_of_nominal_74.4": achieved / FP32_PEAK_NOMINAL,
                         "frac_of_round1_peak_72.0": achieved / FP32_PEAK_FALLBACK,
                         "peak_source": "FFMA rate measured in this run on this device (pinn_measure_fp32_peak: register-resident "
                                        "FFMA loop, best of 8 x 10 launches, %.3f ms per timed kernel, clocks in `clocks`); MEASURED_PEAKS.json has no FP32 entry; "
                                        "round-1 figure of the same loop: %.1f" % (fp32_ms, FP32_PEAK_FALLBACK / 1e12),
                         "flop_per_point": FLOP_PER_POINT,
                         # the SM clock each kernel actually ran at (block 0 times itself: clock64 / %globaltimer): the step
                         # kernel keeps the tensor pipe busy and runs below the clock the FFMA loop (and nvidia-smi) see
                         "effective_sm_mhz": {"step_kernel": round(step_mhz, 1), "ffma_peak_loop": round(fp32_mhz, 1)},
                         "frac_at_the_step_kernels_own_clock": achieved / (fp32_peak * step_mhz / fp32_mhz) if fp32_mhz > 0 and step_mhz > 0 else None,
                         "kernel": "pinn_step_tc_kernel<2,true,false>",
                         "kernel_ms": kern_avg_ms, "kernel_launches_timed": kern_n, "traffic": traffic,
                         "algorithmic_bytes_per_launch": 16 * n, "ncu_pipe_utilisation_pct": ncu_pipes, "ncu_source": ncu_src,
                         "vs_hbm_ceiling": hbm_ceiling(16 * n, kern_avg_ms),
                         "vs_3xtf32_tensor_ceiling": tensor_ceiling(FLOP_PER_POINT * n, kern_avg_ms)},
            "gpu_launches": int(launches), "clocks": clocks, "loss": loss,
        }
        if steady:
            line["value_steady"] = steady
        if parity:
            line["dp_parity"] = parity
        line.update(line_extra)
        if "e2e" not in line:
            line["e2e"] = None
        if "dense_grid_inference" in line:
            line["dense_grid_inference"]["frac_of_fp32_peak"] = line["dense_grid_inference"]["tflops"] * 1e12 / fp32_peak
        if not args.no_cpu_baseline and world == 1 and not args.no_extras and not args.scaling_legs_only:
            v, cores, sample, _ = cpu_reference_points_per_s(np.ascontiguousarray(load_theta()), args.cpu_seconds, n)
            line["cpu_baseline"] = {"value": v, "unit": "points/s", "cores": cores, "kind": "port", "sample": sample}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, loss=last[:3], dtheta=last[8:], sums=last[:8])
        emit(line)
    if fused:
        h.dp_status()
        dp.detach_fused(h)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
