"""GPU tests of the rows next to the hot path (SURVEY.md 8f): sampler, fused Adam, device-resident trainer, training
trajectory parity with the reference run, dense-grid quadrature, E(R) curve.  Everything goes through the C ABI."""
import json
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf
from oracle import layout
from oracle import philox as ph
from oracle import simpson as sp
from oracle import train_loop as tl
from oracle.regimes import REGIMES, regime_theta

pytestmark = pytest.mark.gpu
OFFS = layout.offsets() + [1521]


def dev():
    return torch.device("cuda:0")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


@pytest.fixture(scope="module")
def ck(golden_dir):
    return np.load(os.path.join(golden_dir, "checkpoints.npz"))


@pytest.fixture(scope="module")
def init_theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]


# ---------------------------------------------------------------------------------------------
# sampler: bit-exact with the numpy restatement of the published Philox4x32-10 stream and the reference's clamp rules
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,seed,batch", [(1, 1, 0), (1000, 12345, 0), (4097, 7, 3), (100000, 2 ** 40 + 5, 2 ** 33 + 1)])
def test_sampler_bit_exact(n, seed, batch):
    for box in (pk.trainer.BOX_POC, pk.trainer.BOX_TRAINPY):
        out = pk.sample(n, seed, batch, box=box)
        x, y, z, R, mask, cnt = ph.sample_batch(n, seed, batch, box=box)
        for k, ref in zip("xyzR", (x, y, z, R)):
            assert np.array_equal(out[k].cpu().numpy(), ref), k
        assert np.array_equal(out["mask"].cpu().numpy(), mask)
        assert tuple(out["counts"].cpu().tolist()) == cnt
        assert np.allclose(out["weights"].cpu().numpy(), [1.0 / n, 1.0 / cnt[0] if cnt[0] else np.inf,
                                                          1.0 / cnt[1] if cnt[1] else np.inf], rtol=1e-15)


def test_sampler_clamp_rule_and_full_size():
    out = pk.sample(64, 1, 0, box=(0.999, 1.001, -1e-3, 1e-3, -1e-3, 1e-3, 1.0, 1.0 + 1e-7))
    assert torch.all(out["x"] == 0.005)          # the reference writes the VALUE cutoff into x (train.py:34-35)
    n = 1 << 22                                   # BASELINE config 4 batch: counts == popcount, box respected
    o = pk.sample(n, 99, 5)
    m = o["mask"]
    assert int((m & 1).sum()) == int(o["counts"][0]) and int((m >> 1).sum()) == int(o["counts"][1])
    assert float(o["x"].min()) >= -18 and float(o["x"].max()) <= 18 and 0.2 <= float(o["R"].min()) and float(o["R"].max()) <= 4
    assert abs(float(o["R"].mean()) - 2.1) < 5e-3 and abs(float(o["y"].mean())) < 3e-2
    r1 = torch.sqrt((o["x"].double() - o["R"].double()) ** 2 + o["y"].double() ** 2 + o["z"].double() ** 2)
    far = (r1 - 17.5).abs() > 1e-3
    assert torch.equal(((m & 1) == 1)[far], (r1 >= 17.5)[far])


# ---------------------------------------------------------------------------------------------
# fused Adam vs torch.optim.Adam (the reference's optimizer), float64
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("frozen", [False, True])
def test_adam_step_matches_torch_adam(frozen, init_theta):
    rng = np.random.default_rng(3)
    grads = [rng.standard_normal(1521) * 10.0 ** rng.integers(-8, 0) for _ in range(6)]
    gm = pk.FINE_TUNE_GRAD_MASK if frozen else 0xFFFF
    fz = np.ones(1521, bool)
    for i in range(16):
        if (gm >> i) & 1:
            fz[OFFS[i]:OFFS[i + 1]] = False
    ref = tl.adam_reference(init_theta, grads, lr=8e-3, frozen=fz if frozen else None)
    st = pk.AdamState(init_theta, history_capacity=8, best_mode=0)
    losses = [3.0, 2.0, 2.5, 1.0, float("nan"), 1.5]
    for k, g in enumerate(grads):
        sums = torch.tensor([losses[k], 0.1, 0.2, 7.0 * 50, 0, 0, 0, -0.6], dtype=torch.float64, device=dev())
        pre = st.theta.clone()
        pk.adam_step(st, torch.from_numpy(g).to(dev()), sums, n=50, lr=8e-3, grad_mask=gm)
        torch.cuda.synchronize()
        assert np.allclose(st.theta.cpu().numpy(), ref[k], rtol=1e-13, atol=1e-16), k
        assert torch.equal(st.theta32, st.theta.float())
        if k in (0, 1, 3):   # train.py:58-60: first loss, then every improvement; parameters BEFORE the step are kept
            assert torch.equal(st.best_theta, pre) and float(st.best_loss) == losses[k] and int(st.best_step) == k
    assert int(st.step) == 6 and float(st.best_loss) == 1.0 and int(st.best_step) == 3   # NaN never wins
    h = st.hist.cpu().numpy()
    assert np.allclose(h[:4, 0], losses[:4]) and np.allclose(h[:6, 3], 7.0) and np.isnan(h[4, 0])
    if frozen:
        assert np.array_equal(st.theta.cpu().numpy()[fz], init_theta[fz]) and float(st.m.abs()[torch.from_numpy(fz).to(dev())].max()) == 0


def test_adam_poc_best_rule(init_theta):
    """poc/main.py:414-417: after half the epochs, on improvement over Llim (starts at 10), the POST-step model is saved."""
    st = pk.AdamState(init_theta, history_capacity=4, best_mode=1)
    g = torch.ones(1521, dtype=torch.float64, device=dev())
    for k, L in enumerate([0.5, 0.4, 0.3, 0.35]):
        sums = torch.tensor([L, 0, 0, 0, 0, 0, 0, -0.7], dtype=torch.float64, device=dev())
        pk.adam_step(st, g, sums, n=10, best_after=1, history_mean_E=False)
        torch.cuda.synchronize()
        if k == 2:
            assert torch.equal(st.best_theta, st.theta) and int(st.best_step) == 2
    assert float(st.best_loss) == 0.3 and np.allclose(st.hist.cpu().numpy()[:, 3], -0.7)


# ---------------------------------------------------------------------------------------------
# trainer: graph replay == plain launches == a host loop over the same kernels
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["trainpy", "poc"])
def test_trainer_equals_step_by_step_host_loop(variant, init_theta):
    n, steps, seed = 5000, 6, 4242
    v = 0 if variant == "poc" else 1
    res = {}
    for graph in (True, False):
        tr = pk.Trainer(variant, n, init_theta, seed=seed, lr=8e-3, history_capacity=steps)
        tr.run(steps, use_graph=graph)
        res[graph] = tr.read()
        tr.close()
    for k in ("theta", "m", "v", "best_theta", "history"):
        assert np.array_equal(res[True][k], res[False][k]), k      # graph replay changes nothing
    assert res[True]["steps"] == steps and res[True]["batches"] == steps
    # the same loop driven from the host: sampler -> fused loss -> torch.optim.Adam in float64
    box = pk.trainer.BOX_POC if v == 0 else pk.trainer.BOX_TRAINPY
    p = torch.tensor(init_theta, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([p], lr=8e-3)
    hist = []
    for t in range(steps):
        b = pk.sample(n, seed, t, box=box)
        sums, dth, _ = pk.loss_and_grad_raw(v, b["x"], b["y"], b["z"], b["R"], p.detach().float().to(dev()), b["mask"],
                                            b["weights"], want_E=True)
        hist.append(sums.cpu().numpy())
        p.grad = dth.cpu()
        opt.step()
    assert np.allclose(res[True]["theta"], p.detach().numpy(), rtol=1e-10, atol=1e-13)
    H = np.array(hist)
    assert np.allclose(res[True]["history"][:, :3], H[:, :3], rtol=1e-12)
    col3 = H[:, 3] / n if v == 1 else H[:, 7]
    assert np.allclose(res[True]["history"][:, 3], col3, rtol=1e-12)


def test_trainer_in_flight_does_not_disturb_calls_on_other_streams(init_theta):
    """ADVICE r1: Trainer.run() is asynchronous on the trainer's own stream; evaluations on torch's stream (and a second
    trainer) while it is in flight used to share the handle's partial-row workspace.  Every stream has its own now: the
    results are those of the same calls made alone, and the trainers' trajectories those of trainers run alone."""
    n, steps = 1 << 16, 120
    alone = {}
    for seed in (11, 22):
        tr = pk.Trainer("poc", n, init_theta, seed=seed, lr=8e-3, history_capacity=steps)
        tr.run(steps)
        alone[seed] = tr.read()
        tr.close()
    b = pk.sample(50000, 5, 0)
    th = torch.from_numpy(init_theta.astype(np.float32)).to(dev())
    s0, g0, _ = pk.loss_and_grad_raw(0, b["x"], b["y"], b["z"], b["R"], th, b["mask"], b["weights"])
    s0, g0 = s0.clone(), g0.clone()
    torch.cuda.synchronize()
    t1 = pk.Trainer("poc", n, init_theta, seed=11, lr=8e-3, history_capacity=steps)
    t2 = pk.Trainer("poc", n, init_theta, seed=22, lr=8e-3, history_capacity=steps)
    t1.run(steps)                       # both return at once; ~2 x 120 steps of work are now queued on two streams
    t2.run(steps)
    for _ in range(40):                 # ... and these run concurrently with them on torch's stream
        s, g, _ = pk.loss_and_grad_raw(0, b["x"], b["y"], b["z"], b["R"], th, b["mask"], b["weights"])
        assert torch.equal(s[:7], s0[:7]) and torch.equal(g, g0)
    r1, r2 = t1.read(), t2.read()
    t1.close(); t2.close()
    for r, seed in ((r1, 11), (r2, 22)):
        assert np.array_equal(r["theta"], alone[seed]["theta"]) and np.array_equal(r["history"], alone[seed]["history"])


def test_workspace_recycling_spares_streams_whose_calls_were_captured(init_theta):
    """A handle keeps at most 32 per-stream workspaces and recycles the least recently used one.  A trainer's captured
    graphs carry its workspace's addresses, so that one must survive any number of other streams coming and going; a
    closed trainer gives its workspace back."""
    n, steps = 4096, 8
    ref = pk.Trainer("poc", n, init_theta, seed=3, lr=8e-3, history_capacity=2 * steps)
    ref.run(2 * steps)
    want = ref.read()
    ref.close()
    tr = pk.Trainer("poc", n, init_theta, seed=3, lr=8e-3, history_capacity=2 * steps)
    tr.run(steps)                                         # graphs captured here
    tr.read()
    b = pk.sample(3000, 5, 0)
    th = torch.from_numpy(init_theta.astype(np.float32)).to(dev())
    s0, g0, _ = pk.loss_and_grad_raw(0, b["x"], b["y"], b["z"], b["R"], th, b["mask"], b["weights"])
    s0, g0 = s0.clone(), g0.clone()
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(40)]    # more streams than workspaces: the oldest are recycled
    for st in streams:
        with torch.cuda.stream(st):
            s, g, _ = pk.loss_and_grad_raw(0, b["x"], b["y"], b["z"], b["R"], th, b["mask"], b["weights"])
        st.synchronize()
        assert torch.equal(s[:7], s0[:7]) and torch.equal(g, g0)
    for _ in range(40):                                   # trainers come and go: their slots are given back
        t = pk.Trainer("poc", 512, init_theta, seed=1, history_capacity=2)
        t.run(2)
        t.close()
    tr.run(steps)                                         # graph replay after all that
    got = tr.read()
    tr.close()
    assert np.array_equal(got["theta"], want["theta"]) and np.array_equal(got["history"], want["history"])


def test_trainer_freeze_and_resample_schedule(init_theta):
    """poc/main.py:396: resample iff tt % sc_sampling == 0 and tt < 0.9*epochs."""
    tr = pk.Trainer("poc", 2048, init_theta, sc_sampling=2, freeze_after=5, history_capacity=10)
    tr.run(10)
    r = tr.read()
    tr.close()
    assert r["steps"] == 10 and r["batches"] == 3       # tt = 0, 2, 4
    # the last five steps see one frozen batch: the loss changes only through the parameters, smoothly
    assert np.all(np.isfinite(r["history"]))


def test_trainer_fine_tune_mask_and_resume(ck):
    th = ck["ionHsym"]
    tr = pk.Trainer("poc", 4096, th, lr=5e-4, grad_mask=pk.FINE_TUNE_GRAD_MASK, history_capacity=4)   # poc/main.py:938-942
    tr.run(4)
    r = tr.read()
    same = np.ones(1521, bool)
    same[OFFS[6]:OFFS[12]] = False
    assert np.array_equal(r["theta"][same], th[same]) and not np.array_equal(r["theta"][~same], th[~same])
    tr2 = pk.Trainer("poc", 4096, th, lr=5e-4, grad_mask=pk.FINE_TUNE_GRAD_MASK, history_capacity=4)
    tr2.run(2)
    mid = tr2.read()
    tr3 = pk.Trainer("poc", 4096, th, lr=5e-4, grad_mask=pk.FINE_TUNE_GRAD_MASK, history_capacity=4)
    tr3.load_state(mid["theta"], mid["m"], mid["v"], step=2)     # resume: optimizer state + step count
    tr3.cfg  # batches restart at 0 for the new trainer: feed the batches 2, 3 explicitly to continue the same run
    for t in (2, 3):
        b = pk.sample(4096, 12345, t)
        tr3.set_batch(b["x"], b["y"], b["z"], b["R"], b["mask"], b["weights"].cpu().numpy())
        tr3.run(1, resample=False, use_graph=False)
    r3 = tr3.read()
    assert np.allclose(r3["theta"], r["theta"], rtol=1e-12, atol=1e-15)
    # the resumed run keeps its own history (row 0 = first step after the resume) and its own best-model record
    assert r3["steps"] == 4 and r3["history"].shape == (2, 4) and np.allclose(r3["history"], r["history"][2:4], rtol=1e-12)
    assert r3["best_step"] in (2, 3) and r3["best_loss"] == r3["history"][r3["best_step"] - 2, 0]
    fresh = pk.Trainer("trainpy", 4096, th, history_capacity=4)
    fresh.load_state(mid["theta"], mid["m"], mid["v"], step=2)
    r0 = fresh.read()
    assert np.array_equal(r0["best_theta"], mid["theta"]) and r0["best_step"] == -1 and r0["history"].shape == (0, 4)
    fresh.run(1)                        # train.py rule: the first step after a (re)start is taken unconditionally
    r1 = fresh.read()
    assert r1["best_step"] == 2 and np.array_equal(r1["best_theta"], mid["theta"]) and r1["history"].shape == (1, 4)
    fresh.close()
    for t in (tr, tr2, tr3):
        t.close()


# ---------------------------------------------------------------------------------------------
# training trajectory: the reference run (train.py, n=4096, 40 epochs, torch RNG seed 12345) with the fused op
# ---------------------------------------------------------------------------------------------
def _enet_np(theta, R):
    P = layout.unpack_poc(np.asarray(theta, np.float64))
    sig = lambda u: 1.0 / (1.0 + np.exp(-u))
    e = sig(R[:, None] * P[6][:, 0][None, :] + P[7][None, :])
    e = sig(e @ P[8].T + P[9][None, :])
    return e @ P[10][0] + P[11][0]


@pytest.mark.parametrize("epochs", [40, 200])
def test_reference_training_run_with_fused_loss_matches_golden_model(golden_dir, epochs):
    """BASELINE north star: trained E(R) within 1e-4 Hartree of the reference run; BASELINE config 1 is this run at
    n = 4096, 200 epochs.  The reference's own loop (restated in oracle/train_loop.py, pinned to the real script on the CPU at
    both lengths) is driven with the CUDA op instead of lines 41-57; same torch RNG stream, same Adam, float64 parameters
    on the host.  Measured on B200 (profiles/r02_a_acceptance.txt): max|dE(R)| 8e-8 Ha and max|dtheta| 7e-7 against the real
    script's model.bin after 200 epochs; the bars are 10x that, far inside the north star's 1e-4 Ha."""
    tr = json.load(open(os.path.join(golden_dir, "trainpy_trace_n4096_e%d.json" % epochs)))
    params, trace, hist = tl.trainpy_run(pk.loss_trainpy, n=4096, epochs=epochs)
    assert trace[0] == tr["trace"][0]                      # identical print at step 0
    assert len(trace) == len(tr["trace"])
    fa = lambda ln: [float(v) for v in ln.replace("(", " ").replace(")", " ").replace("[", " ").replace("]", " ").split()[1:]]
    for a, b in zip(trace, tr["trace"]):                   # 3 printed digits: one unit of the last digit is <= 1e-2
        assert np.allclose(fa(a), fa(b), rtol=1.1e-2), (a, b)
    got = pk.pack_trainpy(params, dtype=torch.float64).numpy()
    ref = pk.convert.theta_from_model_bin(os.path.join(golden_dir, "trainpy_model_n4096_e%d.bin" % epochs))
    R = np.linspace(0.2, 3.0, 57)
    dE = np.abs(_enet_np(got, R) - _enet_np(ref, R)).max()
    assert dE < 1e-6, dE
    assert np.abs(got - ref).max() < 1e-5


@pytest.mark.parametrize("epochs", [40, 200])
def test_device_trainer_fed_with_the_reference_points_tracks_the_reference(golden_dir, init_theta, epochs):
    """Same run through the device-resident trainer (fused Adam, float64 state on the GPU): the host only supplies the
    reference's batches (torch RNG, train.py:26-39)."""
    torch.manual_seed(12345)
    tl.trainpy_run  # the parameter draw consumes the generator first, exactly as in the script
    n = 4096
    dtype = torch.double
    shapes = [(2, 16), (16,), (16, 16), (16,), (16, 1), (1,), (1, 10), (10,), (10, 1), (1,), (1, 32), (32,), (32, 32), (32,),
              (32, 1), (1,)]
    ps = []
    for s in shapes:
        t = torch.empty(s, dtype=dtype)
        t.uniform_(-1 / s[0] ** 0.5, 1 / s[0] ** 0.5)
        ps.append(t)
    theta0 = pk.pack_trainpy(ps, dtype=dtype).numpy()
    assert np.array_equal(theta0, init_theta)
    x, y, z, R = [torch.empty(n, 1, dtype=dtype) for _ in range(4)]
    tr = pk.Trainer("trainpy", n, theta0, lr=8e-3, history_capacity=epochs + 1)
    for tt in range(epochs + 1):
        x.uniform_(-18, 18); y.uniform_(-18, 18); z.uniform_(-18, 18); R.uniform_(0.2, 3)
        r1sq = (x - R) ** 2 + y ** 2 + z ** 2
        r2sq = (x + R) ** 2 + y ** 2 + z ** 2
        x[r1sq < 0.005 ** 2] = 0.005
        x[r2sq < 0.005 ** 2] = 0.005
        m1 = ((x - R) ** 2 + y ** 2 + z ** 2 >= 17.5 ** 2)[:, 0]
        m2 = ((x + R) ** 2 + y ** 2 + z ** 2 >= 17.5 ** 2)[:, 0]
        mask = (m1.to(torch.uint8) + 2 * m2.to(torch.uint8))
        tr.set_batch(x.float(), y.float(), z.float(), R.float(), mask, [1.0 / n, 1.0 / int(m1.sum()), 1.0 / int(m2.sum())])
        tr.run(1, resample=False, use_graph=(tt > 0))
    r = tr.read()
    tr.close()
    gt = json.load(open(os.path.join(golden_dir, "trainpy_trace_n4096_e%d.json" % epochs)))["trace"]
    for k, ln in enumerate(gt):
        vals = [float(v) for v in ln.replace("(", " ").replace(")", " ").replace("[", " ").replace("]", " ").split()[1:]]
        assert np.allclose(r["history"][10 * k], vals[:4], rtol=1.1e-2), (k, r["history"][10 * k], vals)
    ref = pk.convert.theta_from_model_bin(os.path.join(golden_dir, "trainpy_model_n4096_e%d.bin" % epochs))
    Rg = np.linspace(0.2, 3.0, 57)
    # measured 8e-8 Ha after 200 epochs (profiles/r02_a_acceptance.txt); the north star asks for 1e-4
    assert np.abs(_enet_np(r["best_theta"], Rg) - _enet_np(ref, Rg)).max() < 1e-6
    best_ref = {40: 7.18217e-06, 200: 1.00569e-06}[epochs]      # last [Lbest] of the real script's trace
    assert abs(r["best_loss"] - best_ref) / best_ref < 1e-4


def test_train_drivers_reduce_the_loss(init_theta):
    best, info = pk.train_trainpy(n=8192, epochs=60, seed=12345)
    assert info["history"].shape == (61, 4) and info["history"][-1, 0] < 0.05 * info["history"][0, 0]
    assert info["best_loss"] == info["history"][:, 0].min() and best.shape == (1521,)
    last, saved, loss = pk.train_poc(init_theta, {"n_train": 8192, "epochs": 40, "lr": 8e-3})
    assert loss["Ltot"].shape == (40, 1) and loss["Ltot"][-1, 0] < loss["Ltot"][0, 0] and saved is not None
    assert set(loss) == {"Ltot", "Lpde", "Lbc", "Energy"}


def test_paper_schedule_on_the_device_matches_the_reference_rerun(golden_dir):
    """north star: 'reference-matching E(R) curves'.  The paper schedule (poc/main.py:919-942: 100 000 points x 5000 Adam steps
    @ 8e-3, then 2000 fine-tune steps @ 5e-4 on the E-net from the saved best model) runs on the device in half a second and
    is compared with the REAL reference run of the same schedule (tests/golden/poc_paper_run_seed0.npz, made on the CPU by
    tests/golden/make_paper_run.py: 85 minutes) and with exactE() (poc/main.py:48-61).

    What the reference itself delivers when re-run (seed 0): max|E_net - exact| = 1.8e-2 after the main stage, 2.4e-2 (R >= 1)
    / 1.9e-2 (R >= 2) after the fine-tune, min Ltot 4.5e-7 / 4.2e-7 - the authors' own table (poc/energy_R_ion.pkl, 6.4e-3 /
    3.1e-3) is a better draw of the same procedure: their checkpoint BEFORE the fine-tune has 2.1e-2 as well, and 2000 steps
    move E_net only part of the way to where it is heading (below).  The runs use different random streams (torch CPU vs
    Philox), so the comparison is statistical: bars = 1.5 x the reference rerun's own errors.  Measured on B200
    (profiles/r02_j_acceptance.txt), seeds 0 / 1 / 2: 1.9e-2 / 5.0e-2 / 2.1e-2 (R >= 1), 1.8e-2 / 1.9e-2 / 1.8e-2 (R >= 2)."""
    ref = np.load(os.path.join(golden_dir, "poc_paper_run_seed0.npz"))
    Rt, Eex = ref["R"], ref["E_exact"]
    err = lambda th, lo: float(np.abs(_enet_np(th, Rt) - Eex)[Rt >= lo - 1e-9].max())
    theta0 = pk.init_poc(0)
    assert np.array_equal(theta0, ref["theta_init"])                     # same starting point as the reference run
    ref_err = {k: (err(ref["theta_" + k + "_saved"], 1.0), err(ref["theta_" + k + "_saved"], 2.0)) for k in ("stage1", "stage2")}
    assert abs(ref_err["stage2"][0] - 2.356e-2) < 1e-4 and abs(ref_err["stage2"][1] - 1.894e-2) < 1e-4
    last1, saved1, loss1 = pk.train_poc(theta0, {"n_train": 100000, "epochs": 5000, "lr": 8e-3}, seed=0)
    assert saved1 is not None and np.all(np.isfinite(loss1["Ltot"]))
    assert loss1["Ltot"].min() < 2 * ref["loss1_Ltot"].min()             # 4.2e-7 measured vs 4.46e-7
    assert err(saved1, 1.0) < 1.5 * max(ref_err["stage1"][0], ref_err["stage2"][0])
    last2, saved2, loss2 = pk.train_poc(saved1, {"n_train": 100000, "epochs": 2000, "lr": 5e-4}, freezeUnits=True, seed=1000)
    assert saved2 is not None and loss2["Ltot"].min() < 2 * ref["loss2_Ltot"].min()
    frozen = np.ones(1521, bool)
    frozen[OFFS[6]:OFFS[12]] = False
    assert np.array_equal(saved2[frozen], saved1[frozen])                 # freezeBase + freezeDecayUnit (poc/main.py:305-319)
    e1, e2 = err(saved2, 1.0), err(saved2, 2.0)
    print("paper schedule on the device: max|E_net - exact| %.2e (R>=1) %.2e (R>=2); reference rerun %.2e / %.2e; authors' table 6.4e-03 / 3.1e-03"
          % (e1, e2, ref_err["stage2"][0], ref_err["stage2"][1]))
    assert e1 < 1.5 * ref_err["stage2"][0] and e2 < 1.5 * ref_err["stage2"][1]
    # the two fine-tuned curves agree with each other as well as either agrees with the exact one
    d = np.abs(_enet_np(saved2, Rt) - ref["E_net_stage2"])
    assert d[Rt >= 2.0 - 1e-9].max() < 1.5e-2 and d[Rt >= 1.0 - 1e-9].max() < 3.5e-2
    # where the fine-tune is heading: with psi frozen, the E(R) minimising mean(res^2) is the Rayleigh quotient of that psi
    _, saved3, _ = pk.train_poc(saved1, {"n_train": 100000, "epochs": 40000, "lr": 5e-4}, freezeUnits=True, seed=2000)
    for Rv in (1.0, 2.0, 3.0):
        g = pk.analysis.grid_sums(saved3, Rv, n=400)
        E_int = g["psiHpsi"] / g["psi2"]
        E_net = float(_enet_np(saved3, np.array([Rv]))[0])
        assert abs(E_net - E_int) < 3e-3, (Rv, E_net, E_int)             # measured 1.6e-3 / 5e-4 / 7e-4
        exact = float(Eex[np.argmin(np.abs(Rt - Rv))])
        assert exact - 1e-3 < E_int < exact + 2e-2                        # variational: above the exact energy, by ~1e-2


# ---------------------------------------------------------------------------------------------
# dense-grid quadrature and the E(R) curve
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [12, 13])
@pytest.mark.parametrize("rule", ["avg", "simpson"])
def test_grid_energies_vs_oracle(n, rule, ck):
    th32 = ck["ionHsym_fineTune"].astype(np.float32)
    prm = {"n_test": n}
    ax = np.linspace(-18, 18, n)
    X, Y, Z = np.meshgrid(ax, ax, ax, indexing="ij")
    for Ri in (0.7, 2.0):
        f = cf.fields("poc", th32.astype(np.float64), X.ravel(), Y.ravel(), Z.ravel(), np.full(X.size, Ri))
        w1 = (sp.weights_avg if rule == "avg" else sp.weights_simpson)(n, ax[1] - ax[0])
        W = np.einsum("i,j,k->ijk", w1, w1, w1).ravel()
        r1 = np.sqrt((X - Ri) ** 2 + Y ** 2 + Z ** 2).ravel()
        r2 = np.sqrt((X + Ri) ** 2 + Y ** 2 + Z ** 2).ravel()
        lc = np.exp(-r1) + np.exp(-r2)
        hl = -0.5 * (np.exp(-r1) * (1 - 2 / r1) + np.exp(-r2) * (1 - 2 / r2)) - (1 / r1 + 1 / r2) * lc
        vr = -(X.ravel() - Ri) / r1 ** 3 + (X.ravel() + Ri) / r2 ** 3
        ref = {"psiHpsi": W @ (f["psi"] * f["hpsi"]), "psi2": W @ f["psi"] ** 2, "lcaoHlcao": W @ (lc * hl), "lcao2": W @ lc ** 2,
               "dVdR_psi2": W @ (vr * f["psi"] ** 2), "E_net": f["E"][-1]}
        got = pk.analysis.grid_sums(th32, Ri, prm, rule=rule)
        for k in ref:
            assert abs(got[k] - ref[k]) <= 2e-5 * abs(ref[k]) + 1e-9, (k, got[k], ref[k])
        if rule == "avg":   # the reference's nested simps (integra3d, poc/main.py:179-186) is the same number
            F = (f["psi"] * f["hpsi"]).reshape(n, n, n)
            assert abs(sp.integra3d(ax, ax, ax, F) - ref["psiHpsi"]) < 1e-10 * abs(ref["psiHpsi"])
        Eint, Enet = pk.analysis.energy_from_psi(th32, Ri, prm, rule=rule)
        assert abs(Eint - ref["psiHpsi"] / ref["psi2"]) < 2e-5 * abs(Eint) and abs(Enet - f["E"][-1]) < 1e-6
        assert abs(pk.analysis.energy_from_psi_LCAO(th32, Ri, prm, rule=rule) - ref["lcaoHlcao"] / ref["lcao2"]) < 1e-5
        assert abs(pk.analysis.dEdR_int(th32, Ri, prm, rule=rule) - (ref["dVdR_psi2"] / ref["psi2"] - 0.5 / Ri ** 2)) < 1e-4


@pytest.mark.parametrize("variant", ["poc", "trainpy"])
def test_grid_sums_equal_the_per_point_fields_summed_on_the_host(variant, ck, init_theta):
    """Grid launches evaluate E(R) and the gate once per CTA and keep the E-net role out of the tile loop; per-point
    inference (`fields`) evaluates them at every point.  Same psi, H psi and E: the quadrature of the per-point fields with
    the same weights is the grid kernel's sums (many super-tiles per CTA, both forms of the model, ragged last tile)."""
    th32 = (ck["ionHsym_fineTune"] if variant == "poc" else init_theta).astype(np.float32)
    n, Ri = 59, 1.3                                        # 205 379 points = 1605 super-tiles, the last one ragged
    ax = np.linspace(-18, 18, n)
    X, Y, Z = np.meshgrid(ax, ax, ax, indexing="ij")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a.ravel())).to(dev())
    f = pk.fields(variant, t(X), t(Y), t(Z), t(np.full(X.size, Ri)), torch.from_numpy(th32).to(dev()))
    psi, hpsi = f["psi"].cpu().numpy(), f["hpsi"].cpu().numpy()
    w1 = sp.weights_avg(n, ax[1] - ax[0])
    W = np.einsum("i,j,k->ijk", w1, w1, w1).ravel()
    got = pk.analysis.grid_sums(th32, Ri, {"n_test": n}, variant=variant)
    ref = {"psiHpsi": W @ (psi * hpsi).astype(np.float64), "psi2": W @ (psi * psi).astype(np.float64)}
    for k in ref:
        assert abs(got[k] - ref[k]) <= 1e-9 * abs(ref[k]), (k, got[k], ref[k])
    assert got["E_net"] == float(f["E"].cpu().numpy()[-1])


def test_grid_point_on_a_nucleus_gives_nan_like_the_reference(ck):
    """Odd n_test puts x = y = z = 0 ... on the grid; with R a multiple of the spacing a grid point sits ON a nucleus, where the
    reference divides by r = 0 without a guard (poc/main.py:111-120, 442-454): its E_integral is NaN, its E_net is fine
    (measured with the real code: n_test = 13, R = 3.0 -> (nan, -0.67800954); n_test = 13, R = 2.0 -> -0.76864690).
    The quadrature kernel does the same - NaN sums, never a silently skipped point - and E_net stays exact."""
    th = ck["ionHsym_fineTune"]
    Eint, Enet = pk.analysis.energy_from_psi(th, 3.0, {"n_test": 13})
    assert np.isnan(Eint) and abs(Enet - (-0.67800954)) < 1e-6
    s = pk.analysis.grid_sums(th, 3.0, {"n_test": 13})
    # (the kernel forms r = q * rsqrt(q), which is NaN at q = 0, so psi itself is NaN at that one point and every sum is;
    # the reference's psi is finite there and only its H psi is not - E_integral is NaN either way)
    assert np.isnan(s["psiHpsi"]) and np.isnan(s["dVdR_psi2"]) and np.isfinite(s["E_net"])
    Eint, Enet = pk.analysis.energy_from_psi(th, 2.0, {"n_test": 13}, rule="simpson")   # off the nuclei: the reference's number
    assert abs(Eint - (-0.7686469036652853)) < 2e-5 and abs(Enet - (-0.79302316)) < 1e-6


def test_grid_at_reference_resolution_and_10_8_points(ck):
    """n_test = 80 (set_params, poc/main.py:39): E_int close to the E-net and to the tabulated exact energy at R = 2;
    a 464^3 = 1.0e8-point grid (BASELINE config 5) runs in the same memory and agrees with the 80^3 one."""
    th = ck["ionHsym_fineTune"]
    Eint, Enet = pk.analysis.energy_from_psi(th, 2.0)
    assert abs(Enet - (-0.7961)) < 5e-3 and abs(Eint - Enet) < 3e-2      # exactE() poc/main.py:52-58: E(R=2.0) = -0.7961
    big = pk.analysis.grid_sums(th, 2.0, n=464)
    # the converged integral: the variational energy of the trained psi lies above the exact one, within ~1e-2 Ha
    assert -0.7961 < big["psiHpsi"] / big["psi2"] < -0.7961 + 2e-2 and abs(big["psiHpsi"] / big["psi2"] - Eint) < 2e-2
    assert abs(big["psi2"] - pk.analysis.grid_sums(th, 2.0, n=80)["psi2"]) < 2e-2 * big["psi2"]


def test_calculate_E_R_against_the_papers_table(ck, golden_dir):
    """poc/energy_R_ion.pkl (the authors' calculate_E_R output for 39 R values) vs the device sweep with the fine-tuned
    checkpoint.  E_net is reproduced exactly.  The grid the authors used for E_int / Elcao is not recorded with the
    table: set_params() says n_test = 80, the model-independent LCAO column is matched best by n_test = 90 (4e-4 at
    R = 0.2, 1e-5 beyond R = 2; CPU scan in DESIGN.md), so those two columns are a loose cross-check, not a parity gate -
    the parity gate for the quadrature is test_grid_energies_vs_oracle."""
    en = np.load(os.path.join(golden_dir, "energy_R_ion.npz"))
    d = pk.analysis.calculate_E_R(ck["ionHsym_fineTune"], {"n_test": 90})
    assert np.allclose(d["R"], en["R"])
    e_net, e_int, e_lcao = [np.abs(d[k] - en[k]).max() for k in ("E_net", "E_int", "Elcao")]
    print("calculate_E_R(n_test=90) vs energy_R_ion.pkl: max|dE_net| %.2e  max|dE_int| %.2e  max|dElcao| %.2e" % (e_net, e_int, e_lcao))
    assert e_net < 1e-6 and e_lcao < 1e-3 and e_int < 5e-3
    # the Hellmann-Feynman column has no counterpart in the table (its integrand ~1/r^2 makes an 80..90^3 grid noisy; the
    # reference plots it only qualitatively, main.py:1346-1370); its parity gate is test_grid_energies_vs_oracle
    assert np.all(np.isfinite(d["dEdR_HF"]))


def enet_curve_reference(th32, R):
    """E, dE/dR, d2E/dR2 and the gate in float64 with sigma' = e^-u / (1 + e^-u)^2 and sigma'' = e^-u (e^-u - 1) /
    (1 + e^-u)^3: accurate where a sigmoid saturates, where s (1 - s) keeps only e^|u| 2^-53 of relative accuracy."""
    P = layout.unpack_poc(th32.astype(np.float64))

    def sig(u):
        e = np.exp(-u)
        return 1.0 / (1.0 + e), e / (1.0 + e) ** 2, e * (e - 1.0) / (1.0 + e) ** 3

    w1 = P[6][:, 0]
    s, sp, spp = sig(R[:, None] * w1 + P[7])
    v, vp, vpp = s @ P[8].T + P[9], (sp * w1) @ P[8].T, (spp * w1 * w1) @ P[8].T
    t, tp, tpp = sig(v)
    wE = P[10][0]
    g = sig(R[:, None] * P[12][:, 0] + P[13])[0] @ P[14][0] + P[15][0]
    return dict(E=t @ wE + P[11][0], dE=(tp * vp) @ wE, d2E=(tpp * vp * vp + tp * vpp) @ wE, gate=g)


@pytest.mark.parametrize("regime", [r for r in sorted(REGIMES) if r.startswith(("enet", "gate"))] + ["mixed"])
def test_enet_curve_at_saturated_sigmoids(regime, init_theta):
    """The E-net and gate layers saturated, u in [8, 12] or [-12, -8] (oracle/regimes.py), at the bars of
    test_enet_curve_vs_autograd against the exp-form float64 reference."""
    Rs = np.linspace(0.2, 4.0, 39)
    th32 = regime_theta(init_theta, regime)
    c, ref = pk.analysis.enet_curve(th32, Rs), enet_curve_reference(th32, Rs)
    errs = {k: rel(c[k], ref[k]) for k in ("E", "dE", "d2E", "gate")}
    print("%s: %s" % (regime, " ".join("%s %.1e" % kv for kv in errs.items())))
    assert errs["E"] < 1e-12 and errs["dE"] < 1e-11 and errs["d2E"] < 1e-10 and errs["gate"] < 1e-12, errs


def test_enet_curve_vs_autograd(ck):
    Rs = np.linspace(0.2, 4.0, 39)
    th32 = ck["ionHsym_fineTune"].astype(np.float32)
    c, ref = pk.analysis.enet_curve(th32, Rs), enet_curve_reference(th32, Rs)
    assert rel(c["dE"], ref["dE"]) < 1e-11 and rel(c["d2E"], ref["d2E"]) < 1e-10
    R = torch.linspace(0.2, 4.0, 39, dtype=torch.float64, requires_grad=True)
    P = [torch.tensor(a.astype(np.float64)) for a in layout.unpack_poc(th32.astype(np.float64))]
    e = torch.sigmoid(R[:, None] * P[6][:, 0][None, :] + P[7][None, :])
    e = torch.sigmoid(e @ P[8].T + P[9][None, :])
    E = e @ P[10][0] + P[11][0]
    dE, = torch.autograd.grad(E.sum(), R, create_graph=True)       # poc/main.py:1324-1332
    d2E, = torch.autograd.grad(dE.sum(), R)
    g = torch.sigmoid(R[:, None] * P[12][:, 0][None, :] + P[13][None, :]) @ P[14][0] + P[15][0]
    c = pk.analysis.enet_curve(th32, R.detach().numpy())
    assert rel(c["E"], E.detach().numpy()) < 1e-12 and rel(c["dE"], dE.detach().numpy()) < 1e-11
    assert rel(c["d2E"], d2E.numpy()) < 1e-10 and rel(c["gate"], g.detach().numpy()) < 1e-12
    # golden E(R) table of the paper run (poc/energy_R_ion.pkl) is the E-net of the fine-tuned checkpoint
    Rg, tot = pk.analysis.energy_curve(ck["ionHsym_fineTune"], 0.2, 4.0, 39)
    assert np.allclose(tot - 1.0 / (2 * Rg), pk.analysis.enet_curve(ck["ionHsym_fineTune"], Rg)["E"])
