"""CPU-only tests: C-ABI exports, parameter packing, the train.py/NN_ion seams, data-parallel algebra."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from pinn_for_quantum_wavefunction_surfaces_b200 import params as P
from oracle import closed_form as cf
from oracle import layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# The two seam tests below patch and run the original project's own scripts (train.py; NN_ion and train() of
# poc/main.py of slitvinov/PINN_for_quantum_wavefunction_surfaces).  Those scripts are not part of this repository and
# no copy is stored in it, so the tests run only where PINN_REFERENCE points at a checkout of the original and skip
# elsewhere.  What they compare against is stored (tests/golden/trainpy_trace_n4096_e40.json); the oracle restatement
# of the same training loop is checked against it without the original by tests/test_oracle_train.py.
REF = os.environ.get("PINN_REFERENCE", "")
NO_REFERENCE = ("runs the original project's own scripts, which are not part of this repository: set PINN_REFERENCE "
                "to a checkout of slitvinov/PINN_for_quantum_wavefunction_surfaces")


def _in_reference(*parts):
    return bool(REF) and os.path.exists(os.path.join(REF, *parts))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    return g.build()


def test_library_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "pinn_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(pinn_[a-z_0-9]+)\s*\(", hdr)) - {"pinn_handle"})
    assert len(declared) >= 12
    L = ctypes.CDLL(built)
    for name in declared:
        assert hasattr(L, name), name
    assert L.pinn_version() >= 100 and L.pinn_theta_size() == 1521
    offs = (ctypes.c_int * 17)()
    L.pinn_theta_offsets(offs)
    assert list(offs) == layout.offsets() + [1521]
    assert sorted(declared) == sorted(set(pk._lib.EXPORTS)), "ctypes binding and header disagree"


def test_no_cpu_fallback(built):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pk.PinnError):
        pk.Handle(0)
    x = torch.zeros(8, 1, dtype=torch.float64)
    with pytest.raises(pk.PinnError):
        pk.fields("poc", x, x, x, x + 1, torch.zeros(1521))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "pinn_for_quantum_wavefunction_surfaces_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|import_module\(.oracle|oracle[/.](closed_form|ref_autograd|layout)",
                                     src, re.M), f


def test_param_packing_matches_oracle_layout():
    rng = np.random.default_rng(0)
    theta = rng.standard_normal(1521)
    tp = [torch.tensor(a) for a in layout.to_trainpy(theta)]
    assert np.array_equal(P.pack_trainpy(tp, dtype=torch.float64).numpy(), theta)
    back = P.unpack_trainpy(torch.tensor(theta))
    for a, b in zip(back, tp):
        assert a.shape == b.shape and torch.equal(a, b)
    poc = [torch.tensor(a) for a in layout.unpack_poc(theta)]
    assert np.array_equal(P.pack_poc(poc, dtype=torch.float64).numpy(), theta)
    ps = [torch.nn.Parameter(t) for t in poc]
    for i in (0, 1, 2, 3, 4, 5, 12, 13, 14, 15):  # freezeBase + freezeDecayUnit
        ps[i].requires_grad = False
    assert P.grad_mask_from_requires_grad(ps, "poc") == P.FINE_TUNE_GRAD_MASK


def test_indices_to_mask():
    m, c1, c2 = pk.indices_to_mask(6, (torch.tensor([0, 2]), torch.tensor([0, 0])), torch.tensor([2, 5, 3]), "cpu")
    assert m.tolist() == [1, 0, 3, 2, 0, 2] and (c1, c2) == (2, 3)


def _oracle_trainpy_op(x, y, z, R, i1, i2, *params):
    """Stand-in for PinnLossTrainPy.apply built on the CPU oracle (tests only): checks the PATCHING."""
    class F(torch.autograd.Function):
        @staticmethod
        def forward(ctx, *ps):
            theta = layout.from_trainpy([p.detach().numpy() for p in ps])
            n = x.shape[0]
            m1 = np.zeros(n); m1[i1.numpy()] = 1
            m2 = np.zeros(n); m2[i2.numpy()] = 1
            o = cf.loss_and_grad("trainpy", theta, x.detach().numpy(), y.detach().numpy(), z.detach().numpy(),
                                 R.numpy(), m1, m2)
            ctx.g = [torch.tensor(a) for a in layout.to_trainpy(o["grad"])]
            t = lambda v: torch.tensor(v, dtype=torch.float64)
            outs = (t(o["Ltot"]), t(o["Lpde"]), t(o["Lbc"]), t(o["E"]).reshape(-1, 1))
            ctx.mark_non_differentiable(*outs[1:])
            return outs

        @staticmethod
        def backward(ctx, g, *_):
            return tuple(g * a for a in ctx.g)
    return F.apply(*params)


@pytest.mark.skipif(not _in_reference("train.py"), reason=NO_REFERENCE)
def test_train_py_seam_reproduces_reference_trace(golden_dir, tmp_path):
    """The reference train.py with lines 41-57 replaced by one call reproduces the unmodified script's trace."""
    tr = json.load(open(os.path.join(golden_dir, "trainpy_trace_n4096_e40.json")))
    ns, out = pk.run_train_py(os.path.join(REF, "train.py"), n=4096, epochs=40, workdir=str(tmp_path),
                              loss_op=_oracle_trainpy_op)
    torch.set_default_dtype(torch.float32)
    lines = [ln.strip() for ln in out.strip().split("\n")]
    assert lines[:3] == tr["trace"][:3]          # identical prints for the first 20 steps
    assert len(lines) == len(tr["trace"])
    for a, b in zip(lines, tr["trace"]):          # later steps: same to print precision up to round-off drift
        fa = [float(v) for v in re.findall(r"[-+]?\d\.\d+e[-+]\d+", a)]
        fb = [float(v) for v in re.findall(r"[-+]?\d\.\d+e[-+]\d+", b)]
        assert np.allclose(fa, fb, rtol=2e-2), (a, b)
    assert os.path.getsize(tmp_path / "model.bin") == tr["model_bin_size"]


def test_trainpy_patch_rejects_unknown_source():
    with pytest.raises(ValueError):
        pk.trainpy_patched_source("print('hello')\n")


def test_patch_nn_ion_signature():
    calls = []

    class Fake:
        def LossFunctions(self, x, y, z, R, params, b1, b2):
            return "orig"

    orig = pk.patch_nn_ion(Fake, loss_fn=lambda m, x, y, z, R, b1, b2: calls.append((x, b2)) or "fused")
    assert Fake().LossFunctions(1, 2, 3, 4, {"BCcutoff": 17.5}, 5, 6) == "fused" and calls == [(1, 6)]
    assert orig(Fake(), 1, 2, 3, 4, None, 5, 6) == "orig"


def _oracle_poc_loss(model, x, y, z, R, bIndex1, bIndex2):
    """Stand-in for ops.loss_poc built on the CPU oracle (tests only): same contract - the model's 16 parameters in
    parameters() order, torch.where tuples as index sets, gradients only for the tensors with requires_grad."""
    ps = list(model.parameters())

    class F(torch.autograd.Function):
        @staticmethod
        def forward(ctx, *tensors):
            theta = layout.pack_poc([t.detach().numpy() for t in tensors])
            n = x.shape[0]
            m1 = np.zeros(n); m1[bIndex1[0].numpy()] = 1
            m2 = np.zeros(n); m2[bIndex2[0].numpy()] = 1
            o = cf.loss_and_grad("poc", theta, *[v.detach().numpy().ravel() for v in (x, y, z, R)], m1, m2)
            ctx.g = [torch.tensor(a) for a in layout.unpack_poc(o["grad"])]
            ctx.needs = [t.requires_grad for t in tensors]
            t = lambda v: torch.tensor(v, dtype=torch.float64)
            outs = (t(o["Ltot"]), t(o["Lpde"]), t(o["Lbc"]), t(o["E"]).reshape(-1, 1))
            ctx.mark_non_differentiable(*outs[1:])
            return outs

        @staticmethod
        def backward(ctx, g, *_):
            return tuple((g * a.reshape(a.shape)) if need else None for a, need in zip(ctx.g, ctx.needs))
    return F.apply(*ps)


@pytest.mark.skipif(not _in_reference("poc", "main.py"), reason=NO_REFERENCE)
def test_patch_the_real_nn_ion_and_run_the_reference_train(tmp_path, golden_dir):
    """The drop-in seam on the REAL class: NN_ion is loaded from the reference file (AST, as tests/golden/make_golden.py
    does), patched with patch_nn_ion, and the reference's own train() (poc/main.py:359-430: sampler, Adam, freeze flags,
    history arrays, .pt writer) runs on top of it - once unpatched, once patched with the oracle loss, same seed.  Also pins
    the assumption the packing relies on: parameters() order == state_dict() order == pk.POC_TENSOR_NAMES."""
    import pickle
    import time
    from os import path
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden as mg
    torch.set_default_dtype(torch.double)
    try:
        cwd = os.getcwd()
        os.chdir(tmp_path)
        os.makedirs("models"); os.makedirs("data")
        hist = {}
        for patched in (False, True):
            ns = mg.load_poc_namespace()
            ns.update(path=path, time=time, pickle=pickle)
            NN_ion = ns["NN_ion"]
            m = NN_ion(ns["params"])
            assert [k for k, _ in m.named_parameters()] == list(m.state_dict().keys()) == pk.POC_TENSOR_NAMES
            if patched:
                orig = pk.patch_nn_ion(NN_ion, loss_fn=_oracle_poc_loss)
                assert orig is not None
            for stage, (epochs, lr, freeze) in enumerate(((6, 8e-3, False), (4, 5e-4, True))):
                prm = ns["set_params"]()
                prm.update(epochs=epochs, n_train=1500, lr=lr, lossPath="data/loss_%d.pkl" % stage,
                           saveModelPath="models/m.pt", loadModelPath="models/m.pt")
                torch.manual_seed(3 + stage)
                ns["train"](prm, loadWeights=freeze, freezeUnits=freeze)
                with open("data/loss_%d.pkl" % stage, "rb") as f:
                    hist[(patched, stage)] = pickle.load(f)
            sd = torch.load("models/m.pt", weights_only=True)["model_state_dict"]
            hist[(patched, "theta")] = layout.pack_poc([v.numpy() for v in sd.values()])
        for stage in (0, 1):
            for k in ("Ltot", "Lpde", "Lbc", "Energy"):
                a, b = hist[(False, stage)][k], hist[(True, stage)][k]
                assert a.shape == b.shape and np.allclose(a, b, rtol=1e-9, atol=1e-14), (stage, k)
        assert np.abs(hist[(False, "theta")] - hist[(True, "theta")]).max() < 1e-10
        # the fine-tune stage moved the E-net tensors only (freezeBase + freezeDecayUnit, poc/main.py:305-319)
        # a model the kernels do not implement is refused instead of silently trained on the wrong loss
        bad = dict(ns["set_params"](), inversion_symmetry=-1)
        mb = NN_ion(bad)
        x, y, z, R = ns["sampling"](bad, 64)
        with pytest.raises(pk.PinnError):
            mb.LossFunctions(x, y, z, R, bad, (torch.tensor([0]), torch.tensor([0])), (torch.tensor([1]), torch.tensor([0])))
    finally:
        os.chdir(cwd)
        torch.set_default_dtype(torch.float32)


def test_unsupported_model_configurations_are_refused():
    P.check_supported_model({"inversion_symmetry": 1, "Ry": 0, "Rz": 0})
    P.check_supported_model(None, None)
    for bad in ({"inversion_symmetry": -1}, {"Ry": 0.5}, {"Rz": -1}):
        with pytest.raises(pk.PinnError):
            P.check_supported_model(bad)
    with pytest.raises(pk.PinnError):
        pk.train_poc(np.zeros(1521), {"inversion_symmetry": -1})


DP_WORKER = r'''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from pinn_for_quantum_wavefunction_surfaces_b200 import dp
from oracle import closed_form as cf
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
gd = os.path.join(sys.argv[1], "tests", "golden")
theta = np.load(os.path.join(gd, "checkpoints.npz"))["ionHsym"]
g = np.load(os.path.join(gd, "poc_seed0_n4096.npz"))
n = g["x"].size
m1 = np.zeros(n); m1[g["i1"]] = 1
m2 = np.zeros(n); m2[g["i2"]] = 1
sl = np.array_split(np.arange(n), world)[rank]
w = dp.global_weights(len(sl), m1[sl].sum(), m2[sl].sum())
def local(weights, out):
    o = cf.loss_and_grad("poc", theta, g["x"][sl], g["y"][sl], g["z"][sl], g["R"][sl], m1[sl], m2[sl], *weights.tolist())
    out[0], out[1], out[2] = o["Ltot"], o["Lpde"], o["Lbc"]
    out[3], out[4], out[5], out[6], out[7] = o["sums"]["E"], o["sums"]["res2"], o["sums"]["psi2_1"], o["sums"]["psi2_2"], 0.0
    out[8:] = torch.from_numpy(o["grad"])
sums, dth = dp.dp_loss_and_grad(local, w)
if rank == 0:
    ref_l, ref_g = g["ionHsym_loss"], g["ionHsym_grad"]
    assert abs(w[0].item() - 1.0 / n) < 1e-18 and abs(w[1].item() - 1.0 / 2151) < 1e-18
    assert abs(sums[0].item() - ref_l[0]) / ref_l[0] < 1e-11, (sums[0].item(), ref_l[0])
    assert abs(sums[2].item() - ref_l[2]) / ref_l[2] < 1e-11
    assert np.abs(dth.numpy() - ref_g).max() / np.abs(ref_g).max() < 1e-10
    print("DP_OK")
dist.destroy_process_group()
'''


def test_data_parallel_two_ranks_gloo(tmp_path):
    """world_size-2 gloo run of the DP step (oracle as the local compute): sharded result == golden full result."""
    script = tmp_path / "dp_worker.py"
    script.write_text(DP_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29541")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29541", str(script), ROOT]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and "DP_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """bench.py --impl reference runs on the host cores alone (oracle port of the reference's nested-autograd step) and
    prints one JSON line with the keys the driver reads; --dump-outputs writes what its last timed step returned."""
    import json
    import subprocess
    # the way the driver launches it for N > 1: torch.distributed.run exports OMP_NUM_THREADS=1 to its workers - the arm
    # must still use every host core it may (round 1 ran single-threaded there and inflated the N >= 2 ratios 8.5x)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1",
                        "--points", "8192", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600,
                       env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len(r.stdout.strip().splitlines()) == 1, r.stdout  # ONE line on stdout
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "points/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["vs_baseline"] is None and line["config"]["workload"].startswith("ionHsym")
    assert line["steps"] == 3                                      # --steps is honoured
    assert line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) == line["config"]["host_threads"]
    assert line["config"]["points_per_gpu"] == 8192 and "full batch" in line["cpu_baseline"]["sample"]
    loss, dth, E = (np.load(tmp_path / (k + ".npy")) for k in ("loss", "dtheta", "E"))
    assert loss.dtype == dth.dtype == E.dtype == np.float64
    assert loss.shape == (3,) and dth.shape == (1521,) and E.shape == (8192, 1)
    assert np.all(np.isfinite(dth)) and np.all(np.isfinite(E)) and loss[0] == loss[1] + loss[2]
    # ranks other than 0 exit 0 without work or output
    r1 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--gpus", "2"],
                        capture_output=True, text=True, timeout=120, env=dict(env, RANK="1", WORLD_SIZE="2"))
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_stash_swizzle_is_conflict_free_for_all_three_access_patterns():
    """The stash swizzle of the tcgen05 engine (csrc/pinn_device.cuh: swz_tc) restated: a row is one point, 64 floats
    (every row starts on bank 0); the 16-byte chunk index of row r is XOR-ed with ((r&3)<<1)|((r>>2)&1).  Checked here
    against the bank model (32 banks x 4 bytes; a 128-bit access is served a quarter-warp at a time, a 64-bit access a
    half-warp at a time): all three access patterns of the kernel touch every bank at most once per phase."""
    src = open(os.path.join(ROOT, "pinn_for_quantum_wavefunction_surfaces_b200", "csrc", "pinn_device.cuh")).read()
    assert "((((row & 3) << 1) | ((row >> 2) & 1)) << 2)" in src      # the formula this test restates
    swz = lambda r: ((((r & 3) << 1) | ((r >> 2) & 1)) << 2)          # in floats
    ROW = 64
    bank = lambda row, col: (row * ROW + (col ^ swz(row))) % 32
    # (a) every lane reads/writes a float4 of ITS OWN row at the same logical column: 8 lanes per phase
    for c4 in range(0, ROW, 4):
        for q in range(4):
            banks = [bank(l, c4 + k) for l in range(8 * q, 8 * q + 8) for k in range(4)]
            assert len(set(banks)) == 32, ("row access", c4, q)
    # (b) mma.sync fragment loads: lane (g, t) reads row p0 + t (or + 4), column c0 + g (or + 8), 32 lanes per phase
    for p0 in range(0, 32, 8):
        for dp in (0, 4):
            for c0 in range(0, ROW, 16):
                for dc in (0, 8):
                    banks = [bank(p0 + dp + t, c0 + dc + g) for g in range(8) for t in range(4)]
                    assert len(set(banks)) == 32, ("fragment", p0, dp, c0, dc)
    # (c) packed column sums: 16 lanes of a half-warp read float2 (columns 2 cp, 2 cp + 1) of ONE row per phase
    for row in range(32):
        for win in (0, 16, 48):   # the three 32-column windows used (wrapping at 64)
            banks = [bank(row, ((win + 2 * cp) & 63) + k) for cp in range(16) for k in range(2)]
            assert len(set(banks)) == 32, ("column sum", row, win)
    # ... and the swizzle it replaced was 2-way conflicted on (a): documented in DESIGN.md
    old = lambda r: (r & 3) << 3
    banks = [(l * ROW + (0 ^ old(l)) + k) % 32 for l in range(8) for k in range(4)]
    assert len(set(banks)) == 16


def test_bench_keeps_library_banners_off_stdout():
    """Whatever a library writes to file descriptor 1 during the run (NCCL's version banner, for one) lands on stderr; the
    result line alone reaches the caller's stdout."""
    import json
    import subprocess
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench.claim_stdout(); os.write(1, b'NCCL version x\\n'); "
            "print('python-level chatter'); bench.emit({'metric': 'm', 'value': 1.0})" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout) == {"metric": "m", "value": 1.0}
    assert "NCCL version x" in r.stderr and "python-level chatter" in r.stderr


def test_tf32_split_model_rounding_and_bias():
    """Bit-level numpy model of the three x = hi + lo splits in csrc/pinn_device.cuh (the tensor core reads the upper 19
    bits of each operand): every split is exact in fp32; what the hardware sees of (hi, lo) is within 2^-21.4 |x|
    (truncating split, always toward zero: a bias) or 2^-23 |x| (rounded hi, with or without the half-ulp pre-rounding of
    lo: the three-instruction form loses nothing against the four-instruction one, and neither is biased)."""
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(1 << 18) * np.exp(rng.uniform(-8, 3, 1 << 18))).astype(np.float32)
    bits = lambda a: a.view(np.uint32)
    seen_by_mma = lambda a: (bits(a) & np.uint32(0xFFFFE000)).view(np.float32)

    def split(x, round_hi, round_lo):
        hi = ((bits(x) + np.uint32(0x1000 if round_hi else 0)) & np.uint32(0xFFFFE000)).view(np.float32)
        lo = (x - hi).astype(np.float32)
        assert np.all(hi.astype(np.float64) + lo.astype(np.float64) == x.astype(np.float64))  # exact
        if round_lo:
            lo = (bits(lo) + np.uint32(0x1000)).view(np.float32)
        seen = seen_by_mma(hi).astype(np.float64) + seen_by_mma(lo).astype(np.float64)
        return (seen - x.astype(np.float64)) / x.astype(np.float64)   # signed relative error

    e_trunc, e_rn3, e_rn4 = split(x, False, False), split(x, True, False), split(x, True, True)
    assert np.abs(e_trunc).max() < 2.0 ** -21 and e_trunc.max() <= 0.0 and e_trunc.mean() < -5e-8   # one-sided
    for e in (e_rn3, e_rn4):
        assert np.abs(e).max() <= 2.0 ** -23 and abs(e.mean()) < 2e-9                                # unbiased
    assert np.abs(e_rn3).max() == np.abs(e_rn4).max()


def test_bench_roofline_denominators():
    """The two contract ceilings bench.py reports beside the FP32 one: measured HBM copy rate and measured tensor rate in
    3xTF32 (MEASURED_PEAKS.json when present, the profiling recipe's fallbacks otherwise)."""
    sys.path.insert(0, ROOT)
    import bench
    n, ms = 1 << 18, 0.1167
    hb = bench.hbm_ceiling(16 * n, ms)
    tc = bench.tensor_ceiling(27044.0 * n, ms)
    assert hb["unit"] == "GB/s" and abs(hb["achieved"] - 16 * n / (ms * 1e-3) / 1e9) < 1e-9
    assert 5000.0 < hb["peak"] < 8000.0 and abs(hb["frac"] - hb["achieved"] / hb["peak"]) < 1e-12
    assert tc["unit"] == "TFLOP/s" and abs(tc["achieved"] - 27044.0 * n / (ms * 1e-3) / 1e12) < 1e-9
    assert 200.0 < tc["peak"] < 400.0 and abs(tc["frac"] - tc["achieved"] / tc["peak"]) < 1e-12
    assert "measured" in hb["peak_source"] or "fallback" in hb["peak_source"]


def test_bench_withholds_ncu_figures_of_another_build(tmp_path, monkeypatch):
    """roofline.traffic / pipe utilisation are copied from the committed ncu capture only while the kernel sources are the
    ones it was captured from (profiles/traffic.json: kernel_source_sha256)."""
    sys.path.insert(0, ROOT)
    import bench
    now = bench.kernel_source_sha256()
    assert len(now) == 64
    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "kernel_source_sha256", lambda: now)
    assert bench.committed_ncu_figures()[:2] == (None, None)
    body = {"dram_bytes_per_launch": 4300000, "ncu_pipe_utilisation_pct": {"fma": 20.0}, "source": "x", "kernel_source_sha256": now}
    (prof / "traffic.json").write_text(json.dumps(body))
    t, pipes, src = bench.committed_ncu_figures()
    assert t == 4300000 and pipes == {"fma": 20.0} and now[:12] in src
    body["kernel_source_sha256"] = "0" * 64
    (prof / "traffic.json").write_text(json.dumps(body))
    t, pipes, src = bench.committed_ncu_figures()
    assert t is None and pipes is None and src.startswith("stale")
