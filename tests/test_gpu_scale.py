"""The fused training step at 6.6e4 to 2.7e8 points per launch against an exact float64 reference, through every training
entry point.

The step kernel keeps its gradient and loss accumulators in float32 registers for the whole launch: a CTA adds one
128-point super-tile after another into them, and they reach double only when the CTA folds them into its partial row.
So a CTA's float32 run grows with the batch, ceil(n / 128) / 148 super-tiles: 14 at the benchmark's 2^18 points, 222 at
BASELINE config 4's 2^22, 14 200 at 2^28.  The other parity tests compare at most 20 000 points with the oracle.
(Training launches past 256 super-tiles per CTA run more CTAs than SMs, 256 or fewer each: train_grid_for, pinn_handle.h.)

No CPU oracle has to run over such a batch.  The batch is K copies of one block B of 2^16 + 37 points followed by the
first r = 101 points of B; the loss weights are the global {1/n, 1/|set 1|, 1/|set 2|}.  The raw sums and the gradient of
each loss term are sums over points, so the float64 reference is K S(B) + S(B[:r]), from six oracle calls on B and B[:r]
with unit weight on one term at a time (a CPU test checks this construction on a materialised batch).  |B| = 37 mod 128,
so the copies of B start at every offset within a super-tile, and the last super-tile is ragged.

A lost or doubled super-tile moves a sum by only ~1 / (number of super-tiles) - 5e-7 relative at 2^28 points, under the
bars - so every case also checks E per point: E_out is filled with NaN before the call and must equal, bit for bit, the E
of a launch over B alone, tiled the same way.  That compares the kernel with itself at small n (only the E of the last
point goes to the oracle here): the accuracy of E per point rests on the small-n parity tests.  With -s every case
prints n, super-tiles per CTA, the worst gradient errors and the loss-term errors against the oracle, and the difference
from launches over B and B[:r] alone combined in float64: that isolates the accumulation over many super-tiles from the
per-point float32 error.
"""
import ctypes
import functools
import gc
import os

import numpy as np
import pytest
import torch

import pinn_for_quantum_wavefunction_surfaces_b200 as pk
from oracle import closed_form as cf
from oracle import layout
from oracle import ref_autograd as ra

OFFS = layout.offsets() + [1521]
FORMS = {0: "poc", 1: "trainpy"}
NB = (1 << 16) + 37                # the block B
R_TAIL = 101                       # the batch ends with B[:R_TAIL]
SEED = 29
KS = [1, 64, 256, 1024, 4096]      # 6.6e4 ... 2.7e8 points: 3.5 ... 14 200 super-tiles per CTA
BIG_K = 4096                       # 4.3 GB of coordinates, 0.27 GB of mask, 1.07 GB of E
BIG_FREE = 8 << 30                 # ... skipped, alone, when the device has less than this free
TRAINED_GRAD_BAR = 1.2e-4          # the bars of test_gpu_parity.py::test_trained_weights_vs_oracle
TRAINED_LBC_BAR = 1.5e-4
TRAINED_ENET_BAR = 2e-5
# Lin_H2.weight and Lin_E2.weight are summed by mma.sync (3xTF32) into float32 register fragments that carry every
# super-tile of a CTA, and the tensor core adds into its accumulator with truncation: their error grows with the
# super-tiles per CTA (DESIGN.md section 4).  They are held to the same bars as everything else, in a test of their own;
# the cases that miss them are strict expected failures until the accumulation is fixed in the kernel.
MMA_TENSORS = ("Lin_H2.weight", "Lin_E2.weight")
MMA_REASON = ("mma.sync sums Lin_H2.weight and Lin_E2.weight in float32 over every super-tile of a CTA and truncates "
              "into its accumulator: 1.6e-4 at 2^22 points (DESIGN.md section 4)")


@pytest.fixture(scope="module")
def init_theta(golden_dir):
    return np.load(os.path.join(golden_dir, "trainpy_n2048.npz"))["theta"]   # train.py's init rule, seed 12345


@pytest.fixture(scope="module")
def ck(golden_dir):
    return np.load(os.path.join(golden_dir, "checkpoints.npz"))


# ---------------------------------------------------------------------------------------------
# the exact reference by tiling
# ---------------------------------------------------------------------------------------------
def sample_block(variant, nb=NB, seed=SEED):
    g = torch.Generator().manual_seed(seed + variant)
    x, y, z, R, i1, i2 = ra.sample_box(nb, FORMS[variant], g)
    a32 = [v.numpy().ravel().astype(np.float32) for v in (x, y, z, R)]
    m1, m2 = np.zeros(nb), np.zeros(nb)
    m1[i1.numpy()] = 1
    m2[i2.numpy()] = 1
    return a32, m1, m2


def tiled_size_and_weights(m1, m2, K, r=R_TAIL):
    """n and the global loss weights {1/n, 1/C1, 1/C2} of K copies of the block followed by its first r points."""
    n = K * m1.size + r
    return n, np.array([1.0 / n, 1.0 / (K * m1.sum() + m1[:r].sum()), 1.0 / (K * m2.sum() + m2[:r].sum())])


def block_terms(variant, th32, a32, m1, m2):
    """The oracle on one block with unit weight on one loss term at a time: the gradient of each term, the raw sums
    {sum E, sum res^2, sum psi^2 over set 1, over set 2} (sums[3:7] of the kernel) and E per point."""
    a64 = [a.astype(np.float64) for a in a32]
    out = {}
    for k, w in enumerate(((1.0, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0))):
        ref = cf.loss_and_grad(FORMS[variant], th32.astype(np.float64), *a64, m1, m2, w_pde=w[0], w_bc1=w[1], w_bc2=w[2])
        out[k] = ref["grad"]
    s = ref["sums"]
    out["sums"] = np.array([s["E"], s["res2"], s["psi2_1"], s["psi2_2"]])
    out["E"] = ref["E"]
    return out


def tiled_reference(blk, tail, K, w):
    """Loss terms, raw sums, E of the last point and dLtot/dtheta of K copies of a block followed by `tail`, by linearity."""
    S = K * blk["sums"] + tail["sums"]
    G = [K * blk[k] + tail[k] for k in range(3)]
    Lpde, Lbc = w[0] * S[1], w[1] * S[2] + w[2] * S[3]
    return dict(Ltot=Lpde + Lbc, Lpde=Lpde, Lbc=Lbc, sums=S, E_last=tail["E"][-1],
                grad=w[0] * G[0] + w[1] * G[1] + w[2] * G[2])


def tile_np(a, K, r=R_TAIL):
    return np.concatenate([np.tile(a, K), a[:r]])


@pytest.mark.parametrize("variant", [0, 1])
def test_tiled_reference_is_exact(variant, init_theta):
    """The oracle on a materialised batch of K = 8 copies of a 4096 + 37-point block and 101 more points equals the
    combination of the six oracle calls on the block and on its head."""
    nb, K = 4096 + 37, 8
    a32, m1, m2 = sample_block(variant, nb, SEED + 100)
    th32 = init_theta.astype(np.float32)
    n, w = tiled_size_and_weights(m1, m2, K)
    head = [a[:R_TAIL] for a in a32]
    ref = tiled_reference(block_terms(variant, th32, a32, m1, m2),
                          block_terms(variant, th32, head, m1[:R_TAIL], m2[:R_TAIL]), K, w)
    big = [tile_np(a.astype(np.float64), K) for a in a32]
    assert big[0].size == n
    full = cf.loss_and_grad(FORMS[variant], th32.astype(np.float64), *big, tile_np(m1, K), tile_np(m2, K),
                            w_pde=w[0], w_bc1=w[1], w_bc2=w[2])
    for k in ("Ltot", "Lpde", "Lbc"):
        assert abs(ref[k] - full[k]) <= 1e-12 * abs(full[k]), k
    s = full["sums"]
    for i, v in enumerate((s["E"], s["res2"], s["psi2_1"], s["psi2_2"])):
        assert abs(ref["sums"][i] - v) <= 1e-12 * abs(v), i
    assert abs(ref["E_last"] - full["E"][-1]) <= 1e-12 * abs(full["E"][-1])
    assert rel(ref["grad"], full["grad"]) < 1e-12


# ---------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------
def dev():
    return torch.device("cuda:0")


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def entry_rel(a, b):
    """Largest relative error over the entries with |b| >= 1e-2 max|b| (Adam takes a full-size step on every entry)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    big = np.abs(b) >= 1e-2 * np.abs(b).max()
    return float((np.abs(a - b)[big] / np.abs(b)[big]).max()) if big.any() else 0.0


def tile_t(a, K, r=R_TAIL):
    """K copies of the 1-D tensor a followed by a[:r], on a's device."""
    nb = a.numel()
    out = torch.empty(K * nb + r, dtype=a.dtype, device=a.device)
    out[:K * nb].view(K, nb).copy_(a.expand(K, nb))
    out[K * nb:].copy_(a[:r])
    return out


def need_memory(K):
    if K == BIG_K:
        free, _ = torch.cuda.mem_get_info(dev())
        if free < BIG_FREE:
            pytest.skip("K = %d needs about 6 GB of device memory; %.1f GB free" % (K, free / 2 ** 30))


@pytest.fixture(autouse=True)
def _release_device_memory():
    yield
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def reference():
    """reference(variant, th32, K) -> the tiled float64 reference; the oracle runs once per (variant, theta)."""
    @functools.lru_cache(maxsize=None)
    def blocks(variant, th_bytes):
        th32 = np.frombuffer(th_bytes, np.float32)
        a32, m1, m2 = sample_block(variant)
        return (block_terms(variant, th32, a32, m1, m2),
                block_terms(variant, th32, [a[:R_TAIL] for a in a32], m1[:R_TAIL], m2[:R_TAIL]))

    def get(variant, th32, K):
        _, m1, m2 = sample_block(variant)
        _, w = tiled_size_and_weights(m1, m2, K)
        return tiled_reference(*blocks(variant, th32.tobytes()), K, w)
    return get


def run_case(variant, th32, K, call, dtype=np.float32, grad_mask=0xFFFF, where="cuda", E_dtype=torch.float32):
    """Build the tiled batch (on the device, or in host memory for where="cpu"), fill E_out with NaN, run
    call(cols, mask, w_host, E_out) -> (sums, dtheta) as numpy, and check E per point against a launch over B alone.
    Also launches B and B[:r] alone (pinn_loss_fwd_bwd, same weights) and returns K S(B) + S(B[:r]) of those.  The
    batch is freed before this returns, so that a failing assertion of the caller does not hold on to it."""
    a32, m1, m2 = sample_block(variant)
    n, w = tiled_size_and_weights(m1, m2, K)
    wd = t(w)
    cols = [t(a.astype(dtype)) for a in a32]
    mask = t((m1 + 2 * m2).astype(np.uint8))
    th = t(th32)
    blk = []
    for m in (NB, R_TAIL):
        s, g, e = pk.loss_and_grad_raw(variant, *[c[:m] for c in cols], th, mask[:m], wd, grad_mask, want_E=True)
        blk.append((s.cpu().numpy(), g.cpu().numpy(), e))
    E_blk = blk[0][2].to(E_dtype)
    on = torch.device(where) if where == "cpu" else dev()
    big = [tile_t(c.to(on), K) for c in cols]
    big_mask = tile_t(mask.to(on), K)
    assert big[0].numel() == n
    E = torch.full((n,), float("nan"), dtype=E_dtype, device=on)
    del cols, mask
    sums, dth = call(big, big_mask, w, E)
    torch.cuda.synchronize()
    E_ref = E_blk.to(on)
    per_point = (torch.equal(E[:K * NB].view(K, NB), E_ref.expand(K, NB)) and torch.equal(E[K * NB:], E_ref[:R_TAIL]))
    last = float(E[n - 1].item())
    del big, big_mask, E, E_ref, E_blk
    return dict(n=n, sums=sums, dth=dth, per_point=per_point, E_last=last,
                pred_sums=K * blk[0][0][:7] + blk[1][0][:7], pred_dth=K * blk[0][1] + blk[1][1])


def packed_call(variant, th32, grad_mask=0xFFFF):
    def call(cols, mask, w, E):
        s, g, _ = pk.loss_and_grad_raw(variant, *cols, t(th32), mask, t(w), grad_mask, E_out=E)
        return s.cpu().numpy(), g.cpu().numpy()
    return call


def errors(res, ref, tensors=range(16)):
    s, S = res["sums"], ref["sums"]
    loss = {"Ltot": s[0] / ref["Ltot"] - 1, "Lpde": s[1] / ref["Lpde"] - 1, "Lbc": s[2] / ref["Lbc"] - 1,
            "sumE": s[3] / S[0] - 1, "res2": s[4] / S[1] - 1, "psi2_1": s[5] / S[2] - 1, "psi2_2": s[6] / S[3] - 1}
    loss = {k: abs(v) for k, v in loss.items()}
    grad = {layout.POC_TENSORS[i][0]: (rel(res["dth"][OFFS[i]:OFFS[i + 1]], ref["grad"][OFFS[i]:OFFS[i + 1]]),
                                       entry_rel(res["dth"][OFFS[i]:OFFS[i + 1]], ref["grad"][OFFS[i]:OFFS[i + 1]]))
            for i in tensors}
    return loss, grad


def tiles_per_cta(n):
    """Super-tiles per CTA of a training launch over n points, and its CTAs (train_grid_for, pinn_handle.h)."""
    sm = torch.cuda.get_device_properties(dev()).multi_processor_count
    tiles = -(-n // 128)
    grid = sm * -(-(-(-tiles // sm)) // 256) if tiles > sm * 256 else min(tiles, sm)
    return tiles / grid, grid


def report(tag, res, loss, grad, tensors=range(16)):
    wt = max(grad, key=lambda k: grad[k][0])
    we = max(grad, key=lambda k: grad[k][1])
    acc = {layout.POC_TENSORS[i][0]: rel(res["dth"][OFFS[i]:OFFS[i + 1]], res["pred_dth"][OFFS[i]:OFFS[i + 1]]) for i in tensors}
    wa = max(acc, key=acc.get)
    acc_s = max(abs(a / b - 1) for a, b in zip(res["sums"][:7], res["pred_sums"]) if b != 0)
    T, grid = tiles_per_cta(res["n"])
    print("\n%-22s n %9d  %5.1f tiles/CTA, %5d CTAs | grad tensor %.1e (%s) entry %.1e (%s) | %s | vs blocks: grad %.1e (%s) sums %.1e"
          % (tag, res["n"], T, grid, grad[wt][0], wt, grad[we][1], we,
             " ".join("%s %.1e" % kv for kv in loss.items()), acc[wa], wa, acc_s))
    for k, (et, ee) in grad.items():
        if et >= 1e-5 or ee >= 1e-4:
            print("    %-18s tensor %.2e  entry %.2e  vs blocks %.2e" % (k, et, ee, acc[k]))


def check(res, ref, loss, grad, trained=False):
    """The per-point checks, and the bars of the small-n parity tests for everything but the two mma.sync-summed tensors
    (test_mma_sync_gradients_at_scale holds those to the same bars)."""
    assert res["per_point"], "E_out differs from the tiled E of the block launch (a super-tile skipped or misplaced)"
    assert res["sums"][7] == res["E_last"], (res["sums"][7], res["E_last"])
    assert abs(res["E_last"] - ref["E_last"]) <= 1e-5 * abs(ref["E_last"])
    if not trained:
        bad = {k: v for k, v in loss.items() if not v < 1e-5}
        bad.update({k: v for k, v in grad.items() if k not in MMA_TENSORS and not (v[0] < 1e-5 and v[1] < 1e-4)})
    else:   # the gradient is a cancelling sum there, and psi at the boundary a 2e-5 cancellation of O(0.1) terms
        lbc = ("Lbc", "psi2_1", "psi2_2")
        bad = {k: v for k, v in loss.items() if not v < (TRAINED_LBC_BAR if k in lbc else 1e-5)}
        keep = np.ones(1521, bool)
        for i, (nm, _) in enumerate(layout.POC_TENSORS):
            keep[OFFS[i]:OFFS[i + 1]] = nm not in MMA_TENSORS
        g = rel(res["dth"][keep], ref["grad"][keep]) * np.abs(ref["grad"][keep]).max() / np.abs(ref["grad"]).max()
        if not g < TRAINED_GRAD_BAR:
            bad["grad"] = g
        bad.update({k: v for i, (k, v) in enumerate(grad.items())
                    if i >= 6 and k not in MMA_TENSORS and not v[0] < TRAINED_ENET_BAR})
    assert not bad, bad


def check_mma_sync_tensors(res, ref, grad, trained):
    if not trained:
        bad = {k: grad[k] for k in MMA_TENSORS if k in grad and not (grad[k][0] < 1e-5 and grad[k][1] < 1e-4)}
    else:
        bad = {k: grad[k][0] for k in MMA_TENSORS if k == "Lin_E2.weight" and not grad[k][0] < TRAINED_ENET_BAR}
        if not rel(res["dth"], ref["grad"]) < TRAINED_GRAD_BAR:
            bad["grad"] = rel(res["dth"], ref["grad"])
    assert not bad, bad


# ---------------------------------------------------------------------------------------------
# the cases: (form, weights, entry point, K); each runs once per module and serves both of its tests
# ---------------------------------------------------------------------------------------------
CASES = {"%s-init-K%d" % (FORMS[v], K): (v, "init", "packed", K) for v in (0, 1) for K in KS}
CASES.update({"poc-trained-K%d" % K: (0, "trained", "packed", K) for K in KS})
CASES.update({"%s-f64-K256" % FORMS[v]: (v, "init", "f64", 256) for v in (0, 1)})
CASES["poc-finetune-K1024"] = (0, "init", "finetune", 1024)
CASES.update({"%s-tensors-K256" % FORMS[v]: (v, "init", "tensors", 256) for v in (0, 1)})
CASES.update({"poc-host-%s-K256" % m: (0, "init", "host-" + m, 256) for m in ("pinned", "pageable")})
# every case past 3.5 super-tiles per CTA at init weights (1.6e-4 at 222, 1.8e-4 at 253 for Lin_E2.weight), and at the
# trained weights the one where Lin_E2.weight reaches 2.0e-5 against its 2e-5 bar
MMA_MISSES = {c for c, (v, weights, kind, K) in CASES.items() if K > 1 and weights == "init"} | {"poc-trained-K4096"}
_RESULTS = {}


def tensor_call(variant, th32):
    th = th32.astype(np.float64)

    def call(cols, mask, w, E):
        parts = layout.unpack_poc(th) if variant == 0 else layout.to_trainpy(th)
        params = [torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device=dev()) for a in parts]
        h = pk.Handle.get(0)
        out = torch.empty(8 + 1521, dtype=torch.float64, device=dev())
        ptrs = (ctypes.c_void_p * 16)(*[p.data_ptr() for p in params])
        rc = h.L.pinn_loss_fwd_bwd_tensors(h.h, variant, cols[0].numel(), *[c.data_ptr() for c in cols], 0, mask.data_ptr(),
                                           ptrs, 1, variant, (ctypes.c_double * 3)(*w), 0xFFFF, 17.5, out.data_ptr(),
                                           out.data_ptr() + 64, E.data_ptr(), 1, torch.cuda.current_stream().cuda_stream)
        h.check(rc, "pinn_loss_fwd_bwd_tensors")
        o = out.cpu().numpy()
        g = o[8:]
        if variant == 1:   # canonical tensor order, each tensor in train.py's (in,out) layout -> back to (out,in)
            g = np.concatenate([g[OFFS[i]:OFFS[i + 1]].reshape(shp[::-1]).T.ravel() if len(shp) == 2 else g[OFFS[i]:OFFS[i + 1]]
                                for i, (_, shp) in enumerate(layout.POC_TENSORS)])
        return o[:8], g
    return call


def host_call(mode, th32):
    th64 = np.ascontiguousarray(th32.astype(np.float64))

    def call(cols, mask, w, E):
        if mode == "pinned":
            cols, mask = [c.pin_memory() for c in cols], mask.pin_memory()
        h = pk.Handle.get(0)
        sums, dth = np.zeros(8), np.zeros(1521)
        wv = np.ascontiguousarray(w)
        P = lambda a: ctypes.c_void_p(a.ctypes.data)
        TP = lambda x: ctypes.c_void_p(x.data_ptr())
        rc = h.L.pinn_loss_fwd_bwd_host(h.h, 0, cols[0].numel(), *[TP(c) for c in cols], 0, TP(mask), P(th64), P(wv),
                                        0xFFFF, 17.5, P(sums), P(dth), TP(E))
        h.check(rc, "pinn_loss_fwd_bwd_host")
        return sums, dth
    return call


def case_result(cid, init_theta, ck, reference):
    """Run case `cid` (once per module) -> (res, ref, loss, grad, trained); prints its line of the table."""
    if cid not in _RESULTS:
        variant, weights, kind, K = CASES[cid]
        need_memory(K)
        th32 = (init_theta if weights == "init" else ck["ionHsym"]).astype(np.float32)
        tensors = range(16)
        if kind in ("packed", "f64"):
            res = run_case(variant, th32, K, packed_call(variant, th32), dtype=np.float64 if kind == "f64" else np.float32)
        elif kind == "finetune":
            res = run_case(variant, th32, K, packed_call(variant, th32, pk.FINE_TUNE_GRAD_MASK), grad_mask=pk.FINE_TUNE_GRAD_MASK)
            tensors = range(6, 12)
        elif kind == "tensors":
            res = run_case(variant, th32, K, tensor_call(variant, th32), E_dtype=torch.float64)
        else:
            res = run_case(variant, th32, K, host_call(kind[5:], th32), where="cpu")
        ref = reference(variant, th32, K)
        loss, grad = errors(res, ref, tensors)
        report(cid, res, loss, grad, tensors)
        _RESULTS[cid] = (res, ref, loss, grad, weights == "trained")
    return _RESULTS[cid]


# ---------------------------------------------------------------------------------------------
# GPU: pinn_loss_fwd_bwd, packed theta
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("variant", [0, 1])
def test_packed_entry_at_scale(variant, K, init_theta, ck, reference):
    check(*case_result("%s-init-K%d" % (FORMS[variant], K), init_theta, ck, reference))


@pytest.mark.gpu
@pytest.mark.parametrize("K", KS)
def test_packed_entry_at_scale_trained_weights(K, init_theta, ck, reference):
    check(*case_result("poc-trained-K%d" % K, init_theta, ck, reference))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 1])
def test_packed_entry_float64_coordinates(variant, init_theta, ck, reference):
    """8-byte coordinates: the per-lane cp.async stage over 886 super-tiles per SM (K = 256)."""
    check(*case_result("%s-f64-K256" % FORMS[variant], init_theta, ck, reference))


@pytest.mark.gpu
def test_fine_tune_mask_at_scale(init_theta, ck, reference):
    """freezeBase + freezeDecayUnit: the MLP warps run no reverse sweep and carry only the loss sums over the launch."""
    res, ref, loss, grad, trained = case_result("poc-finetune-K1024", init_theta, ck, reference)
    assert np.all(res["dth"][:OFFS[6]] == 0) and np.all(res["dth"][OFFS[12]:] == 0)
    check(res, ref, loss, grad, trained)


# ---------------------------------------------------------------------------------------------
# GPU: the other training entry points
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["poc", "trainpy"])
def test_tensor_entry_at_scale(order, init_theta, ck, reference):
    """pinn_loss_fwd_bwd_tensors: 16 float64 parameter tensors in the caller's layout, E_out in float64."""
    check(*case_result("%s-tensors-K256" % order, init_theta, ck, reference))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pinned", "pageable"])
def test_host_entry_at_scale(mode, init_theta, ck, reference):
    """pinn_loss_fwd_bwd_host on 2^24 points in host memory: pinned columns are read in place by the kernel instance that
    takes theta and the weights in its parameters; pageable ones are staged in 4 overlapped chunks."""
    check(*case_result("poc-host-%s-K256" % mode, init_theta, ck, reference))


# ---------------------------------------------------------------------------------------------
# GPU: the two tensors summed by mma.sync, at the same bars, in every case
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cid", [pytest.param(c, marks=pytest.mark.xfail(strict=True, reason=MMA_REASON))
                                 if c in MMA_MISSES else c for c in CASES])
def test_mma_sync_gradients_at_scale(cid, init_theta, ck, reference):
    res, ref, _, grad, trained = case_result(cid, init_theta, ck, reference)
    check_mma_sync_tensors(res, ref, grad, trained)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 1])
def test_trainer_at_scale(variant, init_theta, reference):
    """Trainer.set_batch + run(1) + read: history row 0 is {Ltot, Lpde, Lbc, mean E} of the batch."""
    K = 64
    th32 = init_theta.astype(np.float32)
    a32, m1, m2 = sample_block(variant)
    n, w = tiled_size_and_weights(m1, m2, K)
    cols = [tile_t(t(a), K) for a in a32]
    mask = tile_t(t((m1 + 2 * m2).astype(np.uint8)), K)
    tr = pk.Trainer(variant, n, th32.astype(np.float64), history_capacity=1, history_mean_E=True)
    try:
        tr.set_batch(*cols, mask, w)
        tr.run(1, resample=False)
        row = tr.read()["history"][0]
    finally:
        tr.close()
    del cols, mask
    ref = reference(variant, th32, K)
    err = {"Ltot": row[0] / ref["Ltot"] - 1, "Lpde": row[1] / ref["Lpde"] - 1, "Lbc": row[2] / ref["Lbc"] - 1,
           "meanE": row[3] / (ref["sums"][0] / n) - 1}
    print("\n%-30s n %9d | %s" % ("%s trainer K=%d" % (FORMS[variant], K), n, " ".join("%s %.1e" % kv for kv in err.items())))
    assert all(abs(v) < 1e-5 for v in err.values()), err
