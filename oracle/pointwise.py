"""Per-point error bound of a float32 evaluation of the fields (TEST INFRASTRUCTURE ONLY).

A norm bar max|got - ref| / max|ref| sets one absolute tolerance per array, from its largest point: on most points of a
trained network it would accept a 1 % error, or zero.  A relative bar per point does not work either, because psi and the
residual are cancellations.  ``magnitudes`` is a first-order running-error pass over the same formulas as
closed_form._forward, in the kernel's order of operations: for every quantity q it carries a magnitude M_q such that a
float32 evaluation satisfies |fl(q) - q| <~ u M_q, u = 2^-24, at that point:

    sums            M = sum M_terms + |result|; a sequential chain adds every partial sum
    products        M_ab = M_a |b| + |a| M_b + |ab|
    sigma^(j)(u)    M = |sigma^(j)(u)| + |sigma^(j+1)(u)| M_u   (the function's own sensitivity, which the kernel's
                    sigma' = (e s) s reaches; s - s^2 would not)

Inputs enter with the error of their rounding, so that f = e^-r carries (1 + r)|f| and the alpha terms their cancelling
parts.  ``excess`` is the largest ratio of an error to its bound.  ``forward32`` restates the kernel's forward in float32
(fused multiply-adds, the (e s) s derivative, the three-product TF32 split of the tensor-core layers); it exists to check
the pass, and takes the planted defects of tests/test_oracle_pointwise.py.
"""
import numpy as np

from . import layout
from .closed_form import VARIANTS

U = 2.0 ** -24
NEG_LOG2E = np.float32(-1.4426950408889634)
OUTPUTS = ("psi", "lap", "hpsi", "res", "E")
DEFECTS = ("farfield", "noswap", "tf32", "s_minus_s2")
# the bound the kernel is held to: C u M per point.  The largest excess measured on a B200 over every GPU case is 0.53
# (DESIGN.md section 4); C is that times 4 or more, rounded up to a power of two.
C_KERNEL = 4.0


# ---------------------------------------------------------------------------------------------
# the running-error pass (float64): every quantity is a pair (value, magnitude)
# ---------------------------------------------------------------------------------------------
class _Q:
    __slots__ = ("v", "m")

    def __init__(self, v, m):
        self.v, self.m = v, m


def _in(v):
    """An input rounded once to float32."""
    return _Q(v, np.abs(v))


def _w(v, roundings=0):
    """A weight: exact, or the product of `roundings` float32 roundings (the kernel's pre-scaled and product weights)."""
    return _Q(v, roundings * np.abs(v))


def _add(*ts):
    v = sum(t.v for t in ts)
    return _Q(v, sum(t.m for t in ts) + np.abs(v))


def _mul(a, b):
    v = a.v * b.v
    return _Q(v, a.m * np.abs(b.v) + np.abs(a.v) * b.m + np.abs(v))


def _neg(a):
    return _Q(-a.v, a.m)


def _scale(c, a):
    """Multiplication by an exact power of two (or by a sign): no rounding."""
    return _Q(c * a.v, abs(c) * a.m)


def _dot(A, W, MW):
    """A (points x K) times W (K x J) on the tensor core or in a sequential loop; MW = magnitudes of W's own rounding."""
    v = A.v @ W
    return _Q(v, A.m @ np.abs(W) + np.abs(A.v) @ MW + np.abs(A.v) @ np.abs(W) + np.abs(v))


def _fold(A, w, init, wr):
    """init + sum_j w_j A[:, j] as a sequential chain of fused multiply-adds (the kernel's N, D, E and gate): every
    partial sum is rounded, so each enters M with its own magnitude."""
    v, m = np.broadcast_to(np.asarray(init.v, np.float64), A.v.shape[:1]), init.m
    for j in range(w.size):
        v = v + w[j] * A.v[:, j]
        m = m + abs(w[j]) * (A.m[:, j] + wr * np.abs(A.v[:, j])) + np.abs(v)
    return _Q(v, m)


def _sigmoids(u):
    """s, s', s'' of the pre-activation u (pairs).  s'' = s' (1 - 2 s) is formed as fma(-2 s, s', s'), which cancels at
    s = 1/2: the rounding of s' enters it with |s'|, beyond the function's own sensitivity."""
    s = 1.0 / (1.0 + np.exp(-u.v))
    sp = s * (1.0 - s)
    spp = sp * (1.0 - 2.0 * s)
    sppp = sp * (1.0 - 6.0 * sp)
    return (_Q(s, s + sp * u.m), _Q(sp, sp + np.abs(spp) * u.m), _Q(spp, np.abs(spp) + sp + np.abs(sppp) * u.m))


def _geometry(x, y, z, R):
    dx1, dx2 = _in(x - R), _in(x + R)
    y, z = _in(y), _in(z)
    yz = _add(_mul(y, y), _mul(z, z))
    q1, q2 = _add(_mul(dx1, dx1), yz), _add(_mul(dx2, dx2), yz)
    ir = []
    for q in (q1, q2):
        v = 1.0 / np.sqrt(q.v)
        ir.append(_Q(v, v + 0.5 * v * q.m / q.v))  # rsqrt: relative, plus half the relative error of its argument
    ir1, ir2 = ir
    r1, r2 = _mul(q1, ir1), _mul(q2, ir2)
    f1, f2 = [_Q(np.exp(-r.v), np.exp(-r.v) * (1.0 + r.m)) for r in (r1, r2)]
    one = _w(np.ones_like(x))
    c12 = _mul(_mul(_add(_mul(dx1, dx2), yz), ir1), ir2)
    return dict(f1=f1, f2=f2, ir1=ir1, ir2=ir2,
                al1=_mul(f1, _add(_scale(-2.0, ir1), one)), al2=_mul(f2, _add(_scale(-2.0, ir2), one)),
                al11=_mul(f1, f1), al22=_mul(f2, f2), al12=_scale(2.0, _mul(_mul(f1, f2), c12)), R=_in(R))


def _col(q):
    return _Q(q.v[:, None], q.m[:, None])


def _mlp(P, a, b, al1, al2, al11, al12, al22, wr):
    """The base MLP as tc_mlp_forward evaluates it: the D channel of layer 2 is al1 V1 + al2 V2 + al11 P00 + al12 P01
    + al22 P11, with V1 = s' (W2 w0), ..., P11 = s'' (W2 w1^2) from the tensor core."""
    W1, b1, W2, b2, wo = P[0], P[1], P[2], P[3], P[4].reshape(-1)
    w0, w1 = W1[:, 0], W1[:, 1]
    a, b, al1, al2, al11, al12, al22 = map(_col, (a, b, al1, al2, al11, al12, al22))
    u = _add(_mul(a, _w(w0, 1 + wr)), _mul(b, _w(w1, 1 + wr)), _w(b1, 1 + wr))
    s, sp, spp = _sigmoids(u)
    # B operands W2 w0 ... carry one rounding, W2 w0^2 ... two
    dot = lambda A, c, k: _dot(A, (W2 * c).T, (k + wr) * np.abs((W2 * c).T))
    V0 = dot(s, 1.0, 0)
    V1, V2 = dot(sp, w0, 1), dot(sp, w1, 1)
    P00, P01, P11 = dot(spp, w0 * w0, 2), dot(spp, w0 * w1, 2), dot(spp, w1 * w1, 2)
    v3 = _add(_mul(al1, V1), _mul(al2, V2), _mul(al11, P00), _mul(al12, P01), _mul(al22, P11))
    t, tp, tpp = _sigmoids(_add(_mul(V0, _w(np.ones(1), 1)), _w(b2, 1 + wr)))
    Q = _add(_mul(_mul(al11, V1), V1), _mul(_mul(al12, V1), V2), _mul(_mul(al22, V2), V2))
    gD = _add(_mul(tp, v3), _mul(tpp, Q))
    zero = _w(0.0)
    return _fold(t, wo, zero, wr), _fold(gD, wo, zero, wr)


def _enet_gate(P, R, wr):
    WE1, bE1, WE2, bE2, wE, bE = P[6].reshape(-1), P[7], P[8], P[9], P[10].reshape(-1), P[11]
    Rc = _col(R)
    e1, _, _ = _sigmoids(_add(_mul(Rc, _w(WE1, 1 + wr)), _w(bE1, 1 + wr)))
    e2, _, _ = _sigmoids(_add(_mul(_dot(e1, WE2.T, wr * np.abs(WE2.T)), _w(np.ones(1), 1)), _w(bE2, 1 + wr)))
    E = _fold(e2, wE, _w(bE[0], wr), wr)
    WgL, bgL, wg, bg = P[12].reshape(-1), P[13], P[14].reshape(-1), P[15]
    s, _, _ = _sigmoids(_add(_mul(Rc, _w(WgL, 1 + wr)), _w(bgL, 1 + wr)))
    return E, _fold(s, wg, _w(bg[0], wr), wr)


def magnitudes(variant, theta, x, y, z, R, rounded_weights=False):
    """Per-point M of psi, lap, hpsi, res and E: a float32 evaluation is within about u M of the exact value.
    rounded_weights: the reference holds float64 weights that the evaluation rounds to float32 (one more rounding each)."""
    wr = int(rounded_weights)
    nev, sN, cL, cV, cE = VARIANTS[variant]
    P = layout.unpack_poc(np.asarray(theta, np.float64))
    x, y, z, R = [np.asarray(v, np.float64).reshape(-1) for v in (x, y, z, R)]
    g = _geometry(x, y, z, R)
    f1, f2, ir1, ir2 = g["f1"], g["f2"], g["ir1"], g["ir2"]
    NA, DA = _mlp(P, f1, f2, g["al1"], g["al2"], g["al11"], g["al12"], g["al22"], wr)
    if nev == 2:
        NB, DB = _mlp(P, f2, f1, g["al2"], g["al1"], g["al22"], g["al12"], g["al11"], wr)
        NA, DA = _add(NA, NB), _add(DA, DB)
    N = _add(_scale(sN, NA), _w(P[5][0], wr))
    DN = _scale(sN, DA)
    E, gate = _enet_gate(P, g["R"], wr)
    q = _add(ir1, ir2)
    fs = _add(f1, f2)
    psi = _add(_mul(gate, N), fs)
    cross = _add(_mul(f1, ir2), _mul(f2, ir1))
    lcao = _add(_scale(cL, fs), _mul(_w(cV - 2 * cL), _add(_mul(f1, ir1), _mul(f2, ir2))), _mul(_w(cV), cross))
    inner = _add(_scale(cL, DN), _mul(_mul(_w(cV), q), N))
    res = _add(_mul(gate, inner), _mul(_mul(_w(cE), E), psi), lcao)
    lap = _add(g["al1"], g["al2"], _mul(gate, DN))
    hpsi = _add(_mul(gate, _add(_scale(-0.5, DN), _neg(_mul(q, N)))), _scale(-0.5, fs), _neg(cross))
    return dict(psi=psi.m, lap=lap.m, hpsi=hpsi.m, res=res.m, E=E.m)


def excess(got, ref, M, C):
    """max_i |got_i - ref_i| / (C u M_i): at most 1 when every point is within C times its bound."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return float(np.max(np.abs(got - ref) / (C * U * np.asarray(M, np.float64) + 1e-37)))


def worst(got, ref, M, k=5):
    """Indices of the k points with the largest error over bound, worst first."""
    r = np.abs(np.asarray(got, np.float64) - ref) / (U * np.asarray(M, np.float64) + 1e-37)
    return np.argsort(r)[::-1][:k], r


# ---------------------------------------------------------------------------------------------
# float32 restatement of the kernel's forward
# ---------------------------------------------------------------------------------------------
f32 = np.float32


def _fma(a, b, c):
    """a b + c with one rounding: the float32 product is exact in float64."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(f32)


def _tf32(x, nearest):
    """x with its low 13 mantissa bits cleared, after adding half of their range (nearest) or not (truncation)."""
    b = np.ascontiguousarray(x, f32).view(np.uint32)
    if nearest:
        b = b + np.uint32(0x1000)
    return (b & np.uint32(0xFFFFE000)).view(f32)


def _mma(A, W, plain=False):
    """A (points x K) times W (K x J) as the kernel's tensor core forms it: A = hi + lo rounded to nearest with lo
    truncated to TF32, W = hi + lo both rounded to nearest, products hi hi + hi lo + lo hi accumulated in float32."""
    A, W = np.asarray(A, f32), np.asarray(W, f32)
    ah = _tf32(A, True)
    al = _tf32((A - ah).astype(f32), False)
    wh = _tf32(W, True)
    wl = _tf32((W - wh).astype(f32), True)
    out = ah @ wh
    if not plain:
        out = (out + ah @ wl) + al @ wh
    return out.astype(f32)


def _sig32(up, defect=None):
    """sigm2_pre: s = 1 / (1 + e), e = 2^up, and s' = (e s) s; with defect 's_minus_s2', s' = s - s^2."""
    e = np.exp2(up.astype(np.float64)).astype(f32)
    s = (1.0 / (e.astype(np.float64) + 1.0).astype(f32).astype(np.float64)).astype(f32)
    if defect == "s_minus_s2":
        return s, (s - s * s).astype(f32)
    om = np.clip((e * s).astype(f32), 0.0, 1.0)
    return s, (om * s).astype(f32)


def _mlp32(P, a, b, al1, al2, al11, al12, al22, defect):
    W1, b1, W2, b2, wo = [np.asarray(p, f32) for p in (P[0], P[1], P[2], P[3], P[4].reshape(-1))]
    w0, w1 = W1[:, 0], W1[:, 1]
    c = lambda v: v[:, None]
    w0s, w1s, b1s, b2s = [(v * NEG_LOG2E).astype(f32) for v in (w0, w1, b1, b2)]
    u = _fma(c(a), w0s, _fma(c(b), w1s, b1s))
    s, sp = _sig32(u, defect)
    spp = _fma((f32(-2.0) * s).astype(f32), sp, sp)
    plain = defect == "tf32"
    V0 = _mma(s, W2.T, plain)
    V1 = _mma(sp, ((W2 * w0).astype(f32)).T, plain)
    V2 = _mma(sp, ((W2 * w1).astype(f32)).T, plain)
    P00 = _mma(spp, (W2 * (w0 * w0).astype(f32)).astype(f32).T, plain)
    P01 = _mma(spp, (W2 * (w0 * w1).astype(f32)).astype(f32).T, plain)
    P11 = _mma(spp, (W2 * (w1 * w1).astype(f32)).astype(f32).T, plain)
    v3 = _fma(c(al1), V1, _fma(c(al2), V2, _fma(c(al11), P00, _fma(c(al12), P01, (c(al22) * P11).astype(f32)))))
    t, tp = _sig32(_fma(V0, NEG_LOG2E, b2s), defect)
    tpp = _fma((f32(-2.0) * t).astype(f32), tp, tp)
    Q = _fma((c(al11) * V1).astype(f32), V1, _fma((c(al12) * V1).astype(f32), V2,
                                                 ((c(al22) * V2).astype(f32) * V2).astype(f32)))
    gD = _fma(tp, v3, (tpp * Q).astype(f32))
    accN = np.zeros(a.size, f32)
    accD = np.zeros(a.size, f32)
    for j in range(wo.size):
        accN = _fma(wo[j], t[:, j], accN)
        accD = _fma(wo[j], gD[:, j], accD)
    return accN, accD


def forward32(variant, theta, x, y, z, R, defect=None):
    """The kernel's forward in float32 -> dict of psi, lap, hpsi, res, E (float32 arrays).  x, y, z, R as the kernel
    takes them: float32, or float64 (then x -/+ R is formed in float64 and rounded).  `defect` plants one of DEFECTS:
    'farfield' drops cV (f1/r2 + f2/r1) where f1 + f2 < 1e-5; 'noswap' evaluates the poc form's inversion image without
    swapping al11 and al22; 'tf32' runs the tensor-core layers on hi x hi only; 's_minus_s2' forms s' as s - s^2."""
    assert defect in (None,) + DEFECTS
    nev, sN, cL, cV, cE = [f32(v) for v in VARIANTS[variant]]
    P = layout.unpack_poc(np.asarray(theta, np.float64).astype(f32).astype(np.float64))
    x, y, z, R = [np.asarray(v).reshape(-1) for v in (x, y, z, R)]
    dx1, dx2 = (x - R).astype(f32), (x + R).astype(f32)  # one rounding, from float32 or float64 inputs
    y, z, R = y.astype(f32), z.astype(f32), R.astype(f32)
    yz = _fma(y, y, (z * z).astype(f32))
    q1, q2 = _fma(dx1, dx1, yz), _fma(dx2, dx2, yz)
    ir1 = (1.0 / np.sqrt(q1.astype(np.float64))).astype(f32)
    ir2 = (1.0 / np.sqrt(q2.astype(np.float64))).astype(f32)
    r1, r2 = (q1 * ir1).astype(f32), (q2 * ir2).astype(f32)
    f1, f2 = np.exp(-r1.astype(np.float64)).astype(f32), np.exp(-r2.astype(np.float64)).astype(f32)
    c12 = ((_fma(dx1, dx2, yz) * ir1).astype(f32) * ir2).astype(f32)
    al1, al2 = (f1 * _fma(f32(-2.0), ir1, f32(1.0))).astype(f32), (f2 * _fma(f32(-2.0), ir2, f32(1.0))).astype(f32)
    al11, al22 = (f1 * f1).astype(f32), (f2 * f2).astype(f32)
    al12 = ((f32(2.0) * f1).astype(f32) * f2 * c12).astype(f32)
    NA, DA = _mlp32(P, f1, f2, al1, al2, al11, al12, al22, defect)
    if int(nev) == 2:
        s11, s22 = (al11, al22) if defect == "noswap" else (al22, al11)
        NB, DB = _mlp32(P, f2, f1, al2, al1, s11, al12, s22, defect)
        NA, DA = (NA + NB).astype(f32), (DA + DB).astype(f32)
    N = _fma(sN, NA, f32(P[5][0]))
    DN = (sN * DA).astype(f32)
    # E-net and gate
    WE1s, bE1s, bE2s = [(np.asarray(v, f32).reshape(-1) * NEG_LOG2E).astype(f32) for v in (P[6], P[7], P[9])]
    e1, _ = _sig32(_fma(R[:, None], WE1s, bE1s), defect)
    e2, _ = _sig32(_fma(_mma(e1, np.asarray(P[8], f32).T, defect == "tf32"), NEG_LOG2E, bE2s), defect)
    wE = np.asarray(P[10], f32).reshape(-1)
    E = np.full(R.size, f32(P[11][0]))
    for j in range(wE.size):
        E = _fma(wE[j], e2[:, j], E)
    WgLs, bgLs = [(np.asarray(v, f32).reshape(-1) * NEG_LOG2E).astype(f32) for v in (P[12], P[13])]
    sg, _ = _sig32(_fma(R[:, None], WgLs, bgLs), defect)
    wg = np.asarray(P[14], f32).reshape(-1)
    gate = np.full(R.size, f32(P[15][0]))
    for j in range(wg.size):
        gate = _fma(wg[j], sg[:, j], gate)
    # combine
    q = (ir1 + ir2).astype(f32)
    fs = (f1 + f2).astype(f32)
    psi = _fma(gate, N, fs)
    cross = _fma(f1, ir2, (f2 * ir1).astype(f32))
    if defect == "farfield":
        cross = np.where(fs < 1e-5, f32(0.0), cross)
    lcao = _fma(cL, fs, _fma(cV - f32(2.0) * cL, _fma(f1, ir1, (f2 * ir2).astype(f32)), (cV * cross).astype(f32)))
    inner = _fma(cL, DN, ((cV * q).astype(f32) * N).astype(f32))
    res = _fma(gate, inner, _fma((cE * E).astype(f32), psi, lcao))
    lap = ((al1 + al2).astype(f32) + (gate * DN).astype(f32)).astype(f32)
    hpsi = _fma(gate, _fma(f32(-0.5), DN, (-q * N).astype(f32)), _fma(f32(-0.5), fs, -cross))
    return dict(psi=psi, lap=lap, hpsi=hpsi, res=res, E=E)


def check(tag, got, ref, M, C, coords=None):
    """Assert that every output in `got` (name -> array) is within C u M of `ref` at every point.  Prints the excess at
    C = 1 per output (the figure C is set from) and, on failure, the worst points with their coordinates."""
    ex = {k: excess(got[k], ref[k], M[k], 1.0) for k in got}
    print("%s: excess/C=1 %s" % (tag, " ".join("%s %.3g" % kv for kv in ex.items())))
    bad = {k: v for k, v in ex.items() if not v <= C}
    if bad and coords is not None:
        for k in bad:
            idx, r = worst(got[k], ref[k], M[k])
            for i in idx:
                print("    %s point %d: x y z R = %s  got %.9g ref %.9g M %.3g  ratio %.3g"
                      % (k, i, " ".join("%.9g" % float(c[i]) for c in coords), float(got[k][i]), float(ref[k][i]),
                         float(M[k][i]), r[i]))
    assert not bad, (tag, bad, C)
