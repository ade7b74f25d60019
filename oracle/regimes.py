"""Saturated-sigmoid regimes of the network's weights (TEST INFRASTRUCTURE ONLY).

Built from train.py's init vector by shifting one layer's biases (and shrinking a unit's weights where its input range
would not fit in the band) so that every unit's pre-activation lies in the band for ANY point: the inputs of a layer are
bounded (exp(-r) and sigmoids in [0, 1], R in the union of the two samplers' ranges [0.2, 4]).  In u in [8, 12] and in
[-12, -8], 1 - sigma(u) is e^-u, between 6e-6 and 3e-4.
"""
import numpy as np

from . import layout

BAND = (8.0, 12.0)
HALF = 1.8                        # every unit is put in [10 - HALF, 10 + HALF] (or its negative): inside BAND with margin
R_RANGE = (0.2, 4.0)              # poc samples R in [0.2, 4], train.py in [0.2, 3]

# sigmoid layer: (weight tensor, bias tensor) in the canonical layout; inputs of the base and E-net second layers are
# sigmoids, of the base first layer exp(-r1), exp(-r2), of the E-net and gate first layers R
LAYERS = {"base_L1": (0, 1), "base_L2": (2, 3), "enet_L1": (6, 7), "enet_L2": (8, 9), "gate_L1": (12, 13)}
INPUT_RANGE = {"base_L1": (0.0, 1.0), "base_L2": (0.0, 1.0), "enet_L1": R_RANGE, "enet_L2": (0.0, 1.0), "gate_L1": R_RANGE}


def unit_signs(layer, sign):
    n = layout.POC_TENSORS[LAYERS[layer][1]][1][0]
    if sign != "mixed":
        return np.full(n, 1.0 if sign == "pos" else -1.0)
    # the mixed regime saturates all five layers at once, two units in three on the positive side
    return np.where(np.arange(n) % 3 == 2, -1.0, 1.0)


REGIMES = {f"{layer}_{sign}": {layer: sign} for layer in LAYERS for sign in ("pos", "neg")}
REGIMES["mixed"] = {layer: "mixed" for layer in LAYERS}


def regime_theta(init, name):
    """init (1521,) float64 -> the regime's weights, rounded to float32 (what the kernel is given)."""
    P = [p.copy() for p in layout.unpack_poc(np.asarray(init, np.float64))]
    for layer, sign in REGIMES[name].items():
        iw, ib = LAYERS[layer]
        W = P[iw].reshape(P[ib].size, -1)
        lo_in, hi_in = INPUT_RANGE[layer]
        lo = np.minimum(W * lo_in, W * hi_in).sum(1)          # range of W x over every admissible input x
        hi = np.maximum(W * lo_in, W * hi_in).sum(1)
        shrink = np.minimum(1.0, 2 * HALF / np.maximum(hi - lo, 1e-300))
        W *= shrink[:, None]
        mid = 0.5 * (lo + hi) * shrink
        P[iw] = W.reshape(P[iw].shape)
        P[ib] = 10.0 * unit_signs(layer, sign) - mid
    return layout.pack_poc(P).astype(np.float32)
