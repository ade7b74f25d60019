"""Python mirror of the reference's hot-path call sites on top of the C ABI.

    loss_poc(...)      <->  NN_ion.LossFunctions(x,y,z,R,params,bIndex1,bIndex2)   poc/main.py:341-355
    loss_trainpy(...)  <->  the inline block train.py:41-57
    fields(...)        <->  parametricPsi + hamiltonian                             poc/main.py:321, 118, 451-454

The parameter gradient is produced by the same fused kernel launch as the loss (the upstream
gradient of a scalar loss is a scalar), stashed on the autograd context, and ``backward`` only
scales it - no second kernel, no saved activations (SURVEY.md 8b).
"""
import ctypes

import torch

from . import params as P
from ._lib import Handle, PinnError

VARIANT_POC, VARIANT_TRAINPY = 0, 1
_F32, _F64 = 0, 1
BC_CUTOFF = 17.5  # params['BCcutoff'] poc/main.py:25 ; bcutoff train.py:78


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _col(t, name):
    """(n,1) or (n,) float32/float64 tensor -> contiguous 1-D view + dtype code."""
    if t.dim() == 2 and t.shape[1] == 1:
        t = t[:, 0]
    if t.dim() != 1:
        raise ValueError("%s must have shape (n,) or (n,1), got %s" % (name, tuple(t.shape)))
    if t.dtype not in (torch.float32, torch.float64):
        raise TypeError("%s must be float32 or float64" % name)
    return t.detach().contiguous()


def indices_to_mask(n, idx1, idx2, device):
    """Boundary index sets (torch.where tuples as in poc/main.py:392-393, or 1-D row indices as in
    train.py:38-39) -> per-point uint8 mask (bit0: set 1, bit1: set 2) and the two set sizes."""
    def rows(ix):
        if isinstance(ix, (tuple, list)):
            ix = ix[0]
        return ix.to(device=device, dtype=torch.long).reshape(-1)
    r1, r2 = rows(idx1), rows(idx2)
    mask = torch.zeros(n, dtype=torch.uint8, device=device)
    m2 = torch.zeros(n, dtype=torch.uint8, device=device)
    mask[r1] = 1
    m2[r2] = 2
    mask |= m2
    return mask, int(r1.numel()), int(r2.numel())


def check_point_weights(point_weights, n, device):
    """Refuse malformed per-point loss weights: a contiguous float32 tensor of n finite values >= 0 on `device`.  The
    value check reads the tensor back (one synchronisation of torch's current stream)."""
    w = point_weights
    if not torch.is_tensor(w) or w.dtype != torch.float32 or w.dim() != 1 or w.numel() != n or not w.is_contiguous():
        raise ValueError("point_weights must be a contiguous float32 vector of n = %d elements" % n)
    if w.device != device:
        raise ValueError("point_weights must be on %s, got %s" % (device, w.device))
    if not bool(torch.isfinite(w).all()) or bool((w < 0).any()):
        raise ValueError("point_weights must be finite and >= 0")


def loss_and_grad_raw(variant, x, y, z, R, theta, mask=None, weights=None, grad_mask=0xFFFF, want_E=False,
                      bcutoff=BC_CUTOFF, sums=None, dtheta=None, E_out=None, point_weights=None):
    """Thin wrapper over pinn_loss_fwd_bwd for DEVICE tensors (no allocation when the outputs are given).

    x,y,z,R: CUDA float32/float64 (n,) ; theta: CUDA float32 (1521,) ; mask: CUDA uint8 (n,) or None ;
    weights: CUDA float64 (3,) or None.  Returns (sums[8] f64, dtheta[1521] f64, E_out or None), all on
    the device, enqueued on torch's current stream.
    point_weights: None, or CUDA float32 (n,) per-point loss weights om >= 0 (pinn_loss_fwd_bwd_weighted): every
    per-point term of the sums and of the gradient takes its om, the counted set sizes do not - e.g. the "point_weights"
    of sample_adaptive(importance=True) with its "weights"."""
    if not x.is_cuda:
        raise PinnError("loss_and_grad_raw needs CUDA tensors (there is no CPU path)")
    dev = x.device
    h = Handle.get(dev.index if dev.index is not None else torch.cuda.current_device())
    n = x.numel()
    code = _F64 if x.dtype == torch.float64 else _F32
    for t in (y, z, R):
        if t.dtype != x.dtype or t.numel() != n or not t.is_contiguous():
            raise ValueError("x,y,z,R must share dtype/length and be contiguous")
    if theta.dtype != torch.float32 or theta.numel() != P.N_THETA or not theta.is_contiguous():
        raise ValueError("theta must be a contiguous float32 vector of 1521 elements")
    if sums is None:
        sums = torch.empty(8, dtype=torch.float64, device=dev)
    if dtheta is None:
        dtheta = torch.empty(P.N_THETA, dtype=torch.float64, device=dev)
    if want_E and E_out is None:
        E_out = torch.empty(n, dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    if point_weights is not None:
        check_point_weights(point_weights, n, dev)
        rc = h.L.pinn_loss_fwd_bwd_weighted(h.h, int(variant), n, _ptr(x), _ptr(y), _ptr(z), _ptr(R), code, _ptr(mask),
                                            _ptr(theta), _ptr(weights), _ptr(point_weights), int(grad_mask),
                                            float(bcutoff), _ptr(sums), _ptr(dtheta), _ptr(E_out), ctypes.c_void_p(stream))
        h.check(rc, "pinn_loss_fwd_bwd_weighted")
        return sums, dtheta, E_out
    rc = h.L.pinn_loss_fwd_bwd(h.h, int(variant), n, _ptr(x), _ptr(y), _ptr(z), _ptr(R), code, _ptr(mask),
                               _ptr(theta), _ptr(weights), int(grad_mask), float(bcutoff), _ptr(sums),
                               _ptr(dtheta), _ptr(E_out), ctypes.c_void_p(stream))
    h.check(rc, "pinn_loss_fwd_bwd")
    return sums, dtheta, E_out


def loss_eval(variant, x, y, z, R, theta, mask=None, weights=None, bcutoff=BC_CUTOFF, sums=None):
    """The loss without its gradient (pinn_loss_eval) for DEVICE tensors: a forward-only kernel that accumulates in float64
    and stores nothing per point.

    x,y,z,R: CUDA float32/float64 (n,) ; theta: CUDA float32 (1521,) ; mask: CUDA uint8 (n,) or None (sets by r >= bcutoff);
    weights: CUDA float64 (3,) {w_pde, w_bc1, w_bc2} or None ({1/n, 1/|set1|, 1/|set2|} of the counted sets).  Returns the
    8 sums of loss_and_grad_raw as a float64 CUDA tensor {Ltot, Lpde, Lbc, sum E, sum res^2, sum psi^2 set 1, sum psi^2
    set 2, E of the last point}, enqueued on torch's current stream."""
    variant = {"poc": 0, "trainpy": 1}.get(variant, variant)
    if not x.is_cuda:
        raise PinnError("loss_eval needs CUDA tensors (there is no CPU path)")
    dev = x.device
    h = Handle.get(dev.index if dev.index is not None else torch.cuda.current_device())
    n = x.numel()
    code = _F64 if x.dtype == torch.float64 else _F32
    for t in (x, y, z, R):
        if t.dtype != x.dtype or t.numel() != n or not t.is_contiguous() or t.device != dev:
            raise ValueError("x,y,z,R must share dtype/length/device and be contiguous")
    if theta.dtype != torch.float32 or theta.numel() != P.N_THETA or not theta.is_contiguous() or theta.device != dev:
        raise ValueError("theta must be a contiguous float32 CUDA vector of 1521 elements on the points' device")
    if mask is not None and (mask.dtype != torch.uint8 or mask.numel() != n or not mask.is_contiguous() or mask.device != dev):
        raise ValueError("mask must be a contiguous uint8 CUDA tensor of n elements")
    if weights is not None and (weights.dtype != torch.float64 or weights.numel() < 3 or weights.device != dev):
        raise ValueError("weights must be a float64 CUDA tensor of 3 elements")
    if sums is None:
        sums = torch.empty(8, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    rc = h.L.pinn_loss_eval(h.h, int(variant), n, _ptr(x), _ptr(y), _ptr(z), _ptr(R), code, _ptr(mask), _ptr(theta),
                            _ptr(weights), float(bcutoff), _ptr(sums), ctypes.c_void_p(stream))
    h.check(rc, "pinn_loss_eval")
    return sums


def _host_step(variant, x, y, z, R, theta64, mask, weights, grad_mask, want_E, bcutoff):
    """CPU tensors in, CPU float64 results out, through pinn_loss_fwd_bwd_host on cuda:current."""
    if not torch.cuda.is_available():
        raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
    h = Handle.get(torch.cuda.current_device())
    n = x.numel()
    code = _F64 if x.dtype == torch.float64 else _F32
    sums = torch.empty(8, dtype=torch.float64)
    dtheta = torch.empty(P.N_THETA, dtype=torch.float64)
    E_out = torch.empty(n, dtype=torch.float32) if want_E else None
    w = (ctypes.c_double * 3)(*weights) if weights is not None else None
    rc = h.L.pinn_loss_fwd_bwd_host(h.h, int(variant), n, _ptr(x), _ptr(y), _ptr(z), _ptr(R), code, _ptr(mask),
                                    _ptr(theta64), ctypes.cast(w, ctypes.c_void_p) if w is not None else None,
                                    int(grad_mask), float(bcutoff), _ptr(sums), _ptr(dtheta), _ptr(E_out))
    h.check(rc, "pinn_loss_fwd_bwd_host")
    return sums, dtheta, E_out


class HostStep:
    """A training evaluation on one fixed set of HOST buffers, prepared once and called many times
    (``pinn_loss_fwd_bwd_host``).  Binding the 16 ctypes arguments costs ~15 microseconds in Python, an order of
    magnitude more than the library needs to enqueue the work; a loop that reuses its batch buffers (the reference's
    training loops do) prepares the call once per buffer set.  Pin the tensors (``tensor.pin_memory()``) to let the
    kernel read them in place.

        step = HostStep("poc", x, y, z, R)            # CPU float32/float64 tensors, (n,) or (n,1); optional uint8 mask
        sums, dtheta = step(theta64, weights)         # numpy float64 (1521,), (3,) -> views of reused float64 outputs
    """

    def __init__(self, variant, x, y, z, R, mask=None, grad_mask=0xFFFF, bcutoff=BC_CUTOFF, device=None):
        if not torch.cuda.is_available():
            raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
        import numpy as np
        self.h = Handle.get(torch.cuda.current_device() if device is None else device)
        self._keep = [_col(t, nm) for t, nm in ((x, "x"), (y, "y"), (z, "z"), (R, "R"))]
        if any(t.is_cuda for t in self._keep):
            raise ValueError("HostStep is for host tensors; use loss_and_grad_raw for CUDA tensors")
        n = self._keep[0].numel()
        for t in self._keep[1:]:
            if t.dtype != self._keep[0].dtype or t.numel() != n:
                raise ValueError("x,y,z,R must share dtype and length")
        self._mask = None if mask is None else mask.detach().reshape(-1).to(torch.uint8).contiguous()
        self.sums = np.zeros(8)
        self.dtheta = np.zeros(P.N_THETA)
        vp = ctypes.c_void_p
        self._fn = self.h.L.pinn_loss_fwd_bwd_host
        self._head = (self.h.h, int({"poc": 0, "trainpy": 1}.get(variant, variant)), n) + tuple(vp(t.data_ptr()) for t in self._keep) + (
            _F64 if self._keep[0].dtype == torch.float64 else _F32, None if self._mask is None else vp(self._mask.data_ptr()))
        self._th = self._w = self._thp = self._wp = None
        self._tail = (int(grad_mask), float(bcutoff), vp(self.sums.ctypes.data), vp(self.dtheta.ctypes.data), None)

    def __call__(self, theta64, weights=None):
        """theta64: contiguous numpy float64 (1521,); weights: contiguous numpy float64 (3,) {1/n, 1/|set1|, 1/|set2|} or
        None (sets counted on the device).  Returns (sums[8], dtheta[1521]); the arrays are overwritten by the next call."""
        if theta64 is not self._th:       # `.ctypes.data` is slow; the usual caller passes the same arrays every step
            self._th, self._thp = theta64, theta64.ctypes.data
        if weights is not self._w:
            self._w, self._wp = weights, (None if weights is None else weights.ctypes.data)
        rc = self._fn(*self._head, self._thp, self._wp, *self._tail)
        if rc:
            self.h.check(rc, "pinn_loss_fwd_bwd_host")
        return self.sums, self.dtheta


_OFFS = [0, 32, 48, 304, 320, 336, 337, 369, 401, 1425, 1457, 1489, 1490, 1500, 1510, 1520, 1521]  # pinn_theta_offsets
_SIZES = [_OFFS[i + 1] - _OFFS[i] for i in range(16)]
_DT = {torch.float32: _F32, torch.float64: _F64}


def _rows(ix):
    """torch.where tuple (poc/main.py:392-393) or 1-D row indices (train.py:38-39) -> the row-index tensor"""
    return ix[0] if isinstance(ix, (tuple, list)) else ix


class _MaskCache:
    """The mask bytes of the last few (idx1, idx2) pairs.  The reference loops keep a batch - and with it the two index
    tensors - for many steps (poc/main.py:396: the last 10 % of the epochs; sc_sampling > 1), so the mask of an
    unchanged pair of index tensors (same storage, same version) is reused instead of rebuilt."""

    def __init__(self, keep=4):
        self.keep, self.items = keep, []

    def get(self, h, n, r1, r2, dev, stream):
        key = (n, dev.index, r1.data_ptr(), r1.numel(), r1._version, r2.data_ptr(), r2.numel(), r2._version)
        for k, m, _ in self.items:
            if k == key:
                return m
        n1, n2 = r1.numel(), r2.numel()
        if r1.dtype != torch.int64 or not r1.is_contiguous() or r1.device != dev:
            r1 = r1.to(device=dev, dtype=torch.int64).contiguous()
        if r2.dtype != torch.int64 or not r2.is_contiguous() or r2.device != dev:
            r2 = r2.to(device=dev, dtype=torch.int64).contiguous()
        mask = torch.empty((n + 3) // 4 * 4, dtype=torch.uint8, device=dev)
        rc = h.L.pinn_mask_from_index_sets(h.h, n, _ptr(r1) if n1 else None, n1, _ptr(r2) if n2 else None, n2, _ptr(mask),
                                           ctypes.c_void_p(stream))
        h.check(rc, "pinn_mask_from_index_sets")
        # the index tensors are kept alive with the entry: a freed tensor's address could otherwise come back with
        # different content under the same key
        self.items.insert(0, (key, mask, (r1, r2)))
        del self.items[self.keep:]
        return mask


_mask_cache = _MaskCache()


class _PinnLoss(torch.autograd.Function):
    """forward(variant, order, x, y, z, R, idx1, idx2, *16 params) -> (Ltot, Lpde, Lbc, E).

    CUDA tensors: one library call (pinn_loss_fwd_bwd_tensors) on torch's current stream.  The kernel gathers the 16
    parameter tensors through their pointers (no packing, no dtype conversion in front of the launch), takes the three
    loss weights by value, writes E in the parameters' dtype and the gradient in the parameters' layout; the only other
    device work is the mask of the two index sets (one memset + one kernel, cached while the index tensors are unchanged)
    and, in backward, one multiplication by the upstream gradient.  CPU tensors: pinn_loss_fwd_bwd_host."""

    @staticmethod
    def forward(ctx, variant, order, x, y, z, R, idx1, idx2, *params):
        if len(params) != 16:
            raise ValueError("expected the model's 16 parameter tensors")
        # (n,1) / (n,) contiguous columns are used where they lie: no slicing, no detach - only their pointers travel
        if all(t.is_contiguous() and (t.dim() == 1 or (t.dim() == 2 and t.shape[1] == 1)) and t.dtype in _DT for t in (x, y, z, R)):
            xs, ys, zs, Rs = x, y, z, R
        else:
            xs, ys, zs, Rs = _col(x, "x"), _col(y, "y"), _col(z, "z"), _col(R, "R")
        n = xs.numel()
        dev = xs.device
        pdt = params[0].dtype
        # one pass over the parameters: which want a gradient, their shapes, and whether the kernel can read them in place
        grad_mask, shapes, needs, direct = 0, [], [], dev.type == "cuda" and pdt in _DT
        for k, p in enumerate(params):
            need = p.requires_grad
            if need:
                grad_mask |= 1 << (k if order == "poc" else P.TRAINPY_TO_POC[k])
            shapes.append(p.shape)
            needs.append(need)
            if direct and not (p.dtype == pdt and p.is_cuda and p.is_contiguous()):
                direct = False
        ctx.order, ctx.shapes, ctx.needs = order, shapes, needs
        r1, r2 = _rows(idx1), _rows(idx2)
        c1, c2 = r1.numel(), r2.numel()
        # the reference takes the mean of an empty selection -> NaN loss (SURVEY 7, hard part 6): weight inf
        weights = (1.0 / n, 1.0 / c1 if c1 else float("inf"), 1.0 / c2 if c2 else float("inf"))
        if dev.type == "cuda":
            h = Handle.get(dev.index if dev.index is not None else torch.cuda.current_device())
            stream = torch.cuda.current_stream(dev).cuda_stream
            mask = _mask_cache.get(h, n, r1, r2, dev, stream)
            if ys.dtype != xs.dtype or zs.dtype != xs.dtype or Rs.dtype != xs.dtype:
                raise ValueError("x, y, z, R must share one dtype")
            out = torch.empty(8 + P.N_THETA, dtype=torch.float64, device=dev)
            E = torch.empty(n, dtype=pdt if pdt in _DT else torch.float32, device=dev)
            w = (ctypes.c_double * 3)(*weights)
            if direct:
                ptrs = (ctypes.c_void_p * 16)(*[p.data_ptr() for p in params])
                rc = h.L.pinn_loss_fwd_bwd_tensors(h.h, int(variant), n, xs.data_ptr(), ys.data_ptr(), zs.data_ptr(),
                                                   Rs.data_ptr(), _DT[xs.dtype], mask.data_ptr(), ptrs, _DT[pdt],
                                                   VARIANT_POC if order == "poc" else VARIANT_TRAINPY, w, int(grad_mask),
                                                   BC_CUTOFF, out.data_ptr(), out.data_ptr() + 64, E.data_ptr(), _DT[E.dtype],
                                                   stream)
                h.check(rc, "pinn_loss_fwd_bwd_tensors")
                ctx.native_layout = True
            else:  # mixed dtypes / non-contiguous parameters: pack first
                pack = P.pack_poc if order == "poc" else P.pack_trainpy
                theta = pack(params, dtype=torch.float32, device=dev)
                wdev = torch.tensor(weights, dtype=torch.float64, device=dev)
                E = E.float() if E.dtype != torch.float32 else E
                loss_and_grad_raw(variant, xs, ys, zs, Rs, theta, mask, wdev, grad_mask, sums=out[:8], dtheta=out[8:], E_out=E)
                ctx.native_layout = False
            sums, dtheta = out[:8], out[8:]
        else:
            mask, _, _ = indices_to_mask(n, idx1, idx2, dev)
            pack = P.pack_poc if order == "poc" else P.pack_trainpy
            theta64 = pack(params, dtype=torch.float64).contiguous()
            sums, dtheta, E = _host_step(variant, xs, ys, zs, Rs, theta64, mask, list(weights), grad_mask, True, BC_CUTOFF)
            ctx.native_layout = False
        ctx.save_for_backward(dtheta)
        Ltot, Lpde, Lbc = sums[0], sums[1], sums[2]
        if pdt != torch.float64:
            Ltot, Lpde, Lbc = Ltot.to(pdt), Lpde.to(pdt), Lbc.to(pdt)
        if E.dtype != pdt:
            E = E.to(pdt)
        E = E.view(n, 1)
        ctx.mark_non_differentiable(Lpde, Lbc, E)
        return Ltot, Lpde, Lbc, E

    @staticmethod
    def backward(ctx, gLtot, gLpde, gLbc, gE):
        (dtheta,) = ctx.saved_tensors
        g = dtheta * gLtot.to(dtheta.dtype)
        outs = [None] * 8
        if ctx.native_layout:  # tensors in canonical order, each already in the parameter's own layout: views only
            parts = g.split(_SIZES)     # one call -> 16 views
            for k, (shp, need) in enumerate(zip(ctx.shapes, ctx.needs)):
                if not need:
                    outs.append(None)
                    continue
                part = parts[k if ctx.order == "poc" else P.TRAINPY_TO_POC[k]]
                outs.append(part if len(shp) == 1 else part.view(shp))
            return tuple(outs)
        parts = P.unpack_poc(g) if ctx.order == "poc" else P.unpack_trainpy(g)
        for part, shp, need in zip(parts, ctx.shapes, ctx.needs):
            outs.append(part.reshape(shp) if need else None)
        return tuple(outs)


class PinnLossPoc:
    """Fused replacement of NN_ion.LossFunctions (poc/main.py:341-355); params in state_dict order."""

    @staticmethod
    def apply(x, y, z, R, bIndex1, bIndex2, *params):
        return _PinnLoss.apply(VARIANT_POC, "poc", x, y, z, R, bIndex1, bIndex2, *params)


class PinnLossTrainPy:
    """Fused replacement of train.py:41-57; params in train.py's tuple order/(in,out) layout (train.py:108-109)."""

    @staticmethod
    def apply(x, y, z, R, i1, i2, *params):
        return _PinnLoss.apply(VARIANT_TRAINPY, "trainpy", x, y, z, R, i1, i2, *params)


def loss_poc(model, x, y, z, R, bIndex1, bIndex2):
    """Ltot, LossPDE, Lbc, E for an ``NN_ion``-like module (16 parameters in state_dict order)."""
    # the parameter list of a module is walked once and kept with it (a module that gains or loses parameters, or is
    # moved with .to()/.double() - which replaces the Parameter objects' data in place - keeps the same objects)
    ps = model.__dict__.get("_pinn_parameters")
    if ps is None or len(ps) != 16 or next(model.parameters()) is not ps[0]:
        ps = tuple(model.parameters())
        model.__dict__["_pinn_parameters"] = ps
    return _PinnLoss.apply(VARIANT_POC, "poc", x, y, z, R, bIndex1, bIndex2, *ps)


def loss_trainpy(x, y, z, R, i1, i2, *params):
    """Ltot, Lpde, Lbc, e for train.py's 16 parameter tensors."""
    return PinnLossTrainPy.apply(x, y, z, R, i1, i2, *params)


def fields(variant, x, y, z, R, theta, want=("psi", "lap", "hpsi", "res", "E")):
    """Fused parametricPsi + hamiltonian (poc/main.py:321, 118): per-point psi, laplacian, H psi,
    residual and E as float32 CUDA tensors.  x,y,z,R: CUDA float32/float64 (n,) or (n,1); theta: packed
    parameters (any float dtype/device, converted to CUDA float32)."""
    variant = {"poc": 0, "trainpy": 1}.get(variant, variant)
    xs, ys, zs, Rs = _col(x, "x"), _col(y, "y"), _col(z, "z"), _col(R, "R")
    if not xs.is_cuda:
        if not torch.cuda.is_available():
            raise PinnError("no CUDA device: the PINN hot path has no CPU fallback")
        xs, ys, zs, Rs = (t.cuda() for t in (xs, ys, zs, Rs))
    dev = xs.device
    h = Handle.get(dev.index if dev.index is not None else torch.cuda.current_device())
    n = xs.numel()
    theta = theta.detach().to(device=dev, dtype=torch.float32).contiguous()
    out = {k: torch.empty(n, dtype=torch.float32, device=dev) for k in want}
    code = _F64 if xs.dtype == torch.float64 else _F32
    stream = torch.cuda.current_stream(dev).cuda_stream
    rc = h.L.pinn_fields(h.h, int(variant), n, _ptr(xs), _ptr(ys), _ptr(zs), _ptr(Rs), code, _ptr(theta),
                         _ptr(out.get("psi")), _ptr(out.get("lap")), _ptr(out.get("hpsi")), _ptr(out.get("res")),
                         _ptr(out.get("E")), ctypes.c_void_p(stream))
    h.check(rc, "pinn_fields")
    return out
