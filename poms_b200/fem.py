"""Solving from a source function (EXTENSION): load vectors, error norms and point evaluation on the
tensor-product B-spline spaces of a `Hierarchy` (single device, 2-D and 3-D, p = 1..5, any open knot
vectors).

    load_vector(V, knots, p, f)        b_i = int f phi_i dx              (kernel poms_quad_to_coef_3d)
    error_norms(x, knots, p, u, grad_u) ||u - u_h||_L2, |u - u_h|_H1     (kernel poms_quad_error_3d)
    evaluate(x, knots, p, points)      u_h on a tensor grid              (per-axis poms_axis_gather)

Quadrature: the (p+1)-point Gauss-Legendre rule per element and axis of `bsplines.assemble_1d_bands`, so
`load_vector` and the mass / stiffness bands of the solver integrate with the same points.

The callables f, u and grad_u receive the quadrature coordinates of a chunk of element planes along axis 1
as broadcastable fp64 device tensors, (m1, 1, 1), (1, m2, 1), (1, 1, m3) in 3-D and (m1, 1), (1, m2) in
2-D, and return the values on the chunk: a tensor of the full chunk shape or one that broadcasts to it
(grad_u: a tuple of d such tensors).  The chunk is
`plane_chunk` element planes; by default as many as keep one array of chunk values within
CHUNK_BYTES (1 GiB), so memory stays bounded at any grid size.  The contraction with the basis runs in
the kernels; the values are read in place (any row and plane pitch, unit stride along the last axis).

Slab-partitioned spaces are not supported yet (NotImplementedError).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from . import bsplines as bs
from .mg import _AxisOp, _pitch
from .stencil import DeviceContext, StencilVector, _stream

__all__ = ["load_vector", "error_norms", "evaluate", "CHUNK_BYTES"]

CHUNK_BYTES = 1 << 30


class _Axis:
    """Tables of one axis: per element (quadrature_tables), per output row for the load vector and per
    quadrature point for the error kernel; device copies on first use."""

    def __init__(self, T, p, device):
        t = bs.quadrature_tables(T, p)
        self.n, self.E, self.Q, self.K = t["n"], len(t["first"]), p + 1, p + 1
        self.first = t["first"].astype(np.int32)
        self.x, self.w, self.v, self.d = t["x"], t["w"], t["v"], t["d"]
        self._init(device)

    @classmethod
    def singleton(cls, device):
        """The middle axis of a 2-D space: one coefficient, one point, weight 1, value 1."""
        a = cls.__new__(cls)
        a.n, a.E, a.Q, a.K = 1, 1, 1, 1
        a.first = np.zeros(1, np.int32)
        a.x, a.w = np.zeros((1, 1)), np.ones((1, 1))
        a.v, a.d = np.ones((1, 1, 1)), np.zeros((1, 1, 1))
        a._init(device)
        return a

    def _init(self, device):
        K, Q, E, n = self.K, self.Q, self.E, self.n
        dev = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=device)
        # per element: weighted values b[e, k, q]
        bw = self.v * self.w[:, None, :]
        self.b_elem = dev(bw.reshape(-1))
        self.first_dev = dev(self.first, torch.int32)
        # per output row r: elements e0(r) .. e0(r)+K-1 (weights zero where an element misses r)
        e0 = np.searchsorted(self.first + K - 1, np.arange(n), side="left").astype(np.int32)
        coef = np.zeros((n, K, Q))
        for m in range(K):
            e = e0 + m
            ok = e < E
            k = np.arange(n) - self.first[np.minimum(e, E - 1)]
            ok &= (k >= 0) & (k < K)
            coef[ok, m, :] = bw[e[ok], k[ok], :]
        self.row_e0 = e0
        self.row_e0_dev = dev(e0, torch.int32)
        self.row_q0 = (e0 * Q).astype(np.int32)
        self.row_q0_dev = dev(self.row_q0, torch.int32)
        self.row_coef = dev(coef.reshape(-1))
        # per quadrature point j = e * Q + q
        self.pt_s = np.repeat(self.first, Q).astype(np.int32)
        self.pt_s_dev = dev(self.pt_s, torch.int32)
        self.pt_v = dev(np.moveaxis(self.v, 2, 1).reshape(-1))
        self.pt_d = dev(np.moveaxis(self.d, 2, 1).reshape(-1))
        self.pt_w = dev(self.w.reshape(-1))
        self.coords = dev(self.x.reshape(-1))


def _check(V, knots, p):
    if V.slab is not None and V.slab.size > 1:
        raise NotImplementedError("poms_b200.fem works on single-device spaces; slab-partitioned assembly "
                                  "and norms are not implemented")
    if V.ndim not in (2, 3):
        raise ValueError("2-D and 3-D spaces only (got %d-D)" % V.ndim)
    if not isinstance(p, (int, np.integer)) or not 1 <= p <= 5:
        raise ValueError("p must be an integer in 1..5 (got %r)" % (p,))
    if len(knots) != V.ndim:
        raise ValueError("need one knot vector per axis (%d), got %d" % (V.ndim, len(knots)))
    for a, (T, n) in enumerate(zip(knots, V.npts)):
        T = np.asarray(T, dtype=float)
        if T.ndim != 1 or len(T) != n + p + 1:
            raise ValueError("knot vector %d has %d entries; the space needs npts + p + 1 = %d"
                             % (a, len(T), n + p + 1))
        if np.any(np.diff(T) < 0):
            raise ValueError("knot vector %d is not nondecreasing" % a)


def _axes(V, knots, p):
    dev = V.device
    ax = [_Axis(np.asarray(T, dtype=float), p, dev) for T in knots]
    if V.ndim == 2:
        ax = [ax[0], _Axis.singleton(dev), ax[1]]
    return ax


def _chunk(plane_chunk, ax, arrays):
    if plane_chunk is None:
        per_plane = 8 * ax[0].Q * ax[1].E * ax[1].Q * ax[2].E * ax[2].Q
        return max(1, CHUNK_BYTES // (per_plane * max(1, arrays)))
    if int(plane_chunk) < 1:
        raise ValueError("plane_chunk must be >= 1")
    return int(plane_chunk)


def _coords(ax, d, j0, j1):
    """Broadcastable coordinate tensors of quadrature planes j0 .. j1-1 of axis 1 and all of the others."""
    c1 = ax[0].coords[j0:j1]
    if d == 2:
        return c1.view(-1, 1), ax[2].coords.view(1, -1)
    return c1.view(-1, 1, 1), ax[1].coords.view(1, -1, 1), ax[2].coords.view(1, 1, -1)


def _values(t, name, shape, device):
    """Check a callable's result; returns (tensor, row pitch, plane pitch) for the kernels."""
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s must return a torch.Tensor (got %s)" % (name, type(t).__name__))
    if t.dtype != torch.float64:
        raise ValueError("%s must return float64 values (got %s)" % (name, t.dtype))
    if t.device != device:
        raise ValueError("%s must return values on %s (got %s)" % (name, device, t.device))
    try:
        if torch.broadcast_shapes(tuple(t.shape), tuple(shape)) != tuple(shape):
            raise RuntimeError
    except RuntimeError:
        raise ValueError("%s returned shape %s; the chunk needs %s (or a shape that broadcasts to it)"
                         % (name, tuple(t.shape), tuple(shape))) from None
    t = t.expand(shape)                          # (broadcast dimensions: copied below)
    m3 = shape[-1]
    if len(shape) == 2:
        if t.stride(1) != 1 or t.stride(0) < m3:
            t = t.contiguous()
        return t, m3, t.stride(0)
    if t.stride(2) != 1 or t.stride(1) < m3 or t.stride(0) < shape[1] * t.stride(1):
        t = t.contiguous()
    return t, t.stride(1), t.stride(0)


def _geom(V):
    """(n1, n2, n3, ld, pld) of a single-device vector in the kernels' 3-D view."""
    if V.ndim == 2:
        return V.npts[0], 1, V.npts[1], V.ld, V.ld
    return V.npts[0], V.npts[1], V.npts[2], V.ld, V.npts[1] * V.ld


def load_vector(V, knots, p, f, out=None, plane_chunk=None):
    """b_i = int f phi_i dx on the space V (knot vectors `knots`, degree p) as a StencilVector.

    `out`: a vector of V to write into (e.g. `h.levels[0].ws("b")`, the right-hand side of `mg_pcg`);
    every owned entry is overwritten.  `plane_chunk`: element planes per evaluation of f (default: one
    array of chunk values within CHUNK_BYTES)."""
    _check(V, knots, p)
    ax = _axes(V, knots, p)
    d = V.ndim
    if out is None:
        out = StencilVector(V, zero=False)
    elif not V.compatible(out.space):
        raise ValueError("out is not a vector of V")
    n1, n2, n3, ld, pld = _geom(V)
    a1, a2, a3 = ax
    m2, m3 = a2.E * a2.Q, a3.E * a3.Q
    ch = _chunk(plane_chunk, ax, 1)
    dev = out._buf.device
    L = _lib.lib()
    for E0 in range(0, a1.E, ch):
        E1 = min(a1.E, E0 + ch)
        shape = ((E1 - E0) * a1.Q,) + ((m3,) if d == 2 else (m2, m3))
        F, fld, fpld = _values(f(*_coords(ax, d, E0 * a1.Q, E1 * a1.Q)), "f", shape, dev)
        store_from = 0 if E0 == 0 else int(a1.first[E0 - 1]) + a1.K
        _lib.check(L.poms_quad_to_coef_3d(
            F.data_ptr(), fld, fpld, out.flat.data_ptr(), ld, pld, n1, n2, n3, m2, m3, p, E0, E1, a1.K, a1.Q,
            a1.first_dev.data_ptr(), a1.b_elem.data_ptr(), store_from, a2.row_q0_dev.data_ptr(),
            a2.row_coef.data_ptr(), a2.K * a2.Q, a3.row_e0_dev.data_ptr(), a3.row_coef.data_ptr(), a3.E,
            a1.first.ctypes.data, a2.row_q0.ctypes.data, a3.row_e0.ctypes.data, _stream()),
            "poms_quad_to_coef_3d")
    return out


def error_norms(x, knots, p, u, grad_u=None, plane_chunk=None):
    """{"l2": ||u - u_h||_L2, "h1": |u - u_h|_H1 (None without grad_u)} for u_h = sum_i x_i phi_i, by the
    quadrature of `load_vector`; u_h is evaluated inside the kernel, chunk by chunk."""
    V = x.space
    _check(V, knots, p)
    ax = _axes(V, knots, p)
    d = V.ndim
    n1, n2, n3, ld, pld = _geom(V)
    a1, a2, a3 = ax
    m1, m2, m3 = a1.E * a1.Q, a2.E * a2.Q, a3.E * a3.Q
    dev = x._buf.device
    ch = _chunk(plane_chunk, ax, 1 + (d if grad_u is not None else 0))
    ctx = DeviceContext.get(dev)
    res = torch.zeros(2, dtype=torch.float64, device=dev)
    L = _lib.lib()
    for c, E0 in enumerate(range(0, a1.E, ch)):
        E1 = min(a1.E, E0 + ch)
        j0, j1 = E0 * a1.Q, E1 * a1.Q
        shape = (j1 - j0,) + ((m3,) if d == 2 else (m2, m3))
        xs = _coords(ax, d, j0, j1)
        keep = [_values(u(*xs), "u", shape, dev)]
        if grad_u is not None:
            g = grad_u(*xs)
            if not isinstance(g, (tuple, list)) or len(g) != d:
                raise ValueError("grad_u must return a tuple of %d tensors" % d)
            keep += [_values(t, "grad_u[%d]" % i, shape, dev) for i, t in enumerate(g)]
        comps = keep if d == 3 or grad_u is None else [keep[0], keep[1], None, keep[2]]
        comps = list(comps) + [None] * (4 - len(comps))
        ref = (C.c_void_p * 4)(*[t[0].data_ptr() if t is not None else None for t in comps])
        rld = (C.c_int64 * 4)(*[t[1] if t is not None else 0 for t in comps])
        rpld = (C.c_int64 * 4)(*[t[2] if t is not None else 0 for t in comps])
        _lib.check(L.poms_quad_error_3d(
            x.flat.data_ptr(), ld, pld, n1, n2, n3, m2, m3, p, ref, rld, rpld, j0, j1 - j0,
            a1.K, a1.pt_s_dev.data_ptr(), a1.pt_v.data_ptr(), a1.pt_d.data_ptr(), a1.pt_w.data_ptr(),
            a2.K, a2.pt_s_dev.data_ptr(), a2.pt_v.data_ptr(), a2.pt_d.data_ptr(), a2.pt_w.data_ptr(),
            a3.pt_s_dev.data_ptr(), a3.pt_v.data_ptr(), a3.pt_d.data_ptr(), a3.pt_w.data_ptr(),
            a1.pt_s.ctypes.data, a2.pt_s.ctypes.data, a3.pt_s.ctypes.data, m1,
            int(grad_u is not None), int(c > 0), res.data_ptr(), ctx.ws_ptr, _stream()),
            "poms_quad_error_3d")
        del keep
    sq = res.cpu().numpy()
    return {"l2": float(np.sqrt(max(sq[0], 0.0))),
            "h1": float(np.sqrt(max(sq[1], 0.0))) if grad_u is not None else None}


def evaluate(x, knots, p, points):
    """u_h = sum_i x_i phi_i on the tensor grid points[0] x .. x points[d-1] (1-D arrays inside the
    knot range), as a (len(points[0]), ..) fp64 device tensor: one row-compressed gather per axis,
    rows of width p+1."""
    V = x.space
    _check(V, knots, p)
    if len(points) != V.ndim:
        raise ValueError("need one array of points per axis")
    dev = x._buf.device
    ops = []
    for T, n, pts in zip(knots, V.npts, points):
        T = np.asarray(T, dtype=float)
        pts = np.asarray(pts, dtype=float).reshape(-1)
        if len(pts) == 0 or pts.min() < T[p] or pts.max() > T[n]:
            raise ValueError("points must lie in [%g, %g]" % (T[p], T[n]))
        spans = np.clip(np.searchsorted(T, pts, side="right") - 1, p, n - 1)
        vals, _ = bs._all_basis(T, p, spans, pts[:, None])
        ops.append(_AxisOp((spans - p).astype(np.int32), vals[:, :, 0], n, dev))
    shape = list(V.npts)
    src, ld = x.flat, V.ld
    for axis, op in enumerate(ops):
        last = axis == len(ops) - 1
        ld_out = _pitch(op.n_out) if last else ld
        out_shape = shape[:axis] + [op.n_out] + shape[axis + 1:]
        dst = torch.zeros(out_shape[:-1] + [ld_out], dtype=torch.float64, device=dev)
        op.apply(src, dst, tuple(shape), ld, ld_out, axis)
        src, shape = dst, out_shape
    return src[..., :shape[-1]]

