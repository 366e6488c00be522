"""Solving from a source function (EXTENSION): load vectors, error norms and point evaluation on the
tensor-product B-spline spaces of a `Hierarchy` (single device, 2-D and 3-D, p = 1..5, any open knot
vectors).

    load_vector(V, knots, p, f)        b_i = int f phi_i dx              (kernel poms_quad_to_coef_3d)
    boundary_load(V, knots, p, g, a, s) b_i += int_F g phi_i ds on a face (kernel poms_quad_to_coef_3d)
    error_norms(x, knots, p, u, grad_u) ||u - u_h||_L2, |u - u_h|_H1     (kernel poms_quad_error_3d)
    evaluate(x, knots, p, points)      u_h on a tensor grid              (per-axis poms_axis_gather)
    evaluate_points(x, knots, p, P)    u_h (and grad u_h) at points P    (kernel poms_points_eval)
    deposit(V, knots, p, P, w)         b_i = sum_k w_k phi_i(P_k)        (poms_points_locate, a stable sort,
                                                                          poms_points_moments / _assemble)

Quadrature: the (p+1)-point Gauss-Legendre rule per element and axis of `bsplines.assemble_1d_bands`, so
`load_vector` and the mass / stiffness bands of the solver integrate with the same points.

The callables f, u and grad_u receive the quadrature coordinates of a chunk of element planes along axis 1
as broadcastable fp64 device tensors, (m1, 1, 1), (1, m2, 1), (1, 1, m3) in 3-D and (m1, 1), (1, m2) in
2-D, and return the values on the chunk: a tensor of the full chunk shape or one that broadcasts to it
(grad_u: a tuple of d such tensors).  The chunk is
`plane_chunk` element planes; by default as many as keep one array of chunk values within
CHUNK_BYTES (1 GiB), so memory stays bounded at any grid size.  The contraction with the basis runs in
the kernels; the values are read in place (any row and plane pitch, unit stride along the last axis).

Particle coupling (evaluate_points, deposit): `points` is an (m, d) fp64 tensor on the space's device, each
coordinate inside [T_a[p], T_a[n_a]].  A point belongs to the knot span T[k] <= x < T[k+1], a point at T[n]
to the last non-empty span (scipy's BSpline and `evaluate` do the same), so on a breakpoint a derivative is
the right-hand one.

Boundary data (boundary_load): with `Hierarchy(..., c=c, robin=...)` the solver's operator is the weak form
of -Lap u + c u = f with du/dn + alpha u = g on every face (alpha = 0: Neumann).  The right-hand side is
`load_vector` for f plus one `boundary_load` per face where g is not zero.

Slab-partitioned spaces are not supported yet (NotImplementedError).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from . import bsplines as bs
from .mg import _AxisOp, _pitch
from .stencil import DeviceContext, StencilVector, _stream

__all__ = ["load_vector", "boundary_load", "error_norms", "evaluate", "evaluate_points", "deposit", "CHUNK_BYTES"]

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
    if len(shape) == 1:
        t = t.contiguous()
        return t, m3, m3
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


def boundary_load(V, knots, p, g, axis, side, out=None, plane_chunk=None):
    """b_i += int_F g phi_i ds on the face F = {x_axis = T_axis[p]} (side 0) or {x_axis = T_axis[n]}
    (side 1): the boundary data of a Neumann condition du/dn = g or a Robin condition du/dn + alpha u = g
    (with `Hierarchy(..., robin=...)`), for the weak form of -Lap u + c u = f.

    `g` receives the quadrature coordinates of the d-1 face axes (increasing axis order, the fixed
    coordinate omitted) like `load_vector`'s f: (m1, 1), (1, m2) on a 3-D face, one (m,) tensor on a 2-D
    face.  On an open knot vector only the first (side 0) or last (side 1) basis function along `axis` is
    non-zero on F, with value 1, so the result is a (d-1)-dimensional load vector in that coefficient
    plane; every other entry is left alone.  `out=None`: a new zero vector with the face contribution
    only; `out` given: added into it, so `load_vector` followed by one call per face with data gives the
    whole right-hand side.  `plane_chunk`: element planes along the first face axis per evaluation of g
    (3-D; a 2-D face is one piece).

    The contraction runs in `poms_quad_to_coef_3d` with a singleton middle axis (the layout of a 2-D
    load vector), rows added, never stored.  A face normal to one of the leading axes is written in
    place: its coefficient plane has unit stride along the last axis.  A face normal to the last
    (contiguous) axis has none, so it is contracted into a contiguous scratch plane (line in 2-D) and
    added to the strided face plane: O(N^(d-1)) work and memory.  Deterministic."""
    _check(V, knots, p)
    d = V.ndim
    if isinstance(axis, bool) or not isinstance(axis, (int, np.integer)) or not 0 <= axis < d:
        raise ValueError("axis must be an integer in 0..%d (got %r)" % (d - 1, axis))
    if isinstance(side, bool) or side not in (0, 1):
        raise ValueError("side must be 0 (x = T[p]) or 1 (x = T[n]) (got %r)" % (side,))
    T = np.asarray(knots[axis], dtype=float)
    n = V.npts[axis]
    end = T[:p + 1] if side == 0 else T[n:]
    if np.any(end != end[0]):
        raise ValueError("knot vector %d is not open at side %d: the face term needs p + 1 equal end knots"
                         % (axis, side))
    if plane_chunk is not None and int(plane_chunk) < 1:
        raise ValueError("plane_chunk must be >= 1")
    if out is None:
        out = StencilVector(V)
    elif not V.compatible(out.space):
        raise ValueError("out is not a vector of V")
    dev = out._buf.device
    j = 0 if side == 0 else n - 1
    face = [b for b in range(d) if b != axis]
    single = _Axis.singleton(dev)
    a3 = _Axis(np.asarray(knots[face[-1]], dtype=float), p, dev)
    a1 = _Axis(np.asarray(knots[face[0]], dtype=float), p, dev) if d == 3 else single
    ax = [a1, single, a3]
    n1, n3 = a1.n, a3.n
    if axis == d - 1:
        # the face plane is strided along every axis: contract into a contiguous scratch plane
        ld_s = _pitch(n3)
        scratch = torch.zeros((n1, ld_s), dtype=torch.float64, device=dev)
        y, ld, pld = scratch.data_ptr(), ld_s, ld_s
    elif d == 2:                                                    # row j of the 2-D array
        y, ld, pld = out.flat[j].data_ptr(), V.ld, V.ld
    elif axis == 0:                                                 # plane j: rows along axis 1
        y, ld, pld = out.flat[j].data_ptr(), V.ld, V.ld
    else:                                                           # out[:, j, :]: rows along axis 0
        y, ld, pld = out.flat[:, j].data_ptr(), V.ld, V.npts[1] * V.ld
    m3 = a3.E * a3.Q
    ch = _chunk(plane_chunk, ax, 1)
    L = _lib.lib()
    for E0 in range(0, a1.E, ch):
        E1 = min(a1.E, E0 + ch)
        if d == 2:
            F, fld, fpld = _values(g(a3.coords), "g", (m3,), dev)
        else:
            xs = (a1.coords[E0 * a1.Q:E1 * a1.Q].view(-1, 1), a3.coords.view(1, -1))
            F, fld, fpld = _values(g(*xs), "g", ((E1 - E0) * a1.Q, m3), dev)
        _lib.check(L.poms_quad_to_coef_3d(
            F.data_ptr(), fld, fpld, y, ld, pld, n1, 1, n3, 1, m3, p, E0, E1, a1.K, a1.Q,
            a1.first_dev.data_ptr(), a1.b_elem.data_ptr(), n1, single.row_q0_dev.data_ptr(),
            single.row_coef.data_ptr(), 1, a3.row_e0_dev.data_ptr(), a3.row_coef.data_ptr(), a3.E,
            a1.first.ctypes.data, single.row_q0.ctypes.data, a3.row_e0.ctypes.data, _stream()),
            "poms_quad_to_coef_3d")
    if axis == d - 1:
        out.flat[..., j].add_(scratch[:, :n3].reshape(out.flat[..., j].shape))
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


def _points(knots, p, d, dev, points, weights=None):
    """Check the points (and weights) of `evaluate_points` / `deposit` against a d-dimensional space whose
    storage is on `dev`; returns (points, weights, knot tensor, per-axis knot pointers of the kernels' 3-D
    view).  The range and finiteness check reads one flag from the device."""
    if not isinstance(points, torch.Tensor) or points.dtype != torch.float64:
        raise ValueError("points must be a float64 torch.Tensor")
    if points.device != dev:
        raise ValueError("points must be on %s (got %s)" % (dev, points.device))
    if points.ndim != 2 or points.shape[1] != d:
        raise ValueError("points must have shape (m, %d) (got %s)" % (d, tuple(points.shape)))
    m = points.shape[0]
    if m >= 1 << 31:
        raise ValueError("at most 2^31 - 1 points per call (got %d)" % m)
    if weights is not None:
        if not isinstance(weights, torch.Tensor) or weights.dtype != torch.float64:
            raise ValueError("weights must be a float64 torch.Tensor")
        if weights.device != dev:
            raise ValueError("weights must be on %s (got %s)" % (dev, weights.device))
        if tuple(weights.shape) != (m,):
            raise ValueError("weights must have shape (%d,) (got %s)" % (m, tuple(weights.shape)))
        weights = weights.contiguous()
    Ts = [np.asarray(T, dtype=float) for T in knots]
    lo = torch.tensor([T[p] for T in Ts], dtype=torch.float64, device=dev)
    hi = torch.tensor([T[len(T) - p - 1] for T in Ts], dtype=torch.float64, device=dev)
    points = points.contiguous()
    if m and not bool(((points >= lo) & (points <= hi)).all()):        # NaN and inf fail both comparisons
        bad = ~((points >= lo) & (points <= hi))
        k, a = (int(v) for v in bad.nonzero()[0])
        raise ValueError("point %d has coordinate %r on axis %d; points must be finite and inside [%r, %r]"
                         % (k, float(points[k, a]), a, float(lo[a]), float(hi[a])))
    Tdev = torch.as_tensor(np.concatenate(Ts), dtype=torch.float64, device=dev)
    offs = np.concatenate([[0], np.cumsum([len(T) for T in Ts])])
    ptrs = [Tdev.data_ptr() + 8 * int(o) for o in offs[:-1]]
    if d == 2:
        ptrs = [ptrs[0], None, ptrs[1]]
    return points, weights, Tdev, ptrs


def evaluate_points(x, knots, p, points, grad=False):
    """u_h = sum_i x_i phi_i at the rows of `points` ((m, d) fp64 on the device of x), as an (m,) tensor;
    with grad=True, (u, g) with g[k] = grad u_h(points[k]), (m, d).  One thread per point: binary search
    of each knot vector, the degree-p basis with first derivatives in registers, a gather of the (p+1)^d
    coefficients.  Deterministic.  Raises ValueError for a wrong dtype, device or shape, a non-finite
    coordinate or one outside [T_a[p], T_a[n_a]], and m >= 2^31; that check costs one device-to-host read."""
    V = x.space
    _check(V, knots, p)
    d, dev = V.ndim, x._buf.device
    points, _, Tdev, T = _points(knots, p, d, dev, points)
    m = points.shape[0]
    u = torch.empty(m, dtype=torch.float64, device=dev)
    g = torch.empty((m, d), dtype=torch.float64, device=dev) if grad else None
    if m:
        n1, n2, n3, ld, pld = _geom(V)
        _lib.check(_lib.lib().poms_points_eval(
            x.flat.data_ptr(), ld, pld, n1, n2, n3, p, T[0], T[1], T[2], points.data_ptr(), d, m, u.data_ptr(),
            g.data_ptr() if grad else None, _stream()), "poms_points_eval")
    return (u, g) if grad else u


def deposit(V, knots, p, points, weights, out=None, plane_chunk=None):
    """b_i = sum_k weights[k] phi_i(points[k]) on the space V as a StencilVector (`out`: a vector of V whose
    owned entries are all overwritten).  Point charges, a Monte-Carlo source or measurements as a
    right-hand side; the adjoint of `evaluate_points`.

    Deterministic (bit-identical on repeated calls) and free of atomics: a kernel gives every point its cell
    (knot span per axis) as an int64 key, a stable torch.sort orders the points by cell, one warp per cell
    sums the (p+1)^d basis products of its points in that order, and an output-centric kernel adds the
    moments of the <= (p+1)^d cells of each coefficient in a fixed order.  Scratch: 16 B per point for the
    sorted keys and the permutation (24 B while the sort runs), plus the moments of one chunk of
    `plane_chunk` cell planes along axis 1, 8 (p+1)^d B per cell (default: as many planes as keep them
    within CHUNK_BYTES).  Raises ValueError like `evaluate_points` (also for weights of the wrong dtype,
    device or shape), with the same one device-to-host read."""
    _check(V, knots, p)
    if plane_chunk is not None and int(plane_chunk) < 1:
        raise ValueError("plane_chunk must be >= 1")
    if out is not None and not V.compatible(out.space):
        raise ValueError("out is not a vector of V")
    d = V.ndim
    dev = out._buf.device if out is not None else torch.empty(0, device=V.device).device
    points, weights, Tdev, T = _points(knots, p, d, dev, points, weights)
    m = points.shape[0]
    if out is None:
        out = StencilVector(V, zero=False)
    if m == 0:
        out.data.zero_()
        return out
    n1, n2, n3, ld, pld = _geom(V)
    C1, C2, C3 = n1 - p, (n2 - p if d == 3 else 1), n3 - p
    nt = (p + 1) ** d
    L = _lib.lib()
    key = torch.empty(m, dtype=torch.int64, device=dev)
    _lib.check(L.poms_points_locate(points.data_ptr(), d, m, n1, n2, n3, p, T[0], T[1], T[2], key.data_ptr(),
                                    _stream()), "poms_points_locate")
    skey, perm = torch.sort(key, stable=True)
    del key
    ch = int(plane_chunk) if plane_chunk is not None else max(1, CHUNK_BYTES // (8 * C2 * C3 * nt))
    ch = min(ch, C1)
    mom = torch.empty(ch * C2 * C3 * nt, dtype=torch.float64, device=dev)
    for c0 in range(0, C1, ch):
        c1 = min(C1, c0 + ch)
        cells = torch.arange(c0 * C2 * C3, c1 * C2 * C3 + 1, dtype=torch.int64, device=dev)
        offs = torch.searchsorted(skey, cells)
        _lib.check(L.poms_points_moments(points.data_ptr(), weights.data_ptr(), d, perm.data_ptr(),
                                         offs.data_ptr(), c0, c1, n1, n2, n3, p, T[0], T[1], T[2],
                                         mom.data_ptr(), _stream()), "poms_points_moments")
        _lib.check(L.poms_points_assemble(mom.data_ptr(), c0, c1, n1, n2, n3, p, out.flat.data_ptr(), ld, pld,
                                          0 if c0 == 0 else c0 + p, _stream()), "poms_points_assemble")
    return out
