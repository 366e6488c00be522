"""Grid transfer, two-grid cycle and the multi-level V-cycle / MG-preconditioned CG.

Reference-faithful parts (SURVEY.md section 8a, a13-a17):
  * `Transfer`: restriction r_c = (P1^T (x) P1^T) r_f and prolongation e_f = (P1 (x) P1) e_c of
    /root/reference/sources/mg_jac.py:67-70,94,102, applied one axis at a time with
    row-compressed knot-insertion matrices (never forming the Kronecker matrix);
  * `CoarseSolver`: the replicated direct coarse solve of mg_jac.py:98-99.  The Galerkin operator
    R*Af*P of a nested spline space is the coarse-space Kronecker sum, which is inverted exactly by
    fast diagonalisation (dense 1-D generalised eigenbases, three small contractions);
  * `two_grid`: one two-grid cycle in the exact order of mg_jac.py:85-119 / mg_glt.py:84-123.

EXTENSION beyond the reference (SURVEY.md section 8f-1; labelled in every report):
  * `Hierarchy`, `vcycle`, `mg_pcg`: recursive V-cycle used as the preconditioner of the
    reference's own `pcg` driver; `mg_gmres`: the same V-cycle preconditioning GMRES for the
    non-symmetric convection-diffusion operator (`Hierarchy(beta=)`).  Smoothers are the LINEAR,
    symmetric counterparts of the reference's PCG smoothers -- a Chebyshev iteration preconditioned
    by damped-Jacobi's D^-1 ("jacobi") or by the GLT Kronecker solve T[m_{p-1}] (x) .. (x) T[m_{p-1}] ("glt",
    /root/reference/slides/content.tex:141-153) -- because a fixed SPD preconditioner is what CG
    needs (the reference's omega = 2/3 Jacobi diverges for p >= 3, see DESIGN.md).
"""
import os
from math import sqrt

import numpy as np
import torch

from . import _lib
from . import bsplines as bs
from . import profiling
from .multilevels import knots_to_insert
from .stencil import (StencilVectorSpace, StencilVector, KronSumMatrix, DeviceContext,
                      _stream, EPI_STORE, EPI_RESID, EPI_DINV, EPI_AXPY, reaction_robin, convection_beta)
from .kron_product import BandLU, kron_solve_bnd, kron_solve_bnd_update
from . import solvers

__all__ = ["Transfer", "DistTransfer", "CoarseSolver", "two_grid", "Hierarchy", "vcycle", "mg_pcg",
           "mg_gmres", "fine_knots"]


def fine_knots(Tc, ts):
    """Sorted union of the coarse knots and the inserted ones (mg_jac.py:32-35)."""
    return np.sort(np.concatenate([np.asarray(Tc, float), np.asarray(ts, float)]), kind="stable")


def _dense_mode():
    """How dense per-axis contractions (eigenbases of the coarse solve) are applied: 'dmma' = fp64
    tensor-core kernel poms_axis_dense_dmma (default; measured against the gather kernel in
    profiles/r02_ab_dense_dmma_vs_gather.txt), 'gather' = poms_axis_gather with W = n."""
    import os
    return os.environ.get("POMS_B200_DENSE", "dmma")


def _gather(src_ptr, dst_ptr, start, coef, n_in, n_out, n_outer, so_in, sa_in, so_out, sa_out,
            n_inner, accumulate, dense=False):
    if dense and not accumulate and _dense_mode() == "dmma":
        _lib.check(_lib.lib().poms_axis_dense_dmma(
            src_ptr, dst_ptr, coef.data_ptr(), n_in, n_out, n_outer, so_in, sa_in, so_out, sa_out,
            n_inner, _stream()), "poms_axis_dense_dmma")
        return
    _lib.check(_lib.lib().poms_axis_gather(
        src_ptr, dst_ptr, start.data_ptr(), coef.data_ptr(), coef.shape[1], n_in, n_out, n_outer,
        so_in, sa_in, so_out, sa_out, n_inner, int(accumulate), _stream()), "poms_axis_gather")


class _AxisOp:
    """Row-compressed sparse matrix applied along one axis of a contiguous d-dim array."""

    def __init__(self, start, coef, n_in, device, dense=False):
        self.n_out, self.W = coef.shape
        self.n_in = int(n_in)
        self.dense = bool(dense) and self.W == self.n_in and not np.any(start)
        self._start_host = np.ascontiguousarray(start, dtype=np.int32)
        self.start = torch.as_tensor(self._start_host, device=device)
        self.coef = torch.as_tensor(np.ascontiguousarray(coef, dtype=np.float64), device=device)

    @property
    def start_host(self):
        return self._start_host

    def apply(self, src, dst, shape_in, ld_in, ld_out, axis, accumulate=False):
        """dst = op along `axis` of src.  src/dst are pitched arrays: logical shape `shape_in`
        (resp. with n_out along `axis`), last-dimension pitch ld_in / ld_out, pad columns zero."""
        nd = len(shape_in)
        shape_out = list(shape_in)
        shape_out[axis] = self.n_out
        if axis == nd - 1:
            n_outer = int(np.prod(shape_in[:-1])) if nd > 1 else 1
            so_in, so_out, sa_in, sa_out, n_inner = ld_in, ld_out, 1, 1, 1
        elif axis == 0:
            assert ld_in == ld_out
            rest = int(np.prod(shape_in[1:-1])) * ld_in
            n_outer, so_in, so_out, sa_in, sa_out, n_inner = 1, 0, 0, rest, rest, rest
        else:
            assert ld_in == ld_out
            n_outer = shape_in[0]
            so_in, so_out = shape_in[1] * ld_in, self.n_out * ld_in
            sa_in = sa_out = n_inner = ld_in
        _gather(src.data_ptr(), dst.data_ptr(), self.start, self.coef, self.n_in, self.n_out,
                n_outer, so_in, sa_in, so_out, sa_out, n_inner, accumulate, dense=self.dense)
        return tuple(shape_out)


def _pitch(n):
    return n + (n & 1)


def transfer_v2_min():
    """Fine points per rank from which a transfer uses the round-2 one-pass kernels
    (poms_transfer3d_v2.cu), per operation; None = never.  Measured at p = 3
    (profiles/r02_ab_transfer_v2.txt), 515^3 / 259^3 / 131^3 fine points:
      restriction  0.456 / 0.082 / 0.051 ms  (three per-axis gathers 0.63 / 0.109 / 0.080, round-1
                                              one-pass kernel 0.77 / 0.142 / 0.052)
      prolongation 0.72 / 0.128 / 0.028 ms   (gathers 0.96 / 0.150 / 0.054, round 1 1.41 / 0.209 / 0.044)
    POMS_B200_TRANSFER_V2=0 switches them off (round-2 behaviour before these kernels), =prolong
    keeps the restriction on the gathers; POMS_B200_TRANSFER_V2_MIN=n sets both thresholds (the
    multi-GPU parity script runs a second time with 0, so that its small grids take these kernels)."""
    mode = os.environ.get("POMS_B200_TRANSFER_V2", "all")
    if mode == "0":
        return {"restrict": None, "prolong": None}
    force = os.environ.get("POMS_B200_TRANSFER_V2_MIN")      # tests: one threshold for both
    lo_r, lo_p = (int(force), int(force)) if force is not None else (6_000_000, 1_000_000)
    return {"restrict": None if mode == "prolong" else lo_r, "prolong": lo_p}


def _fused_restrict(ops, fine, shape_f, ld_f, coarse, shape_c, ld_c, v2=False):
    """coarse = (R1 (x) R2 (x) R3) fine in one kernel; False if the rows do not fit its tiles."""
    r1, r2, r3 = ops
    fn = _lib.lib().poms_restrict_3d_v2 if v2 else _lib.lib().poms_restrict_3d
    rc = fn(
        fine.data_ptr(), coarse.data_ptr(), shape_f[0], shape_f[1], shape_f[2], ld_f,
        shape_f[1] * ld_f, shape_c[0], shape_c[1], shape_c[2], ld_c, shape_c[1] * ld_c,
        r1.start.data_ptr(), r1.coef.data_ptr(), r1.W, r2.start.data_ptr(), r2.coef.data_ptr(), r2.W,
        r3.start.data_ptr(), r3.coef.data_ptr(), r3.W, r1.start_host.ctypes.data,
        r2.start_host.ctypes.data, r3.start_host.ctypes.data, _stream())
    if rc < 0:
        return False
    _lib.check(rc, "poms_restrict_3d")
    return True


def _fused_prolong(ops, coarse, shape_c, ld_c, fine, shape_f, ld_f, accumulate, v2=False):
    """fine (+)= (P1 (x) P2 (x) P3) coarse in one kernel; False if the rows do not fit its tiles."""
    p1, p2, p3 = ops
    fn = _lib.lib().poms_prolong_3d_v2 if v2 else _lib.lib().poms_prolong_3d
    rc = fn(
        coarse.data_ptr(), fine.data_ptr(), shape_f[0], shape_f[1], shape_f[2], ld_f,
        shape_f[1] * ld_f, shape_c[0], shape_c[1], shape_c[2], ld_c, shape_c[1] * ld_c,
        p1.start.data_ptr(), p1.coef.data_ptr(), p1.W, p2.start.data_ptr(), p2.coef.data_ptr(), p2.W,
        p3.start.data_ptr(), p3.coef.data_ptr(), p3.W, p2.start_host.ctypes.data,
        p3.start_host.ctypes.data, int(accumulate), _stream())
    if rc < 0:
        return False
    _lib.check(rc, "poms_prolong_3d")
    return True


def _tmp(shape, ld, device, zero=True):
    """Pitched temporary.  zero=False when the producing kernel writes the pad column too (every
    pass along a non-contiguous axis does: it maps the zero pad of its input)."""
    alloc = torch.zeros if zero else torch.empty
    return alloc(tuple(shape[:-1]) + (ld,), dtype=torch.float64, device=device)


class Transfer:
    """Per-axis knot-insertion transfer between a fine and a coarse tensor-product space."""

    def __init__(self, Tc_axes, Tf_axes, p, device):
        self.ndim = len(Tc_axes)
        self.P, self.R = [], []
        self.P1_rows = []
        for Tc, Tf in zip(Tc_axes, Tf_axes):
            nf = len(Tf) - p - 1
            nc = len(Tc) - p - 1
            if nf == nc:
                self.P.append(None)
                self.R.append(None)
                self.P1_rows.append(None)
                continue
            from . import setup_device as sd
            rows = sd.knot_insertion_rows if sd.enabled() else bs.knot_insertion_rows
            st, cf, _ = rows(Tc, Tf, p)
            stt, cft = bs.rows_transpose(st, cf, nc)
            self.P.append(_AxisOp(st, cf, nc, device))
            self.R.append(_AxisOp(stt, cft, nf, device))
            self.P1_rows.append((st, cf, nc))
        self.device = device
        # 3-D with every axis refined: one fused kernel per transfer instead of three gathers, on the
        # levels where launch latency dominates (measured at p = 3, tests/gpu_ab_transfer.py: fused
        # 0.045 / 0.044 ms vs 0.085 / 0.073 ms at 131^3, but 0.77 / 1.41 ms vs 0.61 / 1.01 ms at 515^3,
        # where the three streaming passes run closer to the HBM rate than the fused tile pipeline)
        self.fused = self.ndim == 3 and all(op is not None for op in self.P)
        self.fused_max = 6_000_000      # fine points per rank up to which the round-1 fused kernels are used
        # round-2 one-pass kernels (poms_transfer3d_v2.cu; tests/gpu_ab_transfer.py): thresholds per
        # operation (a dict, or one number for both)
        self.v2_min = transfer_v2_min()
        self.fused_v2 = self.fused
        self._tmps = {}

    def _want_fused(self, shape_f, op):
        """None (per-axis gathers), "v1" (round-1 one-pass kernels) or "v2" (round-2 kernels) for
        `op` = "restrict" / "prolong" on a fine grid of this shape."""
        n = int(np.prod(shape_f))
        v2_min = self.v2_min.get(op) if isinstance(self.v2_min, dict) else self.v2_min
        if self.fused_v2 and v2_min is not None and n >= v2_min:
            return "v2"
        if self.fused and n <= self.fused_max:
            return "v1"
        return None

    def _fused_failed(self, kind):
        if kind == "v2":
            self.fused_v2 = False
        else:
            self.fused = False

    def _tmp(self, key, shape, ld):
        """Intermediate array of a per-axis pass, allocated (and zeroed: pad column) once per
        transfer object and reused by every later application."""
        k = (key, tuple(shape), ld)
        t = self._tmps.get(k)
        if t is None:
            t = self._tmps[k] = _tmp(shape, ld, self.device, zero=True)
        return t

    def restrict(self, rf, Vc, out=None):
        """r_c = (P1^T (x) .. (x) P1^T) r_f.  Axis 1 first: the largest array is read once,
        fully coalesced, and every later pass works on a smaller one.  `out`: vector of Vc that
        receives the result (its pad column must be zero), default a new one."""
        assert rf.space.slab is None or rf.space.slab.size == 1, "use DistTransfer for slabs"
        rc = StencilVector(Vc) if out is None else out
        cur, ld = rf.flat, rf.ld
        shape = tuple(rf.space.local_shape)
        kind = self._want_fused(shape, "restrict")
        if kind:
            if _fused_restrict(self.R, cur, shape, ld, rc.flat, tuple(Vc.local_shape), rc.ld,
                               v2=(kind == "v2")):
                return rc
            self._fused_failed(kind)
        ops = [(ax, op) for ax, op in enumerate(self.R) if op is not None]
        if not ops:
            rc.flat.copy_(cur)
            return rc
        nd = len(shape)
        for n, (ax, op) in enumerate(ops):
            shape_out = list(shape)
            shape_out[ax] = op.n_out
            last = n == len(ops) - 1
            ld_out = _pitch(op.n_out) if ax == nd - 1 else ld
            dst = rc.flat if last else self._tmp(("R", n), shape_out, ld_out)
            if last:
                assert ld_out == rc.ld
            shape = op.apply(cur, dst, shape, ld, ld_out, ax)
            cur, ld = dst, ld_out
        return rc

    def prolong_add(self, ec, xf):
        """x_f += (P1 (x) .. (x) P1) e_c.  Last axis first (small arrays); the final, largest
        pass along axis 1 accumulates straight into x_f (correction fused, mg_jac.py:112)."""
        cur, ld = ec.flat, ec.ld
        shape = tuple(ec.space.local_shape)
        kind = self._want_fused(xf.space.local_shape, "prolong")
        if kind:
            if _fused_prolong(self.P, cur, shape, ld, xf.flat, tuple(xf.space.local_shape), xf.ld,
                              True, v2=(kind == "v2")):
                return xf
            self._fused_failed(kind)
        ops = [(ax, op) for ax, op in reversed(list(enumerate(self.P))) if op is not None]
        if not ops:
            xf.flat.add_(cur)
            return xf
        nd = len(shape)
        for n, (ax, op) in enumerate(ops):
            shape_out = list(shape)
            shape_out[ax] = op.n_out
            last = n == len(ops) - 1
            ld_out = _pitch(op.n_out) if ax == nd - 1 else ld
            dst = xf.flat if last else self._tmp(("P", n), shape_out, ld_out)
            if last:
                assert ld_out == xf.ld
            shape = op.apply(cur, dst, shape, ld, ld_out, ax, accumulate=last)
            cur, ld = dst, ld_out
        return xf


class DistTransfer(Transfer):
    """Transfer whose FINE space is slab-partitioned along axis 1.  The coarse space is either
    partitioned too, or replicated on every rank (the level where the hierarchy is gathered: the
    analogue of `rc = comm.allreduce(rc)`, /root/reference/sources/mg_jac.py:95).

    Axis-1 passes work on plane blocks: the few fine (restriction) or coarse (prolongation) planes
    that belong to a neighbour are fetched with one send/recv pair; axes 2..d are local."""

    def __init__(self, Tc_axes, Tf_axes, p, device, slab, coarse_distributed):
        from .dist import slab_transfer_plan
        super().__init__(Tc_axes, Tf_axes, p, device)
        self.slab = slab
        self.cdist = coarse_distributed
        assert self.P[0] is not None, "the partitioned axis must be refined between levels"
        st, cf, nc = self.P1_rows[0]
        plan = slab_transfer_plan(st, cf, nc, slab.size, coarse_distributed)
        r = slab.rank
        self.tf, self.tc = plan["tf"], plan["tc"]
        self.need_f, self.need_c = plan["need_f"], plan["need_c"]
        self.R0 = _AxisOp(plan["R0"][r][0], plan["R0"][r][1], plan["R0"][r][2], device)
        self.P0 = _AxisOp(plan["P0"][r][0], plan["P0"][r][1], plan["P0"][r][2], device)

    def _ghost_view(self, v, table, need):
        """Planes need[rank] of `v` as a VIEW of its storage after a halo exchange (no copy), or
        None when they reach beyond the ghost planes."""
        from .dist import ghost_view_range
        V = v.space
        if V.slab is None:
            return None
        rng = ghost_view_range(table, need, self.slab.rank, V.pads[0], V.glo, V.local_shape[0])
        if rng is None:
            return None
        self.slab.exchange(v)
        return v._buf[rng[0]:rng[1]]

    def restrict(self, rf, Vc, out=None):
        slab = self.slab
        nd = len(rf.space.local_shape)
        ld = rf.ld
        cs, ce = self.tc[slab.rank]
        # the neighbours' fine planes through the ghost planes (a view: no copy of the slab);
        # gathered into a new array only when they reach beyond the ghosts
        planes = self._ghost_view(rf, self.tf, self.need_f)
        if planes is None:
            planes = slab.gather_planes(rf.flat, self.tf, self.need_f)
        shape_f = (planes.shape[0],) + tuple(rf.space.local_shape[1:])
        kind = self._want_fused(shape_f, "restrict")
        if kind:
            rc = StencilVector(Vc) if out is None else out
            shape_c = (ce - cs + 1,) + tuple(Vc.local_shape[1:])
            dst = rc.flat if self.cdist else _tmp(shape_c, rc.ld, self.device)
            if _fused_restrict((self.R0, self.R[1], self.R[2]), planes, shape_f, ld, dst, shape_c,
                               rc.ld, v2=(kind == "v2")):
                if not self.cdist:
                    rc.flat.copy_(slab.allgather_planes(dst, self.tc))
                return rc
            self._fused_failed(kind)
        shape = (planes.shape[0],) + tuple(rf.space.local_shape[1:])
        ops = [(ax, op) for ax, op in enumerate(self.R) if op is not None and ax > 0]
        rc = StencilVector(Vc) if out is None else out
        own_view = rc.flat if self.cdist else None
        # axis 1 (slab axis)
        last = not ops
        if last and self.cdist:
            dst = own_view
        else:
            dst = _tmp((ce - cs + 1,) + shape[1:], ld, self.device, zero=False)
        shape = self.R0.apply(planes, dst, shape, ld, ld, 0)
        cur = dst
        for n, (ax, op) in enumerate(ops):
            shape_out = list(shape)
            shape_out[ax] = op.n_out
            last = n == len(ops) - 1
            ld_out = _pitch(op.n_out) if ax == nd - 1 else ld
            if last and self.cdist:
                dst = own_view
            else:
                dst = _tmp(shape_out, ld_out, self.device, zero=(ax == nd - 1))
            shape = op.apply(cur, dst, shape, ld, ld_out, ax)
            cur, ld = dst, ld_out
        if not self.cdist:
            full = slab.allgather_planes(cur, self.tc)
            rc.flat.copy_(full)
        return rc

    def prolong_add(self, ec, xf):
        slab = self.slab
        cur, ld = ec.flat, ec.ld
        shape = tuple(ec.space.local_shape)
        nd = len(shape)
        # coarse planes of the neighbours through the ghost planes of e_c (a view), so that the
        # in-plane passes below run on them too and no intermediate array has to be re-gathered
        gview = self._ghost_view(ec, self.tc, self.need_c) if self.cdist else None
        if gview is not None:
            cur = gview
            shape = (cur.shape[0],) + tuple(shape[1:])
        kind = (self._want_fused(xf.space.local_shape, "prolong")
                if (gview is not None or not self.cdist) else None)
        if kind:
            if _fused_prolong((self.P0, self.P[1], self.P[2]), cur, shape, ld, xf.flat,
                              tuple(xf.space.local_shape), xf.ld, True, v2=(kind == "v2")):
                return xf
            self._fused_failed(kind)
        ops = [(ax, op) for ax, op in reversed(list(enumerate(self.P))) if op is not None and ax > 0]
        for ax, op in ops:
            shape_out = list(shape)
            shape_out[ax] = op.n_out
            ld_out = _pitch(op.n_out) if ax == nd - 1 else ld
            dst = _tmp(shape_out, ld_out, self.device, zero=(ax == nd - 1))
            shape = op.apply(cur, dst, shape, ld, ld_out, ax)
            cur, ld = dst, ld_out
        assert ld == xf.ld
        if self.cdist and gview is None:
            planes = slab.gather_planes(cur, self.tc, self.need_c)
        else:
            planes = cur
        shape = (planes.shape[0],) + tuple(shape[1:])
        self.P0.apply(planes, xf.flat, shape, ld, ld, 0, accumulate=True)
        return xf


class CoarseSolver:
    """Exact inverse of a Kronecker-sum operator by fast diagonalisation:
    K_a Q_a = M_a Q_a L_a, Q_a^T M_a Q_a = I  =>  A^-1 = (x)Q_a . diag(1/sum_a l_a) . (x)Q_a^T.
    Replaces splu(csc_matrix(Ac)).solve(rc) (mg_jac.py:98-99); the 1-D eigenbases are dense
    n_c x n_c and are applied as per-axis contractions."""

    def __init__(self, A, device):
        from scipy.linalg import eigh
        assert A.form == 1, "fast diagonalisation needs the Kronecker-sum form"
        self.ndim = A.ndim
        self.npts = A.npts
        lam, self.Q, self.Qt = [], [], []
        for a in range(A.ndim):
            Kd = bs.band_to_dense(A.Ks[a])
            Md = bs.band_to_dense(A.Ms[a])
            from . import setup_device as sd
            if sd.enabled():
                w, Q = sd.gen_eigh(Kd, Md, device)
            else:
                w, Q = eigh(0.5 * (Kd + Kd.T), 0.5 * (Md + Md.T))
            lam.append(w)
            n = Q.shape[0]
            z = np.zeros(n, dtype=np.int32)
            self.Q.append(_AxisOp(z, Q, n, device, dense=True))
            self.Qt.append(_AxisOp(z, np.ascontiguousarray(Q.T), n, device, dense=True))
        D = 0.0
        for a in range(A.ndim):
            t = np.ones(())
            for c in range(A.ndim):
                t = np.multiply.outer(t, lam[c] if c == a else np.ones_like(lam[c]))
            D = D + t
        ld = _pitch(D.shape[-1])
        Dp = np.ones(D.shape[:-1] + (ld,))          # pad column: 1 so that 0/1 stays 0
        Dp[..., :D.shape[-1]] = D
        self.D = torch.as_tensor(np.ascontiguousarray(Dp), device=device)
        self.device = device

    def solve(self, b, out=None):
        """x = A^-1 b (a new vector, or `out`)."""
        V = b.space
        shape = tuple(V.local_shape)
        ld = V.ld
        if getattr(self, "_t", None) is None:
            self._t = (_tmp(shape, ld, self.device), _tmp(shape, ld, self.device))
        t0, t1 = self._t
        cur = b.flat
        bufs = [t0, t1]
        for a in range(self.ndim):
            dst = bufs[a % 2]
            self.Qt[a].apply(cur, dst, shape, ld, ld, a)
            cur = dst
        other = bufs[self.ndim % 2]
        ctx = DeviceContext.get(self.device)
        _lib.check(_lib.lib().poms_diag_scale(other.data_ptr(), cur.data_ptr(), self.D.data_ptr(),
                                               cur.numel(), 1.0, None, ctx.ws_ptr, _stream()),
                   "poms_diag_scale")
        cur = other
        x = StencilVector(V) if out is None else out
        for a in range(self.ndim):
            last = a == self.ndim - 1
            dst = x.flat if last else (t0 if cur is t1 else t1)
            self.Q[a].apply(cur, dst, shape, ld, ld, a)
            cur = dst
        return x


# ==========================================================================================
# two-grid cycle of the reference scripts
# ==========================================================================================
def two_grid(A, transfer, coarse, b, Vc, post="jac", M1=None, M2=None, p=None,
             pre_maxiter=10, post_maxiter=10, tol=1e-6):
    """One two-grid cycle in the order of /root/reference/sources/mg_jac.py:85-119
    (post='jac') or /root/reference/sources/mg_glt.py:84-123 (post='glt')."""
    ctx = DeviceContext.get(b.space.device)
    xf, info_pre = solvers.pcg(A, solvers.damped_jacobi, b, tol=tol, maxiter=pre_maxiter)
    rf = StencilVector(b.space)
    A.apply(xf, rf, EPI_RESID, b=b, dot_ptr=ctx.sptr(solvers.S_TMP))   # rf = bf - Af.dot(xf)
    rc = transfer.restrict(rf, Vc)                                     # rc = R.dot(rf)
    xc = coarse.solve(rc)                                              # splu(Ac).solve(rc)
    x_corr = xf.copy()
    transfer.prolong_add(xc, x_corr)                                   # xf = xf + P.dot(xc)
    if post == "jac":
        xf2, info_post = solvers.pcg(A, solvers.damped_jacobi, b, x0=x_corr, tol=tol,
                                     maxiter=post_maxiter)
    else:
        xf2, info_post = solvers.pcg_glt(A, M1, M2, b, x0=x_corr, tol=tol, maxiter=p + 1)
    return dict(x_pre=xf, info_pre=info_pre, r_f=rf, r_c=rc, x_c=xc, x_corr=x_corr,
                x_post=xf2, info_post=info_post)


# ==========================================================================================
# EXTENSION: multi-level V-cycle and MG-preconditioned CG
# ==========================================================================================
def _gen_eig_max(Kb, Tb):
    """Largest generalised eigenvalue of K x = mu T x for banded SPD 1-D matrices (host).
    n <= 1500: dense LAPACK (exact; what the oracle does).  Larger n: Lanczos on T^-1 K with banded
    solves, tolerance 1e-3 (the top of these spectra is a dense cluster: a tight tolerance took
    256 s at n = 8197, and the Chebyshev interval carries a 10 % safety factor anyway)."""
    n = Kb.shape[0]
    from . import setup_device as sd
    if sd.enabled():
        return sd.gen_eig_max(Kb, Tb)
    if n <= 1500:
        from scipy.linalg import eigh
        return float(eigh(bs.band_to_dense(Kb), bs.band_to_dense(Tb), eigvals_only=True,
                          subset_by_index=[n - 1, n - 1])[0])
    from scipy.linalg import solve_banded
    from scipy.sparse.linalg import eigsh, LinearOperator

    def trimmed(band):
        p = (band.shape[1] - 1) // 2
        q = p
        while q > 0 and not band[:, p - q].any() and not band[:, p + q].any():
            q -= 1
        return band[:, p - q:p + q + 1], q

    def apply(band, q, x):
        y = np.zeros(n)
        for k in range(-q, q + 1):
            lo, hi = max(0, -k), min(n, n - k)
            y[lo:hi] += band[lo:hi, k + q] * x[lo + k:hi + k]
        return y

    Kt, qk = trimmed(Kb)
    Tt, qt = trimmed(Tb)
    ab = np.zeros((2 * qt + 1, n))
    for k in range(-qt, qt + 1):
        i = np.arange(max(0, -k), min(n, n - k))
        ab[qt - k, i + k] = Tt[i, k + qt]
    op = LinearOperator((n, n), matvec=lambda v: apply(Kt, qk, v), dtype=float)
    M = LinearOperator((n, n), matvec=lambda v: apply(Tt, qt, v), dtype=float)
    Minv = LinearOperator((n, n), matvec=lambda v: solve_banded((qt, qt), ab, v), dtype=float)
    v0 = np.cos(np.arange(n) * 0.7) + 1.5          # deterministic start vector
    return float(eigsh(op, k=1, M=M, Minv=Minv, which="LA", tol=1e-3, ncv=24, v0=v0,
                       return_eigenvectors=False)[0])


class Level:
    def ws(self, name):
        """Persistent work vector of this level (zero-initialised once, then reused by every cycle):
        no allocation, no memset and stable device addresses inside the V-cycle, which is what lets
        the cycle be captured in a CUDA graph."""
        d = self.__dict__.setdefault("_ws", {})
        v = d.get(name)
        if v is None:
            v = d[name] = StencilVector(self.V, peer=True)
        return v


class Hierarchy:
    """Dyadic hierarchy of nested spline spaces for -Lap u + c u on [0,1]^d with du/dn + alpha u = 0
    on the boundary (default c = 1, alpha = 0: the reference's problem; `KronSumMatrix.poisson`).
    Every level has the same c and alpha: the prolongation keeps boundary values on open knot vectors,
    so P^T A_f P = A_c holds with the reaction and Robin terms too.

    N: elements per axis on the fine level (int or per-axis sequence); every level halves each
    axis that still has more than `Nc` elements (coarsen='semi') or all axes together until one
    reaches `Nc` (coarsen='uniform').  smoother: 'glt' | 'glt_poly' | 'jacobi'.
    """

    def __init__(self, p, N, ndim=None, Nc=8, device="cuda", smoother="glt", nu=1, ratio=4.0,
                 safety=1.1, slab=None, lengths=None, min_planes=32, coarsen="semi", setup="host",
                 c=1.0, robin=None, beta=None):
        """setup='device': the 1-D setup (assembly, knot-insertion rows, banded LU, eigenproblems)
        runs on the GPU (setup_device.py); 'host' (default): NumPy / SciPy.
        c, robin: reaction coefficient and Robin coefficients of every level's operator
        (`KronSumMatrix.poisson`; ValueError for negative values or a singular operator).
        beta: constant velocity (one component per axis) of a convection term beta . grad u.  Only the
        fine-level operator `h.op` carries it; every level keeps the symmetric operator -Lap + c with
        the same Robin faces, whose V-cycle preconditions `mg_gmres` (ValueError when the symmetric
        part of `h.op` is not positive definite).  Without beta, `h.op` is `levels[0].A`."""
        if setup == "device":
            from . import setup_device as sd
            with sd.device_setup(True, device):
                self.__init__(p, N, ndim=ndim, Nc=Nc, device=device, smoother=smoother, nu=nu, ratio=ratio,
                              safety=safety, slab=slab, lengths=lengths, min_planes=min_planes,
                              coarsen=coarsen, setup="host", c=c, robin=robin, beta=beta)
            self.setup = "device"
            return
        self.setup = "host"
        if np.isscalar(N):
            N = [int(N)] * int(ndim)
        # domain [0, L_1] x .. x [0, L_d] (default the unit cube).  Weak scaling extends the domain
        # along the slab axis (L_1 = number of GPUs) so that the elements stay cubes.
        self.lengths = [1.0] * len(N) if lengths is None else [float(v) for v in lengths]
        self.p, self.ndim = p, len(N)
        self.c, self.robin = reaction_robin(c, robin, self.ndim)
        self.beta = convection_beta(beta, self.ndim)
        if self.beta is not None:
            # built (and checked) first, so that a rejected velocity costs no hierarchy
            fine_knots_ = [bs.make_open_knots(p, n + p) * L for n, L in zip(N, self.lengths)]
            op = KronSumMatrix.poisson(p, fine_knots_, c=self.c, robin=self.robin, beta=self.beta)
        self.device = torch.device(device)
        self.smoother, self.nu, self.ratio, self.safety = smoother, nu, ratio, safety
        self.levels = []
        # grids of the hierarchy
        grids = [list(N)]
        while True:
            Ns = grids[-1]
            if all(n <= Nc for n in Ns):
                break
            # coarsen='uniform': stop as soon as one axis cannot be halved, so the elements keep their
            # shape on every level (elongated weak-scaling domains: semi-coarsening the long axis
            # alone costs 5 of 22 iterations at 8 slabs); 'semi': keep halving the longer axes
            if coarsen == "uniform" and not all(n > Nc and n % 2 == 0 for n in Ns):
                break
            nxt = [n // 2 if (n > Nc and n % 2 == 0) else n for n in Ns]
            if nxt == Ns:
                break
            grids.append(nxt)
        for i, Ns in enumerate(grids):
            lv = Level()
            lv.N = list(Ns)
            lv.knots = [bs.make_open_knots(p, n + p) * L for n, L in zip(Ns, self.lengths)]
            lv.A = KronSumMatrix.poisson(p, lv.knots, c=self.c, robin=self.robin)
            # a level stays slab-partitioned while every slab keeps at least `min_planes` planes
            # (and enough for the p-wide halo and the 2q interface planes of the partitioned solve);
            # below that the per-operation latency of the exchanges exceeds the work, so the level is
            # gathered and every rank works on the whole (small) grid redundantly.  The coarsest
            # level is always replicated: its exact solve is a replicated dense contraction.
            lv.distributed = (slab is not None and slab.size > 1 and i < len(grids) - 1
                              and (not self.levels or self.levels[-1].distributed)
                              and (Ns[0] + p) >= slab.size * max(2 * p + 2, min_planes))
            # ghost planes along the slab axis: p for the operator, 2q for the F2 pass of glt_poly
            gp = max(p, 2 * max(p - 1, 1)) if smoother == "glt_poly" else p
            lv.V = StencilVectorSpace([n + p for n in Ns], [gp] + [p] * (self.ndim - 1),
                                      [False] * self.ndim, device=self.device,
                                      slab=slab if lv.distributed else None)
            self.levels.append(lv)
        for f, c in zip(self.levels[:-1], self.levels[1:]):
            if f.distributed:
                f.transfer = DistTransfer(c.knots, f.knots, p, self.device, slab, c.distributed)
            else:
                f.transfer = Transfer(c.knots, f.knots, p, self.device)
        self.op = self.levels[0].A if self.beta is None else op
        self.coarse = CoarseSolver(self.levels[-1].A, self.device)
        for lv in self.levels[:-1]:
            self._setup_smoother(lv)

    def _setup_smoother(self, lv):
        p = self.p
        A = lv.A
        if self.smoother == "glt":
            q = max(2 * p - 1, 1)
            lv.glt_bands = [bs.glt_band(p, n, degree=q) for n in A.npts]
            lv.glt_lu = [BandLU.from_band(b, self.device) for b in lv.glt_bands]
            lv.lmax = self.safety * self._glt_lmax(lv)
        elif self.smoother == "glt_poly":
            # B^-1 ~ q(T) (x) .. (x) q(T): degree-3 Chebyshev approximation of the GLT solve, applied
            # as TWO fused Kronecker band passes (F1: half-bandwidth q, F2: 2q) instead of 2d
            # sequential triangular sweeps.  Same lambda_max formula as 'glt' (B is spectrally within
            # (1 +- 0.1)^d of the exact Kronecker solve).
            q = max(2 * p - 1, 1)
            lv.glt_bands = [bs.glt_band(p, n, degree=q) for n in A.npts]
            F = [bs.poly_inverse_factors(b_, 3) for b_ in lv.glt_bands]
            lv.S1 = KronSumMatrix([f[0] for f in F])
            lv.S2 = KronSumMatrix([f[1] for f in F])
            lv.lmax = self.safety * self._glt_lmax(lv)    # q(t) t = 0.9 at the high-frequency end of the symbol
        elif self.smoother == "jacobi":
            lv.lmax = self.safety * self._power_lmax_jacobi(lv)
        else:
            raise ValueError("smoother must be 'glt', 'glt_poly' or 'jacobi'")
        lv.lmin = lv.lmax / self.ratio

    def _glt_lmax(self, lv):
        """lambda_max(B^-1 A) ~ max_a mu(K_a + c M_a) prod_{b != a} mu(M_b), B = T (x) .. (x) T: 1-D
        generalised eigenvalues wrt T (accurate to ~1 % in 2-D/3-D, see DESIGN.md).  K_a here is the
        level's band, so it carries the Robin entries of its axis (and the last one c M already)."""
        A, d = lv.A, self.ndim
        muM = [_gen_eig_max(A.mass_bands[a], lv.glt_bands[a]) for a in range(d)]
        best = 0.0
        for a in range(d):
            Kb = A.Ks[a] + (self.c * A.mass_bands[a] if a != d - 1 else 0.0)  # K_a + c M_a
            muK = _gen_eig_max(bs.pad_band(Kb, A.P), bs.pad_band(lv.glt_bands[a], A.P))
            best = max(best, muK * float(np.prod([muM[b] for b in range(d) if b != a])))
        return best

    def _power_lmax_jacobi(self, lv, iters=30):
        """lambda_max(D^-1 A) by power iteration on the device (setup; deterministic start)."""
        V = lv.V
        ctx = DeviceContext.get(self.device)
        g = torch.Generator(device="cpu").manual_seed(1234)
        # from_array keeps the owned planes of the (identical on every rank) global start vector
        v = StencilVector.from_array(V, torch.rand(V.npts, generator=g, dtype=torch.float64)
                                     .numpy() + 0.5)
        zero = StencilVector(V)
        w = StencilVector(V)
        lam = 1.0
        for _ in range(iters):
            # w = -D^-1 (0 - A v) = D^-1 A v
            lv.A.apply(v, w, EPI_DINV, b=zero, omega=-1.0, dot_ptr=ctx.sptr(solvers.S_TMP))
            nw = sqrt(solvers._read(ctx, V, solvers.S_TMP))    # all-reduced over the slabs
            nv = sqrt(v.dot(v))
            lam = nw / nv
            v = w * (1.0 / nw)
        return lam

    # ---- smoothing: nu Chebyshev steps on B^-1 A --------------------------------------------
    def smooth(self, lv, b, x, zero_guess, final_dot=None):
        """final_dot = (vector r, device scalar pointer): ask the LAST pass of the smoother to leave
        x . r in the scalar (fused epilogue of the polynomial smoother); returns (x, fused)."""
        self._dot_fused = False
        A = lv.A
        V = lv.V
        L = _lib.lib()
        ctx = DeviceContext.get(self.device)
        theta = 0.5 * (lv.lmax + lv.lmin)
        delta = 0.5 * (lv.lmax - lv.lmin)
        sigma = theta / delta
        rho = 1.0 / sigma
        if self.smoother == "glt_poly":
            # nu Richardson steps x <- x + (1/theta) S2 S1 (b - A x): three fused Kronecker passes
            t1 = lv.ws("t1")
            for k in range(self.nu):
                if k == 0 and zero_guess:
                    src = b
                else:
                    r = lv.ws("r")
                    A.apply(x, r, EPI_RESID, b=b)
                    src = r
                lv.S1.apply(src, t1, EPI_STORE)
                # in place: the epilogue reads x[i] and writes x[i] from the same thread, and the
                # mat-vec input is t1, so no other thread reads x.  Zero guess: x = (1/theta) S2 t1,
                # x is neither cleared nor read (b = None).
                last = final_dot is not None and k == self.nu - 1
                fused = lv.S2.apply(t1, x, EPI_AXPY, b=None if (k == 0 and zero_guess) else x,
                                    omega=1.0 / theta, dot_ptr=final_dot[1] if last else None,
                                    dot_with=final_dot[0] if last else None)
                if last:
                    self._dot_fused = bool(fused)
            return x
        if self.smoother == "glt" and self.nu == 1 and all(lu.nopiv for lu in lv.glt_lu):
            # one step: x <- x + (1/theta) B^-1 (b - A x); the update is fused into the last line
            # solve (d = c1*d + c2*z with c1 = 0, so x + d == x + c2*z)
            work = lv.ws("t1")
            if zero_guess:
                kron_solve_bnd_update(lv.glt_lu, b, work, x, 1.0 / theta)
            else:
                r = lv.ws("r")
                A.apply(x, r, EPI_RESID, b=b)
                kron_solve_bnd_update(lv.glt_lu, r, work, x, 1.0 / theta, add=x)
            return x
        r = lv.ws("r")
        z = lv.ws("t1") if self.smoother == "glt" else r
        d = lv.ws("d")                        # written (c1 = 0) by the first Chebyshev step
        for k in range(self.nu):
            if self.smoother == "glt":
                if k == 0 and zero_guess:
                    src = b                                      # r = b - A.0 = b
                else:
                    A.apply(x, r, EPI_RESID, b=b)                # r = b - A x
                    src = r
                kron_solve_bnd(lv.glt_lu, src, z)                # z = B^-1 r
            else:
                if k == 0 and zero_guess:
                    A.jacobi_first(z, b, 1.0, None)              # z = D^-1 b
                else:
                    A.apply(x, z, EPI_DINV, b=b, omega=1.0)      # z = D^-1 (b - A x)
            if k == 0:
                c1, c2 = 0.0, 1.0 / theta
            else:
                rho_n = 1.0 / (2.0 * sigma - rho)
                c1, c2 = rho_n * rho, 2.0 * rho_n / delta
                rho = rho_n
            with profiling.region("cheb_update", 40 * x.n_owned):
                _lib.check(L.poms_cheb_update(x.ptr, d.ptr, z.ptr, c1, c2, x.n_owned, _stream()),
                           "poms_cheb_update")
        return x


def vcycle(h, l, b, final_dot=None):
    """One V(nu,nu) cycle from a zero initial guess on level l.  Returns the level's persistent
    solution vector `lv.ws("x")`: it is overwritten by the next cycle, copy it to keep it.
    final_dot = (r, scalar pointer): the post-smoother's last pass also leaves x . r there when it
    can (`h._dot_fused` tells)."""
    h._dot_fused = False
    lv = h.levels[l]
    if l == len(h.levels) - 1:
        return h.coarse.solve(b, out=lv.ws("x"))
    x = lv.ws("x")
    # the polynomial smoother and the fused GLT update overwrite x on a zero guess; the Chebyshev
    # recurrences accumulate into it
    if not (h.smoother == "glt_poly" or (h.smoother == "glt" and h.nu == 1
                                         and all(lu.nopiv for lu in lv.glt_lu))):
        x.flat.zero_()
    h.smooth(lv, b, x, True)
    r = lv.ws("r")
    lv.A.apply(x, r, EPI_RESID, b=b)
    with profiling.region("restrict", 8 * lv.V.local_size, launches=None):
        rc = lv.transfer.restrict(r, h.levels[l + 1].V, out=h.levels[l + 1].ws("b"))
    ec = vcycle(h, l + 1, rc)
    with profiling.region("prolong_add", 16 * lv.V.local_size, launches=None):
        lv.transfer.prolong_add(ec, x)
    h.smooth(lv, b, x, False, final_dot=final_dot)
    return x


def _graphs_wanted(h, b):
    """How the PCG iteration is driven: 'graph' = two CUDA graphs per iteration (one device, no
    per-kernel instrumentation, not disabled by POMS_B200_GRAPH=0); 'persistent' = the same two
    bodies launched eagerly on the hierarchy's persistent vectors (slab-partitioned runs: the
    vectors then live in the peer arena and every halo exchange is a peer store); None = the
    launch-by-launch driver of solvers.py."""
    import os
    V = b.space
    if not (V.compatible(h.levels[0].V) and V.pads == h.levels[0].V.pads):
        return None
    if V.slab is not None and V.slab.size > 1:
        # POMS_B200_GRAPH_DIST=1 (experimental): capture the slab iteration too -- the peer-store halo
        # kernels and the NCCL collectives capture and replay correctly (measured on 2 GPUs: C5 265.7
        # vs 266.2 ms, C4 332 vs 348 ms), but the processes then hang in NCCL teardown at exit, so the
        # default stays: eager launches on the persistent vectors
        if (os.environ.get("POMS_B200_GRAPH_DIST", "0") == "1" and not profiling.enabled()
                and os.environ.get("POMS_B200_GRAPH", "1") != "0"):
            return "graph"
        return "persistent"
    if os.environ.get("POMS_B200_GRAPH", "1") != "0" and not profiling.enabled():
        return "graph"
    return None


class _PcgGraphs:
    """Persistent PCG state of one hierarchy (x, r, p, q on the fine level) and the two halves of
    an iteration of /root/reference/sources/solvers.py:101-124 with the V-cycle as psolve:
        G1: q = A p ; p.q ; x += alpha p ; r -= alpha q ; r.r          (lines 103-111)
        G2: s = V-cycle(r) ; s.r ; p = s + beta p ; sr_old = sr         (lines 117-124)
    The break test between them (line 113) reads one scalar on the host.  The launch sequence of a
    hierarchy is fixed and alpha / beta already live on the device, so on one device the ~60 (C5)
    to ~90 launches of an iteration are captured as two CUDA graphs: the coarse levels stop being
    launch-latency bound.  capture=False (slab-partitioned runs) launches the same bodies eagerly;
    the scalars are then all-reduced in place on the device."""

    def __init__(self, h, capture=True):
        import weakref
        from .solvers import S_RR, S_PQ, S_SR0, S_SR1
        lv = h.levels[0]
        self._h = weakref.ref(h)          # no reference cycle: the graphs die with the hierarchy
        self.capture = capture
        self.x, self.r, self.p, self.q = (lv.ws(n) for n in ("pcg_x", "pcg_r", "pcg_p", "pcg_q"))
        self.ctx = DeviceContext.get(h.device)
        self.S_OLD, self.S_NEW = S_SR0, S_SR1
        self.n_g1 = self.n_g2 = 0
        if not capture:
            return
        L = _lib.lib()
        # eager dry run: creates every work vector, tensor map and function attribute, then capture
        self.r.flat.fill_(1.0)
        self.p.flat.zero_()
        self.x.flat.zero_()
        self.ctx.scal[self.S_OLD] = 1.0
        self._g2_body()
        self._g1_body()
        torch.cuda.synchronize()
        # collect dead reference cycles NOW: torch.cuda.graph does not, and a CUDA graph or tensor
        # freed by the cyclic collector in the middle of a capture invalidates it
        import gc
        gc.collect()
        self.g1, self.g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        n0 = L.poms_launch_count()
        with torch.cuda.graph(self.g1):
            self._g1_body()
        n1 = L.poms_launch_count()
        with torch.cuda.graph(self.g2):
            self._g2_body()
        self.n_g1, self.n_g2 = n1 - n0, L.poms_launch_count() - n1
        self.pad_clean()

    @property
    def h(self):
        return self._h()

    def pad_clean(self):
        for v in (self.x, self.r, self.p, self.q):
            V = v.space
            if V.ld != V.local_shape[-1]:
                v._buf[..., V.local_shape[-1]:] = 0.0

    def _g1_body(self):
        from .solvers import S_RR, S_PQ, _reduce
        A, ctx, L = self.h.levels[0].A, self.ctx, _lib.lib()
        V = self.x.space
        A.apply(self.p, self.q, EPI_STORE, dot_ptr=ctx.sptr(S_PQ))
        _reduce(ctx, V, S_PQ)
        with profiling.region("cg_update", 48 * self.x.n_owned):
            _lib.check(L.poms_cg_update(self.x.ptr, self.r.ptr, self.p.ptr, self.q.ptr, self.x.n_owned,
                                        ctx.sptr(self.S_OLD), ctx.sptr(S_PQ), ctx.sptr(S_RR), ctx.ws_ptr,
                                        _stream()), "poms_cg_update")
        _reduce(ctx, V, S_RR)

    def _g2_body(self):
        from .stencil import dot_into
        from .solvers import _reduce
        ctx, L = self.ctx, _lib.lib()
        V = self.x.space
        # s.r (sources/solvers.py:117-118) can ride in the last smoother pass (POMS_B200_FUSE_SR=1):
        # measured on C5 it does NOT pay yet -- the extra tile ring of r pushes the p = 4 smoother
        # pass from two CTAs per SM to one (117.6 KB of shared memory), which costs more than the
        # 6.5 ms dot kernel it removes (236.9 vs 233.1 ms per solve) -- so the default keeps the
        # separate dot kernel
        import os
        fd = (self.r, ctx.sptr(self.S_NEW)) if os.environ.get("POMS_B200_FUSE_SR") == "1" else None
        s = vcycle(self.h, 0, self.r, final_dot=fd)
        if not self.h._dot_fused:
            with profiling.region("dot", 16 * self.x.n_owned):
                dot_into(s, self.r, ctx.sptr(self.S_NEW), ctx)
        _reduce(ctx, V, self.S_NEW)
        with profiling.region("p_update", 24 * self.x.n_owned):
            _lib.check(L.poms_p_update(self.p.ptr, s.ptr, self.p.n_owned, ctx.sptr(self.S_NEW),
                                       ctx.sptr(self.S_OLD), _stream()), "poms_p_update")
        ctx.scal[self.S_OLD:self.S_OLD + 1].copy_(ctx.scal[self.S_NEW:self.S_NEW + 1])

    def run_g1(self):
        if not self.capture:
            return self._g1_body()
        self.g1.replay()
        _lib.lib().poms_launch_count_add(self.n_g1)

    def run_g2(self):
        if not self.capture:
            return self._g2_body()
        self.g2.replay()
        _lib.lib().poms_launch_count_add(self.n_g2)


def _pcg_graphed(h, b, x0, tol, maxiter, abs_thresh=None, capture=True):
    """`solvers._pcg_driver(relative=True)` on the persistent state of `_PcgGraphs` (same operations,
    same order, same device scalars; p = s is realised as p = s + beta*0)."""
    from .solvers import S_RR, _reduce
    from .stencil import dot_into
    g = h.__dict__.get("_pcg_graphs")
    if g is None or g.capture != capture:
        g = h._pcg_graphs = _PcgGraphs(h, capture=capture)
    ctx, A = g.ctx, h.levels[0].A
    x, r, p = g.x, g.r, g.p
    if x0 is None:
        x.flat.zero_()
        r.flat.copy_(b.flat)
        dot_into(r, r, ctx.sptr(S_RR), ctx)
    else:
        if x0 is not x:
            x.flat.copy_(x0.flat)
        A.apply(x, r, EPI_RESID, b=b, dot_ptr=ctx.sptr(S_RR))
    _reduce(ctx, b.space, S_RR)
    nrmr0 = sqrt(float(ctx.scal[S_RR].item()))
    thresh = (tol * nrmr0) ** 2
    if abs_thresh is not None:
        thresh = abs_thresh
        if nrmr0 * nrmr0 <= thresh:
            return x, {"niter": 0, "success": True, "res_norm": nrmr0, "history": [],
                       "res_norm0": nrmr0}
    p.flat.zero_()
    ctx.scal[g.S_OLD] = 1.0
    g.run_g2()                       # s = psolve(r); p = s; sr
    hist = []
    k = 0
    nrmr = nrmr0 * nrmr0
    for k in range(1, maxiter + 1):
        g.run_g1()
        nrmr = float(ctx.scal[S_RR].item())
        hist.append(sqrt(nrmr))
        if nrmr <= thresh:
            k -= 1
            break
        g.run_g2()
    info = {"niter": k, "success": bool(nrmr <= thresh), "res_norm": sqrt(nrmr), "history": hist,
            "res_norm0": nrmr0}
    return x, info


def mg_pcg(h, b, x0=None, tol=1e-10, maxiter=200, criterion="relative", verbose=False,
           max_restarts=3):
    """MG-preconditioned CG: the reference's `pcg` driver (same operation order) with one V-cycle
    as `psolve`.  criterion='relative': stop when ||r|| <= tol*||r0|| (the BASELINE metric);
    criterion='reference': the reference's own mixed rule r.r < tol*||r0||.
    On one device the iteration runs as two CUDA graphs (`_PcgGraphs`; POMS_B200_GRAPH=0 or an
    enabled profiler selects the launch-by-launch driver); the returned x is then the hierarchy's
    persistent solution vector, overwritten by the next solve on the same hierarchy."""
    if h.beta is not None:
        raise ValueError("mg_pcg needs a symmetric operator: a hierarchy with a convection term (beta) is "
                         "solved by mg_gmres")
    A = h.levels[0].A

    def psolve(A_, r):
        return vcycle(h, 0, r)

    if criterion == "reference":
        return solvers.pcg(A, psolve, b, x0=x0, tol=tol, maxiter=maxiter, verbose=verbose)
    mode = None if verbose else _graphs_wanted(h, b)
    graphed = mode == "graph"

    def drive(x0_, tol_, maxiter_, title, abs_thresh=None):
        if mode is not None:
            return _pcg_graphed(h, b, x0_, tol_, maxiter_, abs_thresh=abs_thresh, capture=graphed)
        return solvers._pcg_driver(A, psolve, b, x0_, tol_, maxiter_, verbose, title,
                                   relative=True, abs_thresh=abs_thresh)

    x, info = drive(x0, tol, maxiter, "MG-PCG solver:")
    # The CG recurrence residual drifts from b - A x on ill-conditioned problems (2-D 2048^2: 1e-10
    # claimed, 9e-10 true).  Verify with the TRUE residual and restart from x until it meets the
    # target (each restart recomputes r = b - A x; it returns at once when the target is met).
    target = (tol * info["res_norm0"]) ** 2
    info["restarts"] = 0
    while info["restarts"] < max_restarts and info["niter"] < maxiter:
        x2, i2 = drive(x, tol, maxiter - info["niter"], "MG-PCG restart:", abs_thresh=target)
        info["res_norm"] = i2["res_norm"] if i2["niter"] else i2["res_norm0"]
        info["true_res_norm"] = i2["res_norm0"] if not i2["niter"] else None
        if i2["niter"] == 0:
            break
        x = x2
        info["niter"] += i2["niter"]
        info["history"] = list(info["history"]) + list(i2["history"])
        info["restarts"] += 1
    info["success"] = bool(info["res_norm"] ** 2 <= target)
    info["graphed"] = bool(graphed)
    return x, info


def mg_gmres(h, b, x0=None, tol=1e-10, maxiter=300, restart=30):
    """Solve h.op x = b (the convection-diffusion operator of `Hierarchy(beta=)`, or the symmetric one)
    by `solvers.gmres` with right preconditioning by one V-cycle of the symmetric hierarchy.  The V-cycle
    from a zero guess is a fixed linear map (what GMRES needs of its preconditioner), spectrally
    equivalent to h.op at fixed beta and c, so the iteration count does not grow with the grid.  Its
    result lives in the hierarchy's workspace, which the next cycle overwrites, so it is copied into a
    vector that gmres owns.  Works on slab-partitioned hierarchies (the dots of gmres are all-reduced,
    the mat-vecs exchange halos).  Returns (x, info) like mg_pcg:
    info['res_norm'] is the true residual ||b - h.op x|| (gmres recomputes it before it stops), and
    info['success'] says whether it is <= tol * ||b - h.op x0||."""
    def psolve(A_, v):
        return vcycle(h, 0, v).copy()

    return solvers.gmres(h.op, b, x0=x0, tol=tol, maxiter=maxiter, restart=restart, psolve=psolve)
