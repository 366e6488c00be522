"""Reaction coefficient c and Robin / Neumann boundary terms: -Lap u + c u with du/dn + alpha u = g (CPU).

The oracle (tests/robin_oracle.py) against a dense assembly from scipy BSpline with its own Gauss rule and
face terms; the Galerkin identity P^T A_f P = A_c with c and Robin terms on every level; the bands of
KronSumMatrix.poisson against the oracle, and bit-identical to the previous operator at the defaults; the
lambda_max bound of the GLT smoothers against dense eigenvalues of B^-1 A; every ValueError of the
validation; the host-side checks of fem.boundary_load; the oracle's boundary load against scipy."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from scipy.interpolate import BSpline
from scipy.linalg import eigh

import robin_oracle as ro
from oracle import poms_oracle as po
from poms_b200 import bsplines as bs
from poms_b200.stencil import KronSumMatrix, StencilVectorSpace, StencilVector


def _knots(p, N, graded=False):
    T = bs.make_open_knots(p, N + p)
    if graded:
        T[p + 1:N + p] = T[p + 1:N + p] ** 1.5
    return T


def _scipy_axis(T, p):
    """Dense 1-D mass and stiffness from scipy BSpline with a (p+2)-point Gauss rule per element, and the
    basis values at both ends of the knot vector."""
    n = len(T) - p - 1
    u, w = np.polynomial.legendre.leggauss(p + 2)
    br = np.unique(T)
    x = np.concatenate([0.5 * (a + b) + 0.5 * (b - a) * u for a, b in zip(br[:-1], br[1:])])
    wq = np.concatenate([0.5 * (b - a) * w for a, b in zip(br[:-1], br[1:])])
    sp = [BSpline(T, np.eye(n)[i], p) for i in range(n)]
    B = np.array([s(x) for s in sp])
    D = np.array([s.derivative()(x) for s in sp])
    ends = np.array([[s(T[p]) for s in sp], [s(T[n]) for s in sp]])
    return (B * wq) @ B.T, (D * wq) @ D.T, ends


def _kron(mats):
    out = np.ones((1, 1))
    for m in mats:
        out = np.kron(out, m)
    return out


def _dense_scipy(p, knots, c, robin):
    ax = [_scipy_axis(T, p) for T in knots]
    d = len(ax)
    A = c * _kron([M for M, _, _ in ax])
    for a in range(d):
        A = A + _kron([ax[b][1] if b == a else ax[b][0] for b in range(d)])
    if robin is not None:                      # alpha int_F u v ds, face by face
        for a, pair in enumerate(robin):
            for side, alpha in enumerate(pair):
                e = ax[a][2][side]
                A = A + alpha * _kron([np.outer(e, e) if b == a else ax[b][0] for b in range(d)])
    return A


CASES = [(1.0, None), (0.0, "one"), (1e-3, "all"), (1e4, None), (2.5, "mixed")]


def _robin(kind, d):
    if kind is None:
        return None
    if kind == "one":
        return [(10.0, 0.0)] + [(0.0, 0.0)] * (d - 1)
    if kind == "all":
        return [(1.0, 1e3)] * d
    return [(0.0, 3.0), (0.5, 0.0), (2.0, 7.0)][:d]


# ------------------------------------------------------------------------------------- operator
@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("d", [2, 3])
@pytest.mark.parametrize("graded", [False, True])
def test_oracle_operator_vs_scipy(p, d, graded):
    Ns = (6, 5, 4)[:d] if d == 3 else (9, 7)
    knots = [_knots(p, N, graded and a != 1) for a, N in enumerate(Ns)]
    for c, kind in CASES:
        robin = _robin(kind, d)
        A = ro.poisson_operator(p, knots, c, robin)[0].tocsr().toarray()
        ref = _dense_scipy(p, knots, c, robin)
        assert np.abs(A - ref).max() < 1e-12 * np.abs(ref).max(), (c, kind)


def test_oracle_defaults_are_the_pinned_operator():
    p, knots = 3, [_knots(3, 7), _knots(3, 5, True), _knots(3, 6)]
    A0, M0, K0 = po.poisson_operator(p, knots)
    A1, M1, K1 = ro.poisson_operator(p, knots)
    for t0, t1 in zip(A0.terms, A1.terms):
        assert all(np.array_equal(a, b) for a, b in zip(t0, t1))
    assert all(np.array_equal(a, b) for a, b in zip(M0 + K0, M1 + K1))


@pytest.mark.parametrize("p,N,Nc", [(3, (16, 16), 4), (2, (16, 8, 8), 2), (1, (8, 16), 2), (5, (12, 12), 6)])
def test_galerkin_identity_every_level(p, N, Nc):
    d = len(N)
    for c, kind in CASES:
        h = ro.MGHierarchy(p, N, Nc=Nc, c=c, robin=_robin(kind, d))
        assert len(h.levels) >= 2
        for f, cl in zip(h.levels[:-1], h.levels[1:]):
            Ac = po.galerkin_dense(f["A"].tocsr(), f["P1s"])
            ref = cl["A"].tocsr().toarray()
            assert np.abs(Ac - ref).max() < 1e-12 * np.abs(ref).max(), (c, kind)


@pytest.mark.parametrize("p", [1, 3, 5])
@pytest.mark.parametrize("d", [2, 3])
def test_poisson_bands_vs_oracle(p, d):
    knots = [_knots(p, N, a == 0) for a, N in enumerate((7, 9, 6)[:d])]
    for c, kind in CASES:
        robin = _robin(kind, d)
        A = KronSumMatrix.poisson(p, knots, c=c, robin=robin)
        _, Mb, Kb = ro.poisson_operator(p, knots, c, robin)
        for a in range(d):
            K = Kb[a] + (c * Mb[a] if a == d - 1 else 0.0)
            assert np.abs(A.Ms[a] - Mb[a]).max() < 1e-14 * np.abs(Mb[a]).max()
            assert np.abs(A.Ks[a] - K).max() < 1e-12 * np.abs(K).max(), (a, c, kind)
            assert A.mass_bands[a] is A.Ms[a] or np.array_equal(A.mass_bands[a], A.Ms[a])


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_poisson_defaults_bit_identical(p):
    """c = 1 and no (or zero) Robin terms build exactly the bands of the operator before c and robin
    existed: K (x) M (x) M + M (x) K (x) M + M (x) M (x) (K + M)."""
    knots = [_knots(p, 40), _knots(p, 12, True), _knots(p, 33)]
    MK = [bs.assemble_1d_bands(p, T) for T in knots]
    old_K = [k for _, k in MK]
    old_K[-1] = old_K[-1] + MK[-1][0]
    ref = KronSumMatrix.poisson(p, knots)
    for A in (ref, KronSumMatrix.poisson(p, knots, c=1.0, robin=None),
              KronSumMatrix.poisson(p, knots, c=1, robin=[(0, 0)] * 3)):
        for a in range(3):
            assert np.array_equal(A.Ks[a], ref.Ks[a]) and np.array_equal(A.Ms[a], ref.Ms[a])
            assert np.array_equal(A.Ks[a], old_K[a]) and np.array_equal(A.Ms[a], MK[a][0])
        assert all(np.array_equal(x, y) for x, y in zip(A._toeplitz(), ref._toeplitz()))


def test_robin_and_reaction_keep_the_toeplitz_ranges():
    """A Robin entry changes a boundary row only and c M changes every row of the last axis alike, so the
    interior (Toeplitz) ranges the mat-vec kernels take from the constant bank stay the same."""
    p = 3
    knots = [_knots(p, N) for N in (40, 36, 50)]
    rng0 = KronSumMatrix.poisson(p, knots)._toeplitz()[1]
    for c, kind in CASES:
        rng = KronSumMatrix.poisson(p, knots, c=c, robin=_robin(kind, 3))._toeplitz()[1]
        assert np.array_equal(rng, rng0), (c, kind)


# ------------------------------------------------------------------------------------- lambda_max
LMAX_CASES = [(1.0, None), (0.0, "one"), (0.0, "all1"), (1e-3, None), (1e4, None), (1.0, "big"), (0.0, "big1")]


def _lmax_robin(kind, d):
    return {None: None, "one": [(10.0, 0.0)] + [(0.0, 0.0)] * (d - 1), "all1": [(1.0, 1.0)] * d,
            "big": [(1e3, 1e3)] * d, "big1": [(0.0, 0.0)] * (d - 1) + [(0.0, 1e3)]}[kind]


@pytest.mark.parametrize("p,N", [(1, (16, 16)), (2, (16, 16)), (3, (24, 8)), (5, (16, 16)), (2, (8, 8, 8)),
                                 (3, (8, 8, 8)), (5, (6, 6, 6))])
def test_glt_lmax_bound_vs_dense_eigenvalues(p, N):
    """lmax (with the 1.1 safety factor) >= lambda_max(B^-1 A) and <= 1.25 lambda_max, B = T (x) .. (x) T:
    the Chebyshev / Richardson smoothers stay convergent on [lmax / 4, lmax].  The package's bound and the
    oracle's agree."""
    from poms_b200.mg import Hierarchy
    d = len(N)
    knots = [bs.make_open_knots(p, n + p) for n in N]
    q = max(2 * p - 1, 1)
    for c, kind in LMAX_CASES:
        robin = _lmax_robin(kind, d)
        A = KronSumMatrix.poisson(p, knots, c=c, robin=robin)
        gb = [bs.glt_band(p, n, degree=q) for n in A.npts]
        est = Hierarchy._glt_lmax(SimpleNamespace(c=c, ndim=d), SimpleNamespace(A=A, glt_bands=gb))
        h = SimpleNamespace(c=c)
        _, Mb, Kb = ro.poisson_operator(p, knots, c, robin)
        est_o = ro.MGHierarchy.glt_lmax(h, dict(Mb=Mb, Kb=Kb), gb)
        assert abs(est - est_o) < 1e-10 * est_o
        Ad = ro.poisson_operator(p, knots, c, robin)[0].tocsr().toarray()
        B = _kron([bs.band_to_dense(g) for g in gb])
        lam = eigh(Ad, B, eigvals_only=True)[-1]
        lmax = 1.1 * est
        assert lam <= lmax <= 1.25 * lam, (c, kind, lmax / lam)


# ------------------------------------------------------------------------------------- validation
BAD = [dict(c=-1.0), dict(c=float("nan")), dict(c=float("inf")), dict(c="one"), dict(c=0.0),
       dict(c=0.0, robin=[(0.0, 0.0), (0.0, 0.0)]), dict(robin=[(1.0, 1.0)]),
       dict(robin=[(1.0, 1.0)] * 3), dict(robin=[(1.0, -1.0), (0.0, 0.0)]),
       dict(robin=[(1.0, float("nan")), (0.0, 0.0)]), dict(robin=[(1.0, float("inf")), (0.0, 0.0)]),
       dict(robin=[(1.0,), (0.0, 0.0)]), dict(robin=[(1.0, 2.0, 3.0), (0.0, 0.0)]), dict(robin=[1.0, 2.0]),
       dict(robin=[("a", 1.0), (0.0, 0.0)]), dict(c=-0.5, robin=[(1.0, 1.0)] * 2)]


@pytest.mark.parametrize("kw", BAD)
def test_bad_reaction_or_robin_raise(kw):
    from poms_b200.mg import Hierarchy
    knots = [_knots(2, 8), _knots(2, 8)]
    with pytest.raises(ValueError):
        KronSumMatrix.poisson(2, knots, **kw)
    with pytest.raises(ValueError):
        Hierarchy(2, [8, 8], device="cpu", **kw)
    with pytest.raises(ValueError):
        Hierarchy(2, [8, 8], device="cpu", setup="device", **kw)


def test_good_reaction_and_robin_accepted():
    from poms_b200.stencil import reaction_robin
    assert reaction_robin(0, [(0, 1e-300), (0, 0)], 2) == (0.0, [(0.0, 1e-300), (0.0, 0.0)])
    assert reaction_robin(np.float32(2), None, 3) == (2.0, None)
    assert reaction_robin(1.0, np.array([[1, 2], [3, 4]]), 2) == (1.0, [(1.0, 2.0), (3.0, 4.0)])


# ------------------------------------------------------------------------------------- boundary load
def _cpu_space(npts, p, slab=None):
    return StencilVectorSpace(list(npts), [p] * len(npts), [False] * len(npts), device="cpu", slab=slab)


class _TwoRankSlab:
    rank, size, device = 0, 2, None

    def bounds(self, n):
        return 0, n // 2 - 1


def test_boundary_load_argument_checks():
    from poms_b200 import fem
    p, Ns = 2, (5, 4, 6)
    knots = [_knots(p, N) for N in Ns]
    V = _cpu_space([N + p for N in Ns], p)
    g = lambda x, y: x * y
    for axis in (-1, 3, 1.0, True, None):
        with pytest.raises(ValueError):
            fem.boundary_load(V, knots, p, g, axis, 0)
    for side in (-1, 2, 0.5, None, True):
        with pytest.raises(ValueError):
            fem.boundary_load(V, knots, p, g, 0, side)
    with pytest.raises(ValueError):
        fem.boundary_load(V, knots, p, g, 0, 0, plane_chunk=0)
    with pytest.raises(ValueError):                                     # out of another space
        fem.boundary_load(V, knots, p, g, 0, 0, out=StencilVector(_cpu_space([N + p + 1 for N in Ns], p)))
    with pytest.raises(ValueError):                                     # p, knots: _check
        fem.boundary_load(V, knots, 6, g, 0, 0)
    with pytest.raises(ValueError):
        fem.boundary_load(V, knots[:2], p, g, 0, 0)
    with pytest.raises(ValueError):
        fem.boundary_load(V, [knots[0], _knots(p, 5), knots[2]], p, g, 0, 0)
    # a knot vector that is not open at the face: the end function is not the only one there
    T = knots[1].copy()
    T[0] = -0.25
    with pytest.raises(ValueError):
        fem.boundary_load(V, [knots[0], T, knots[2]], p, g, 1, 0)
    Vs = _cpu_space([N + p for N in (8, 6, 5)], p, slab=_TwoRankSlab())
    with pytest.raises(NotImplementedError):
        fem.boundary_load(Vs, [_knots(p, N) for N in (8, 6, 5)], p, g, 0, 0)


@pytest.mark.parametrize("p", [1, 2, 3, 5])
@pytest.mark.parametrize("d", [2, 3])
def test_oracle_boundary_load_vs_scipy(p, d):
    Ns = (6, 4, 5)[:d] if d == 3 else (7, 5)
    knots = [_knots(p, N, graded=(a == 0)) for a, N in enumerate(Ns)]
    npts = [N + p for N in Ns]
    g3 = lambda x, y: np.exp(x) * np.cos(2.0 * y) + x * x
    g2 = lambda x: np.exp(x) + x ** 3
    for axis in range(d):
        face = [b for b in range(d) if b != axis]
        vecs = []
        for b in face:
            u, w = np.polynomial.legendre.leggauss(p + 1)          # the rule of bsplines.quadrature_tables
            br = np.unique(knots[b])
            x = np.concatenate([0.5 * (s + t) + 0.5 * (t - s) * u for s, t in zip(br[:-1], br[1:])])
            wq = np.concatenate([0.5 * (t - s) * w for s, t in zip(br[:-1], br[1:])])
            B = np.array([BSpline(knots[b], np.eye(npts[b])[i], p)(x) for i in range(npts[b])])
            vecs.append((x, wq, B))
        for side in (0, 1):
            T = knots[axis]
            e = np.array([BSpline(T, np.eye(npts[axis])[i], p)(T[p] if side == 0 else T[-1])
                          for i in range(npts[axis])])
            if d == 2:
                (x, wq, B), = vecs
                plane = B @ (wq * g2(x))
                ref = np.moveaxis(np.multiply.outer(e, plane), 0, axis)
                got = ro.boundary_load(knots, p, g2, axis, side)
            else:
                (x1, w1, B1), (x2, w2, B2) = vecs
                G = g3(x1[:, None], x2[None, :]) * w1[:, None] * w2[None, :]
                plane = B1 @ G @ B2.T
                ref = np.moveaxis(np.multiply.outer(e, plane), 0, axis)
                got = ro.boundary_load(knots, p, g3, axis, side)
            assert np.abs(got - ref).max() < 1e-14 * np.abs(ref).max(), (axis, side)
