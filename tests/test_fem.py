"""poms_b200.fem: load vectors, error norms and evaluation on B-spline spaces.

CPU: the NumPy oracle (oracle/fem_oracle.py) against an independent computation (scipy BSpline basis,
numpy leggauss), the shared quadrature tables against the assembled mass / stiffness bands, argument checks.
GPU: exact identities against the device Kronecker operators, both kernels against the oracle (p = 1..5, 2-D
and 3-D, ragged shapes, graded knots, chunks of 1, 3 and all planes), determinism, `evaluate` against scipy,
and the convergence orders of a manufactured solution solved with mg_pcg."""
import numpy as np
import pytest
from scipy.interpolate import BSpline

from oracle import fem_oracle as fo
from poms_b200 import bsplines as bs


@pytest.fixture(scope="module")
def dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _knots(p, N, graded=False):
    T = bs.make_open_knots(p, N + p)
    if graded:
        T[p + 1:N + p] = T[p + 1:N + p] ** 1.5
    return T


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("p,N,graded", [(1, 5, False), (3, 7, True), (5, 6, False), (2, 9, True)])
def test_oracle_tables_vs_scipy(p, N, graded):
    T = _knots(p, N, graded)
    ax = fo.axis_matrices(T, p)
    n = len(T) - p - 1
    u, w = np.polynomial.legendre.leggauss(p + 1)
    xs, ws = [], []
    for a, b in zip(np.unique(T)[:-1], np.unique(T)[1:]):
        xs += list(0.5 * (a + b) + 0.5 * (b - a) * u)
        ws += list(0.5 * (b - a) * w)
    xs, ws = np.array(xs), np.array(ws)
    B = np.array([BSpline(T, np.eye(n)[i], p)(xs) for i in range(n)])
    D = np.array([BSpline(T, np.eye(n)[i], p).derivative()(xs) for i in range(n)])
    assert np.abs(ax["x"] - xs).max() < 1e-15 and np.abs(ax["w"] - ws).max() < 1e-15
    assert np.abs(ax["B"] - B).max() < 1e-13 and np.abs(ax["D"] - D).max() < 1e-11 * max(1, np.abs(D).max())
    # load vector of f = exp(x) sin(y) in 2-D against the scipy tables
    b = fo.load_vector([T, T], p, lambda x, y: np.exp(x) * np.sin(y))
    ref = (B * ws) @ np.exp(xs)[:, None] * ((B * ws) @ np.sin(xs))[None, :]
    assert np.abs(b - ref).max() < 1e-14 * np.abs(ref).max()


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_quadrature_tables_match_assembled_bands(p):
    T = _knots(p, 11, True)
    M, K = bs.assemble_1d_bands(p, T)
    ax = fo.axis_matrices(T, p)
    Md = (ax["B"] * ax["w"]) @ ax["B"].T
    Kd = (ax["D"] * ax["w"]) @ ax["D"].T
    assert np.abs(bs.band_to_dense(M) - Md).max() < 1e-15
    assert np.abs(bs.band_to_dense(K) - Kd).max() < 1e-12 * np.abs(Kd).max()


def test_bad_arguments_raise():
    from poms_b200 import fem
    from poms_b200.stencil import StencilVectorSpace
    V = StencilVectorSpace([8, 9], [3, 3], [False, False], device="cpu")
    good = [_knots(3, 5), _knots(3, 6)]
    with pytest.raises(ValueError):
        fem.load_vector(V, [_knots(3, 6), _knots(3, 6)], 3, None)
    with pytest.raises(ValueError):
        fem.load_vector(V, good, 6, None)
    with pytest.raises(ValueError):
        fem.load_vector(V, good[:1], 3, None)


class _TwoRankSlab:
    """Rank 0 of a two-rank slab partition along axis 1 (only what the space constructor reads)."""
    rank, size, device = 0, 2, None

    def bounds(self, n):
        return 0, n // 2 - 1


def test_slab_partitioned_space_raises():
    from types import SimpleNamespace
    from poms_b200 import fem
    from poms_b200.stencil import StencilVectorSpace
    p, Ns = 2, (8, 6, 5)
    V = StencilVectorSpace([N + p for N in Ns], [p] * 3, [False] * 3, device="cpu", slab=_TwoRankSlab())
    knots = [_knots(p, N) for N in Ns]
    with pytest.raises(NotImplementedError):
        fem.load_vector(V, knots, p, None)
    x = SimpleNamespace(space=V)
    with pytest.raises(NotImplementedError):
        fem.error_norms(x, knots, p, None)
    with pytest.raises(NotImplementedError):
        fem.evaluate(x, knots, p, [np.zeros(1)] * 3)


# ---------------------------------------------------------------------------------------------- GPU
def _space(dev, npts, p):
    from poms_b200.stencil import StencilVectorSpace
    return StencilVectorSpace(list(npts), [p] * len(npts), [False] * len(npts), device=dev)


def _vec(V, arr):
    import torch
    from poms_b200.stencil import StencilVector
    v = StencilVector(V)
    v.data.copy_(torch.as_tensor(arr.reshape(V.npts)))
    return v


def rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


F3 = (lambda x, y, z, m: m.cos(2.0 * x) * (1.0 + y * y) + z * m.sin(3.0 * y) + 0.5)
F2 = (lambda x, y, m: m.cos(2.0 * x) * (1.0 + y * y) + y * m.sin(3.0 * x) + 0.5)


def _f(d, m):
    return (lambda x, y, z: F3(x, y, z, m)) if d == 3 else (lambda x, y: F2(x, y, m))


GPU_CASES = [(p, Ns, g, c) for p in (1, 2, 3, 4, 5)
             for Ns, g, c in (((9, 13, 70), False, 3), ((6, 7, 40), True, 1), ((5, 37), True, None))] + \
            [(3, (8, 8, 8), False, None), (2, (12, 20), False, 3), (4, (33, 9), False, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("p,Ns,graded,chunk", GPU_CASES)
def test_kernels_vs_oracle(dev, p, Ns, graded, chunk):
    import torch
    from poms_b200 import fem
    knots = [_knots(p, N, graded) for N in Ns]
    d = len(Ns)
    V = _space(dev, [N + p for N in Ns], p)
    b = fem.load_vector(V, knots, p, _f(d, torch), plane_chunk=chunk)
    bo = fo.load_vector(knots, p, _f(d, np))
    assert rel(b.data.cpu().numpy(), bo) < 1e-13
    b2 = fem.load_vector(V, knots, p, _f(d, torch), plane_chunk=chunk)
    assert torch.equal(b.flat, b2.flat)                       # deterministic, pad column zero
    assert not b.flat[..., V.npts[-1]:].any()
    x = np.random.default_rng(5).standard_normal(V.npts)
    xv = _vec(V, x)
    if d == 3:
        u = lambda X, Y, Z, m=torch: m.sin(X) * m.cos(Y) + Z
        g = lambda X, Y, Z, m=torch: (m.cos(X) * m.cos(Y), -m.sin(X) * m.sin(Y), 1.0 + 0 * X * Y * Z)
    else:
        u = lambda X, Y, m=torch: m.sin(X) * m.cos(Y)
        g = lambda X, Y, m=torch: (m.cos(X) * m.cos(Y), -m.sin(X) * m.sin(Y))
    e = fem.error_norms(xv, knots, p, u, g, plane_chunk=chunk)
    eo = fo.error_norms(knots, p, x, lambda *X: u(*X, m=np), lambda *X: g(*X, m=np))
    assert abs(e["l2"] - eo["l2"]) < 1e-13 * eo["l2"] and abs(e["h1"] - eo["h1"]) < 1e-13 * eo["h1"], (e, eo)
    e2 = fem.error_norms(xv, knots, p, u, g, plane_chunk=chunk)
    assert e2 == e
    assert fem.error_norms(xv, knots, p, u, plane_chunk=chunk)["h1"] is None


@pytest.mark.gpu
@pytest.mark.parametrize("p,Ns", [(1, (6, 5, 9)), (3, (9, 13, 70)), (5, (5, 6, 7)), (2, (20, 11)), (4, (7, 9))])
def test_identities(dev, p, Ns):
    import torch
    from poms_b200 import fem
    from poms_b200.stencil import KronSumMatrix, StencilVector
    d = len(Ns)
    knots = [_knots(p, N, graded=(a == 0)) for a, N in enumerate(Ns)]
    V = _space(dev, [N + p for N in Ns], p)
    bands = [bs.assemble_1d_bands(p, T) for T in knots]
    Ms, Ks = [m for m, _ in bands], [k for _, k in bands]
    Mop = KronSumMatrix(Ms)
    one = StencilVector(V)
    one.data.fill_(1.0)
    # (1) f = 1: (M1 (x) .. (x) Md) 1
    b = fem.load_vector(V, knots, p, lambda *X: torch.ones(torch.broadcast_shapes(*[t.shape for t in X]),
                                                          dtype=torch.float64, device=dev), plane_chunk=2)
    ref = Mop.dot(one).data.cpu().numpy()
    assert rel(b.data.cpu().numpy(), ref) < 1e-13
    # (2) f = prod g_a, g_a in the spline space: (x)M_a (x)c_a
    cs, gs = [], []
    for a, T in enumerate(knots):
        n = len(T) - p - 1
        c = np.cos(np.arange(n) * (0.7 + a)) + 1.5
        cs.append(c)
        gs.append(BSpline(T, c, p))
    def f(*X):
        out = None
        for a, t in enumerate(X):
            v = torch.as_tensor(gs[a](t.cpu().numpy()), device=dev)
            out = v if out is None else out * v
        return out
    b = fem.load_vector(V, knots, p, f, plane_chunk=3)
    cv = _vec(V, np.einsum(*sum(([c, [a]] for a, c in enumerate(cs)), []), list(range(d))))
    ref = Mop.dot(cv).data.cpu().numpy()
    assert rel(b.data.cpu().numpy(), ref) < 1e-13
    # (3) u = 0: l2^2 = x'Mx, h1^2 = x'(sum K..M)x
    x = np.random.default_rng(2).standard_normal(V.npts)
    xv = _vec(V, x)
    zero = lambda *X: torch.zeros(torch.broadcast_shapes(*[t.shape for t in X]), dtype=torch.float64, device=dev)
    e = fem.error_norms(xv, knots, p, zero, lambda *X: tuple(zero(*X) for _ in X), plane_chunk=1)
    l2sq = float((Mop.dot(xv).data * xv.data).sum())
    h1sq = float((KronSumMatrix(Ms, Ks).dot(xv).data * xv.data).sum())
    assert abs(e["l2"] ** 2 - l2sq) < 1e-12 * l2sq and abs(e["h1"] ** 2 - h1sq) < 1e-12 * h1sq
    # (4) u in the spline space: zero error
    def u(*X):
        out = None
        for a, t in enumerate(X):
            v = torch.as_tensor(gs[a](t.cpu().numpy()), device=dev)
            out = v if out is None else out * v
        return out
    def gu(*X):
        res = []
        for k in range(d):
            out = None
            for a, t in enumerate(X):
                fn = gs[a].derivative() if a == k else gs[a]
                v = torch.as_tensor(fn(t.cpu().numpy()), device=dev)
                out = v if out is None else out * v
            res.append(out)
        return tuple(res)
    e = fem.error_norms(cv, knots, p, u, gu)
    nrm = fem.error_norms(cv, knots, p, zero, lambda *X: tuple(zero(*X) for _ in X))
    assert e["l2"] < 1e-12 * nrm["l2"] and e["h1"] < 1e-12 * nrm["h1"], (e, nrm)


@pytest.mark.gpu
@pytest.mark.parametrize("p,Ns", [(3, (7, 9, 12)), (2, (10, 13)), (5, (6, 5, 7))])
def test_evaluate_vs_scipy(dev, p, Ns):
    from poms_b200 import fem
    d = len(Ns)
    knots = [_knots(p, N, graded=(a == 1)) for a, N in enumerate(Ns)]
    V = _space(dev, [N + p for N in Ns], p)
    x = np.random.default_rng(4).standard_normal(V.npts)
    pts = [np.linspace(0.0, 1.0, 11 + 3 * a) for a in range(d)]
    got = fem.evaluate(_vec(V, x), knots, p, pts).cpu().numpy()
    ref = x
    for a in range(d):
        n = V.npts[a]
        Ba = np.array([BSpline(knots[a], np.eye(n)[i], p)(pts[a]) for i in range(n)])   # (n, np)
        ref = np.moveaxis(np.tensordot(ref, Ba, axes=([a], [0])), -1, a)
    assert rel(got, ref) < 1e-13


@pytest.mark.gpu
def test_bad_values_raise(dev):
    import torch
    from poms_b200 import fem
    p, Ns = 2, (5, 6, 7)
    knots = [_knots(p, N) for N in Ns]
    V = _space(dev, [N + p for N in Ns], p)
    with pytest.raises(ValueError):
        fem.load_vector(V, knots, p, lambda x, y, z: (x * y * z)[:, :, :-1])   # shape
    with pytest.raises(ValueError):
        fem.load_vector(V, knots, p, lambda x, y, z: (x * y * z).float())      # dtype
    with pytest.raises(ValueError):
        fem.load_vector(V, knots, p, lambda x, y, z: (x * y * z).cpu())        # device
    with pytest.raises(ValueError):
        fem.error_norms(fem.load_vector(V, knots, p, lambda x, y, z: x * y * z), knots, p,
                        lambda x, y, z: x * y * z, lambda x, y, z: (x * y * z,))


def manufactured(dev, p, d, Ns, k=1):
    """Errors of u = prod cos(k pi x_a) solved from f = (1 + d k^2 pi^2) u with mg_pcg."""
    import torch
    from poms_b200 import fem
    from poms_b200.mg import Hierarchy, mg_pcg
    kp = k * np.pi
    u = lambda *X: torch.cos(kp * X[0]) * (torch.cos(kp * X[1]) if d == 2 else torch.cos(kp * X[1]) * torch.cos(kp * X[2]))
    f = lambda *X: (1.0 + d * kp * kp) * u(*X)
    def gu(*X):
        c = [torch.cos(kp * t) for t in X]
        s = [-kp * torch.sin(kp * t) for t in X]
        res = []
        for a in range(d):
            out = None
            for b in range(d):
                v = s[b] if a == b else c[b]
                out = v if out is None else out * v
            res.append(out)
        return tuple(res)
    rows = []
    for N in Ns:
        h = Hierarchy(p, [N] * d, device=dev)
        lv = h.levels[0]
        b = fem.load_vector(lv.V, lv.knots, p, f, out=lv.ws("b"))
        x, info = mg_pcg(h, b, tol=1e-12, maxiter=200)
        e = fem.error_norms(x, lv.knots, p, u, gu)
        rows.append((N, e["l2"], e["h1"], info["niter"]))
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("p,d,Ns", [(1, 3, (16, 32, 64)), (2, 3, (8, 16, 32)), (3, 3, (8, 16, 32)), (4, 3, (8, 16)),
                                    (1, 2, (64, 128, 256)), (2, 2, (32, 64, 128)), (3, 2, (16, 32, 64)),
                                    (4, 2, (16, 32)), (5, 2, (8, 16))])
def test_manufactured_convergence(dev, p, d, Ns):
    rows = manufactured(dev, p, d, Ns)
    rows = [r for r in rows if r[1] > 1e-10]
    assert len(rows) >= 2, rows
    (N0, l0, h0, _), (N1, l1, h1, _) = rows[-2], rows[-1]
    ol2, oh1 = np.log(l0 / l1) / np.log(N1 / N0), np.log(h0 / h1) / np.log(N1 / N0)
    assert ol2 >= p + 1 - 0.3 and oh1 >= p - 0.3, (rows, ol2, oh1)
