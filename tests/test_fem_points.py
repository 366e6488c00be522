"""poms_b200.fem.evaluate_points / deposit: particle coupling on B-spline spaces.

CPU: the oracle's point design matrices against scipy BSpline (values and derivatives, on breakpoints and at the
ends too), argument checks, slab-partitioned spaces, and the host-side argument checks of the C entries.
GPU (p = 1..5, 2-D and 3-D, uniform, graded and C0 knots): evaluate_points against scipy and against
fem.evaluate, linear reproduction, the adjoint identity between deposit and evaluate_points, deposit of the
Gauss points against fem.load_vector, deposit against the oracle (chunks, a crowded cell, empty cells, m = 0
and 1), determinism, and a deposit -> mg_pcg -> gradient round trip against a dense NumPy solve."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from scipy.interpolate import BSpline

import points_oracle as po
from poms_b200 import bsplines as bs


def _knots(p, N, kind="uniform"):
    """Open knots of N elements on [0, 1]: uniform, graded (T^1.5) or with one interior breakpoint of
    multiplicity p (a C0 joint)."""
    if kind == "c0":
        br = np.arange(1, N) / N
        inner = np.sort(np.concatenate([br, np.full(p - 1, br[len(br) // 2])]))
        return np.concatenate([np.zeros(p + 1), inner, np.ones(p + 1)])
    T = bs.make_open_knots(p, N + p)
    if kind == "graded":
        T[p + 1:N + p] = T[p + 1:N + p] ** 1.5
    return T


def _scipy_matrices(T, p, x):
    n = len(T) - p - 1
    B = np.array([BSpline(T, np.eye(n)[i], p)(x) for i in range(n)]).T
    D = np.array([BSpline(T, np.eye(n)[i], p).derivative()(x) for i in range(n)]).T
    return B, D


def _test_points(rng, knots, m):
    """Random points, every breakpoint of every axis (the other coordinates random) and the corners."""
    d = len(knots)
    P = [rng.uniform(0.0, 1.0, (m, d))]
    for a, T in enumerate(knots):
        br = np.unique(T)
        q = rng.uniform(0.0, 1.0, (len(br), d))
        q[:, a] = br
        P.append(q)
    P.append(np.array(np.meshgrid(*[[0.0, 1.0]] * d, indexing="ij")).reshape(d, -1).T)
    return np.concatenate(P)


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("kind", ["uniform", "graded", "c0"])
def test_oracle_point_matrices_vs_scipy(p, kind):
    T = _knots(p, 7, kind)
    x = np.concatenate([np.random.default_rng(p).uniform(0, 1, 200), np.unique(T)])
    B, D = po.point_matrices(T, p, x)
    Bs, Ds = _scipy_matrices(T, p, x)
    assert np.abs(B - Bs).max() < 1e-14 and np.abs(D - Ds).max() < 1e-12 * np.abs(Ds).max()
    assert np.abs(B.sum(axis=1) - 1.0).max() < 1e-14                  # partition of unity


def _cpu_space(npts, p):
    from poms_b200.stencil import StencilVectorSpace
    return StencilVectorSpace(list(npts), [p] * len(npts), [False] * len(npts), device="cpu")


def test_bad_points_raise():
    from poms_b200 import fem
    p, Ns = 2, (5, 4, 6)
    knots = [_knots(p, N) for N in Ns]
    V = _cpu_space([N + p for N in Ns], p)
    x = SimpleNamespace(space=V, _buf=torch.zeros(1))
    good = torch.full((4, 3), 0.5, dtype=torch.float64)
    w = torch.ones(4, dtype=torch.float64)
    bad_points = [good.float(), good.numpy(), good.to("meta"), good[:, :2], good[0], good.reshape(2, 6)]
    for v, a in ((float("nan"), 0), (float("inf"), 1), (-float("inf"), 2), (-1e-12, 0), (1.0 + 1e-12, 2)):
        q = good.clone()
        q[2, a] = v
        bad_points.append(q)
    bad_points.append(torch.zeros(1, 3, dtype=torch.float64).expand(1 << 31, 3))         # m = 2^31 (no memory)
    for q in bad_points:
        with pytest.raises(ValueError):
            fem.evaluate_points(x, knots, p, q)
        with pytest.raises(ValueError):
            fem.deposit(V, knots, p, q, w if q.ndim == 2 and q.shape[0] == 4 else w[:1])
    for ww in (w.float(), w[:3], w.reshape(4, 1), w.to("meta"), w.numpy()):
        with pytest.raises(ValueError):
            fem.deposit(V, knots, p, good, ww)
    with pytest.raises(ValueError):
        fem.deposit(V, knots, p, good, w, plane_chunk=0)
    with pytest.raises(ValueError):
        fem.evaluate_points(x, knots, 6, good)
    V2 = _cpu_space([N + p for N in Ns[:2]], p)
    with pytest.raises(ValueError):                                   # 3 coordinates on a 2-D space
        fem.deposit(V2, knots[:2], p, good, w)


def test_slab_partitioned_space_raises():
    from poms_b200 import fem
    from poms_b200.stencil import StencilVectorSpace

    class TwoRankSlab:
        rank, size, device = 0, 2, None

        def bounds(self, n):
            return 0, n // 2 - 1

    p, Ns = 2, (8, 6, 5)
    V = StencilVectorSpace([N + p for N in Ns], [p] * 3, [False] * 3, device="cpu", slab=TwoRankSlab())
    knots = [_knots(p, N) for N in Ns]
    pts = torch.full((2, 3), 0.5, dtype=torch.float64)
    with pytest.raises(NotImplementedError):
        fem.evaluate_points(SimpleNamespace(space=V), knots, p, pts)
    with pytest.raises(NotImplementedError):
        fem.deposit(V, knots, p, pts, torch.ones(2, dtype=torch.float64))


def test_c_entries_check_arguments_before_cuda():
    """Bad arguments give a negative status (minus the argument index) without a CUDA call."""
    from poms_b200 import _lib
    L = _lib.lib()
    T = np.ascontiguousarray(_knots(3, 5))
    t = T.ctypes.data
    # poms_points_eval(x, ld, pld, n1, n2, n3, p, T1, T2, T3, pts, d, m, u, g, stream)
    assert L.poms_points_eval(None, 8, 64, 8, 8, 8, 3, t, t, t, 1, 3, 1, 1, None, None) == -1
    assert L.poms_points_eval(1, 7, 64, 8, 8, 8, 3, t, t, t, 1, 3, 1, 1, None, None) == -2      # ld < n3
    assert L.poms_points_eval(1, 8, 64, 8, 8, 8, 6, t, t, t, 1, 3, 1, 1, None, None) == -7      # p
    assert L.poms_points_eval(1, 8, 64, 3, 8, 8, 3, t, t, t, 1, 3, 1, 1, None, None) == -4      # n1 <= p
    assert L.poms_points_eval(1, 8, 64, 8, 8, 8, 3, t, None, t, 1, 3, 1, 1, None, None) == -5   # 2-D needs n2 = 1
    assert L.poms_points_eval(1, 8, 64, 8, 8, 8, 3, t, t, t, 1, 2, 1, 1, None, None) == -12     # d
    assert L.poms_points_eval(1, 8, 64, 8, 8, 8, 3, t, t, t, 1, 3, 1 << 31, 1, None, None) == -13
    assert L.poms_points_eval(1, 8, 64, 8, 8, 8, 3, t, t, t, None, 3, 1, 1, None, None) == -11
    assert b"bad argument" in L.poms_last_error()
    assert L.poms_points_eval(1, 8, 64, 8, 8, 8, 3, t, t, t, None, 3, 0, None, None, None) == 0  # m = 0: no launch
    # poms_points_locate(pts, d, m, n1, n2, n3, p, T1, T2, T3, key, stream)
    assert L.poms_points_locate(1, 3, -1, 8, 8, 8, 3, t, t, t, 1, None) == -3
    assert L.poms_points_locate(None, 3, 4, 8, 8, 8, 3, t, t, t, 1, None) == -1
    assert L.poms_points_locate(1, 3, 4, 8, 8, 8, 3, None, t, t, 1, None) == -8
    # poms_points_moments(pts, w, d, perm, offs, c1_lo, c1_hi, n1, n2, n3, p, T1, T2, T3, mom, stream)
    assert L.poms_points_moments(1, None, 3, 1, 1, 0, 5, 8, 8, 8, 3, t, t, t, 1, None) == -1
    assert L.poms_points_moments(1, 1, 3, 1, 1, 0, 6, 8, 8, 8, 3, t, t, t, 1, None) == -6       # c1_hi > n1 - p
    assert L.poms_points_moments(1, 1, 3, 1, 1, 2, 2, 8, 8, 8, 3, t, t, t, 1, None) == -6
    # poms_points_assemble(mom, c1_lo, c1_hi, n1, n2, n3, p, y, ld, pld, store_from, stream)
    assert L.poms_points_assemble(1, 0, 5, 8, 8, 8, 3, None, 8, 64, 0, None) == -1
    assert L.poms_points_assemble(1, 0, 5, 8, 8, 8, 3, 1, 8, 63, 0, None) == -9                # pld < n2 ld
    assert L.poms_points_assemble(1, 0, 5, 8, 8, 8, 3, 1, 8, 64, 9, None) == -11
    assert L.poms_points_assemble(1, 0, 5, 8, 8, 8, 0, 1, 8, 64, 0, None) == -7


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _space(dev, npts, p):
    from poms_b200.stencil import StencilVectorSpace
    return StencilVectorSpace(list(npts), [p] * len(npts), [False] * len(npts), device=dev)


def _vec(V, arr):
    from poms_b200.stencil import StencilVector
    v = StencilVector(V)
    v.data.copy_(torch.as_tensor(arr.reshape(V.npts)))
    return v


def _t(a, dev):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device=dev)


SHAPES = {3: (6, 5, 7), 2: (9, 11)}
GPU_CASES = [(p, d, kind) for p in (1, 2, 3, 4, 5) for d in (3, 2) for kind in ("uniform", "graded", "c0")]


def _setup(dev, p, d, kind):
    knots = [_knots(p, N, kind) for N in SHAPES[d]]
    V = _space(dev, [len(T) - p - 1 for T in knots], p)
    return knots, V


@pytest.mark.gpu
@pytest.mark.parametrize("p,d,kind", GPU_CASES)
def test_evaluate_points(dev, p, d, kind):
    from poms_b200 import fem
    knots, V = _setup(dev, p, d, kind)
    rng = np.random.default_rng(p + 7 * d)
    x = rng.standard_normal(V.npts)
    xv = _vec(V, x)
    # (1) against scipy: random points, every breakpoint, both ends
    P = _test_points(rng, knots, 400)
    u, g = fem.evaluate_points(xv, knots, p, _t(P, dev), grad=True)
    u, g = u.cpu().numpy(), g.cpu().numpy()
    mats = [_scipy_matrices(T, p, P[:, a]) for a, T in enumerate(knots)]
    uo = po._at_points([B for B, _ in mats], x)
    go = np.stack([po._at_points([mats[b][1] if b == a else mats[b][0] for b in range(d)], x)
                   for a in range(d)], axis=1)
    assert rel(u, uo) < 1e-13 and rel(g, go) < 1e-11
    assert torch.equal(fem.evaluate_points(xv, knots, p, _t(P, dev)).cpu(), torch.as_tensor(u))
    # (2) on a tensor grid: the same values as fem.evaluate
    axes = [np.linspace(0.0, 1.0, 9 + 2 * a) for a in range(d)]
    grid = np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, d)
    ug = fem.evaluate_points(xv, knots, p, _t(grid, dev)).cpu().numpy()
    ue = fem.evaluate(xv, knots, p, axes).cpu().numpy().reshape(-1)
    assert rel(ug, ue) < 1e-14
    # (3) linear reproduction from the Greville abscissae
    c = np.array([0.3, -1.2, 0.7, 2.1])[:d + 1]
    gr = [np.array([T[i + 1:i + p + 1].mean() for i in range(len(T) - p - 1)]) for T in knots]
    lin = c[0] + sum(c[a + 1] * gr[a].reshape([-1 if b == a else 1 for b in range(d)]) for a in range(d))
    ul, gl = fem.evaluate_points(_vec(V, np.broadcast_to(lin, V.npts).copy()), knots, p, _t(P, dev), grad=True)
    assert np.abs(ul.cpu().numpy() - (c[0] + P @ c[1:])).max() < 1e-13
    assert np.abs(gl.cpu().numpy() - c[1:]).max() < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("p,d,kind", GPU_CASES)
def test_deposit(dev, p, d, kind):
    from poms_b200 import fem
    from poms_b200.stencil import StencilVector
    knots, V = _setup(dev, p, d, kind)
    rng = np.random.default_rng(3 * p + d)
    P = _test_points(rng, knots, 3000)
    w = rng.standard_normal(len(P))
    Pt, wt = _t(P, dev), _t(w, dev)
    bo = po.deposit(knots, p, P, w)
    # (6) against the oracle, chunks of 1, 3 and all cell planes; every owned entry overwritten, pad zero
    b = None
    for ch in (1, 3, None):
        out = StencilVector(V)
        out.data.fill_(np.nan)
        b = fem.deposit(V, knots, p, Pt, wt, out=out, plane_chunk=ch)
        assert rel(b.data.cpu().numpy(), bo) < 1e-13, ch
        assert not b.flat[..., V.npts[-1]:].any()
    # (7) deterministic; a permuted input agrees
    b2 = fem.deposit(V, knots, p, Pt, wt, plane_chunk=None)
    assert torch.equal(b.flat, b2.flat)
    perm = torch.as_tensor(rng.permutation(len(P)), device=dev)
    b3 = fem.deposit(V, knots, p, Pt[perm], wt[perm])
    assert rel(b3.data.cpu().numpy(), bo) < 1e-13
    # (4) adjointness: <deposit(P, w), x> = sum_k w_k u_h(P_k)
    x = rng.standard_normal(V.npts)
    uP = fem.evaluate_points(_vec(V, x), knots, p, Pt)
    lhs = float((b.data * _t(x, dev)).sum())
    terms = wt * uP
    assert abs(lhs - float(terms.sum())) < 1e-13 * float(terms.abs().sum())
    # (5) the tensor Gauss points with weights w_q f(x_q) give fem.load_vector(f)
    tabs = [bs.quadrature_tables(T, p) for T in knots]
    xs = [t["x"].reshape(-1) for t in tabs]
    ws = [t["w"].reshape(-1) for t in tabs]
    G = np.stack(np.meshgrid(*xs, indexing="ij"), axis=-1).reshape(-1, d)
    W = np.einsum(*sum(([wa, [a]] for a, wa in enumerate(ws)), []), list(range(d))).reshape(-1)
    f = (lambda X, m=np: m.cos(2.0 * X[0]) * (1.0 + X[1] ** 2) + X[-1] * m.sin(3.0 * X[1]) + 0.5)
    bq = fem.deposit(V, knots, p, _t(G, dev), _t(W * f(G.T), dev), plane_chunk=2)
    bl = fem.load_vector(V, knots, p, lambda *X: f(X, torch))
    assert rel(bq.data.cpu().numpy(), bl.data.cpu().numpy()) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("p,d", [(3, 3), (5, 3), (1, 2), (4, 2)])
def test_deposit_crowded_and_tiny(dev, p, d):
    """>= 10^5 points in one cell beside empty cells; m = 0 and m = 1."""
    from poms_b200 import fem
    from poms_b200.stencil import StencilVector
    knots, V = _setup(dev, p, d, "graded")
    rng = np.random.default_rng(11)
    lo = [np.unique(T)[2] for T in knots]
    hi = [np.unique(T)[3] for T in knots]
    P = rng.uniform(lo, hi, (100_003, d))
    w = rng.uniform(-1.0, 1.0, len(P))
    b = fem.deposit(V, knots, p, _t(P, dev), _t(w, dev), plane_chunk=2)
    assert rel(b.data.cpu().numpy(), po.deposit(knots, p, P, w)) < 1e-13
    for m in (0, 1):
        out = StencilVector(V)
        out.data.fill_(np.nan)
        b = fem.deposit(V, knots, p, _t(P[:m], dev), _t(w[:m], dev), out=out)
        assert rel(b.data.cpu().numpy(), po.deposit(knots, p, P[:m], w[:m])) < 1e-13 if m else not b.flat.any()
        assert not b.flat[..., V.npts[-1]:].any()
    u0, g0 = fem.evaluate_points(_vec(V, np.ones(V.npts)), knots, p, _t(P[:0], dev), grad=True)
    assert u0.shape == (0,) and g0.shape == (0, d)


@pytest.mark.gpu
@pytest.mark.parametrize("p,d,N", [(3, 2, 16), (2, 3, 8)])
def test_particles_solve_field(dev, p, d, N):
    """Deposit particle charges, solve -Lap u + u = b with mg_pcg, evaluate grad u_h at the particles; the
    same chain with the oracle and a dense NumPy solve of the Kronecker-sum operator."""
    from poms_b200 import fem
    from poms_b200.mg import Hierarchy, mg_pcg
    h = Hierarchy(p, [N] * d, device="cuda")          # the default device: no index
    lv = h.levels[0]
    rng = np.random.default_rng(5)
    P = rng.uniform(0.0, 1.0, (4000, d))
    w = rng.uniform(0.5, 1.5, len(P))
    b = fem.deposit(lv.V, lv.knots, p, _t(P, dev), _t(w, dev), out=lv.ws("b"))
    x, info = mg_pcg(h, b, tol=1e-12, maxiter=200)
    u, g = fem.evaluate_points(x, lv.knots, p, _t(P, dev), grad=True)
    M, K = zip(*[(bs.band_to_dense(m), bs.band_to_dense(k)) for m, k in (bs.assemble_1d_bands(p, T) for T in lv.knots)])
    A = 0
    for a in range(d + 1):                    # sum_a K_a (x) M_others, plus M (x) .. (x) M
        mats = [K[b] if b == a else M[b] for b in range(d)]
        term = mats[0]
        for mm in mats[1:]:
            term = np.kron(term, mm)
        A = A + term
    xd = np.linalg.solve(A, po.deposit(lv.knots, p, P, w).reshape(-1)).reshape(lv.V.npts)
    uo, go = po.evaluate_points(lv.knots, p, xd, P)
    assert rel(g.cpu().numpy(), go) < 1e-9 and rel(u.cpu().numpy(), uo) < 1e-9, info
