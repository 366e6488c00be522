"""GPU: the reaction coefficient c, Robin / Neumann boundary terms and fem.boundary_load.

* the operator with c and Robin terms against the oracle (tests/robin_oracle.py), 2-D and 3-D, p = 1..5,
  every epilogue and mat-vec path, with the Toeplitz ranges of the default operator (fast path kept);
* mg_pcg against the oracle hierarchy for a grid of (c, robin), for the glt, glt_poly and jacobi smoothers
  and once with the device setup: iteration counts, histories and solutions;
* boundary_load against the oracle on every face, chunks, accumulation into `out`, determinism;
* manufactured solutions with non-zero normal derivatives (pure Neumann with c > 0, and c = 0 with Robin
  faces): L2 / H1 convergence orders;
* backward Euler for u_t = Lap u with c = 1 / tau, right-hand side M u^n / tau."""
import numpy as np
import pytest

import robin_oracle as ro
from test_gpu_nonuniform import _all_epilogues, _run_all_paths, rel, _space, _vec, _arr

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _knots(p, N):
    from poms_b200 import bsplines as bs
    return bs.make_open_knots(p, N + p)


def _robin(kind, d):
    return {None: None,
            "one": [(10.0, 0.0)] + [(0.0, 0.0)] * (d - 1),
            "one_last": [(0.0, 0.0)] * (d - 1) + [(0.0, 1e3)],
            "all1": [(1.0, 1.0)] * d,
            "big": [(1e3, 1e3)] * d,
            "mixed": [(0.0, 3.0), (0.5, 0.0), (2.0, 7.0)][:d]}[kind]


# ----------------------------------------------------------------------------- operator
SHAPE3 = {1: (37, 147, 297), 2: (68, 129, 260), 3: (37, 147, 297), 4: (21, 60, 200), 5: (21, 60, 200)}
OP_CASES = [(0.0, "one"), (2.5, "mixed"), (1e4, None)]


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("c,kind", OP_CASES)
def test_operator3d_all_paths_vs_oracle(dev, p, c, kind):
    from poms_b200.stencil import KronSumMatrix
    knots = [_knots(p, N) for N in SHAPE3[p]]
    A = KronSumMatrix.poisson(p, knots, c=c, robin=_robin(kind, 3))
    Ao = ro.poisson_operator(p, knots, c, _robin(kind, 3))[0]
    rng0, rng = KronSumMatrix.poisson(p, knots)._toeplitz()[1], A._toeplitz()[1]
    assert np.array_equal(rng[2:], rng0[2:]) and rng[3] - rng[2] > 1 and rng[5] - rng[4] > 64
    _run_all_paths(A, Ao, _space(A.npts, [p] * 3, dev), dev, seed=p)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("c,kind", OP_CASES)
def test_operator2d_vs_oracle(dev, p, c, kind):
    from poms_b200.stencil import KronSumMatrix
    knots = [_knots(p, N) for N in (120, 500)]
    A = KronSumMatrix.poisson(p, knots, c=c, robin=_robin(kind, 2))
    Ao = ro.poisson_operator(p, knots, c, _robin(kind, 2))[0]
    rng0, rng = KronSumMatrix.poisson(p, knots)._toeplitz()[1], A._toeplitz()[1]
    assert np.array_equal(rng[2:], rng0[2:]) and rng[3] - rng[2] > 64
    _all_epilogues(A, Ao, _space(A.npts, [p, p], dev), dev, 3 + p, "2-D")


# ----------------------------------------------------------------------------- MG-PCG
PCG_CASES = [(0.0, "one"), (1e4, None), (1.0, "big"), (1e-3, None), (0.0, "all1"), (0.0, "one_last")]


def _compare_pcg(h, ho, dev, tol=1e-10):
    """Iteration counts, residual histories and solutions.  With the jacobi smoother only the first 5 history
    entries are compared: its ~100-iteration runs amplify rounding in the middle of the history (on the CPU
    oracle alone, scaling lmax by 1 + 1e-13 moves the history of the c = 1e4, 16^3 case by 4e-3 at iteration
    59 of 98, and the solution by 1e-15)."""
    from poms_b200.mg import mg_pcg
    from poms_b200.stencil import StencilVector
    assert len(h.levels) == len(ho.levels)
    for a, b in zip(h.levels[:-1], ho.levels[:-1]):
        assert abs(a.lmax - b["lmax"]) < 1e-9 * b["lmax"]
    npts = h.levels[0].V.npts
    rhs = np.random.default_rng(7).standard_normal(npts)
    b = StencilVector.from_array(h.levels[0].V, rhs)
    x, info = mg_pcg(h, b, tol=tol, maxiter=200)
    xo, io = ho.mg_pcg(rhs, tol=tol, maxiter=200)
    assert info["niter"] == io["niter"] and info["success"] and io["success"], (info["niter"], io["niter"])
    if h.smoother != "jacobi":
        assert np.allclose(info["history"], io["history"], rtol=1e-6)
    assert np.allclose(info["history"][:5], io["history"][:5], rtol=1e-10)
    assert rel(_arr(x), xo) < 1e-9
    return info["niter"]


@pytest.mark.parametrize("smoother", ["glt", "glt_poly", "jacobi"])
@pytest.mark.parametrize("p,N", [(3, (32, 32)), (2, (16, 16, 16)), (1, (32, 16))])
@pytest.mark.parametrize("c,kind", PCG_CASES)
def test_mg_pcg_vs_oracle(dev, p, N, smoother, c, kind):
    from poms_b200.mg import Hierarchy
    if smoother == "glt_poly" and p == 1:
        pytest.skip("T[m_0] is the identity for p = 1: nothing to approximate")
    robin = _robin(kind, len(N))
    h = Hierarchy(p, list(N), device=dev, smoother=smoother, nu=1, c=c, robin=robin)
    ho = ro.MGHierarchy(p, list(N), smoother=smoother, nu=1, c=c, robin=robin)
    # c = 1e-3 without Robin terms is nearly singular: the true relative residual of fp64 floors near 1e-10
    _compare_pcg(h, ho, dev, tol=1e-8 if c == 1e-3 else 1e-10)


@pytest.mark.parametrize("c,kind", [(0.0, "one"), (1.0, "big")])
def test_mg_pcg_device_setup_vs_oracle(dev, c, kind):
    from poms_b200.mg import Hierarchy
    robin = _robin(kind, 3)
    h = Hierarchy(3, [16, 16, 16], device=dev, c=c, robin=robin, setup="device")
    hh = Hierarchy(3, [16, 16, 16], device=dev, c=c, robin=robin)
    for a, b in zip(h.levels, hh.levels):
        for x, y in zip(a.A.Ks + a.A.Ms, b.A.Ks + b.A.Ms):
            assert np.abs(x - y).max() < 1e-12 * np.abs(y).max()
    _compare_pcg(h, ro.MGHierarchy(3, [16, 16, 16], c=c, robin=robin), dev)


def test_defaults_unchanged(dev):
    """c = 1 and no Robin terms: the same bands, lambda_max and iterations as the hierarchy without them."""
    from poms_b200.mg import Hierarchy, mg_pcg
    from poms_b200.stencil import StencilVector
    h0 = Hierarchy(3, [32, 32, 32], device=dev, smoother="glt_poly")
    h1 = Hierarchy(3, [32, 32, 32], device=dev, smoother="glt_poly", c=1.0, robin=[(0.0, 0.0)] * 3)
    for a, b in zip(h0.levels, h1.levels):
        assert all(np.array_equal(x, y) for x, y in zip(a.A.Ks + a.A.Ms, b.A.Ks + b.A.Ms))
        assert getattr(a, "lmax", None) == getattr(b, "lmax", None)
    its = []
    for h in (h0, h1):
        b = StencilVector(h.levels[0].V)
        b.data.fill_(1.0)
        its.append(mg_pcg(h, b, tol=1e-10, maxiter=100)[1]["niter"])
    assert its[0] == its[1]


# ----------------------------------------------------------------------------- boundary_load
G3 = lambda x, y, m: m.exp(x) * m.cos(2.0 * y) + x * y + 0.25
G2 = lambda x, m: m.exp(x) + x ** 3 - 0.5

BL_CASES = [(p, Ns, ch) for p in (1, 2, 3, 4, 5) for Ns, ch in (((9, 13, 70), None), ((6, 7, 40), 1), ((5, 37), None))] \
    + [(3, (8, 35, 9), 3), (2, (12, 20), 1), (4, (33, 9, 6), 2)]


@pytest.mark.parametrize("p,Ns,chunk", BL_CASES)
def test_boundary_load_vs_oracle(dev, p, Ns, chunk):
    from poms_b200 import fem
    from poms_b200.stencil import StencilVector
    d = len(Ns)
    knots = [_knots(p, N) for N in Ns]
    if d == 3:
        knots[1][p + 1:Ns[1] + p] = knots[1][p + 1:Ns[1] + p] ** 1.5           # one graded axis
    V = _space([N + p for N in Ns], [p] * d, dev)
    gt = (lambda x, y: G3(x, y, torch)) if d == 3 else (lambda x: G2(x, torch))
    gn = (lambda x, y: G3(x, y, np)) if d == 3 else (lambda x: G2(x, np))
    acc = StencilVector(V)
    acc.data.fill_(1.0)
    total = np.ones(V.npts)
    for axis in range(d):
        for side in (0, 1):
            b = fem.boundary_load(V, knots, p, gt, axis, side, plane_chunk=chunk)
            bo = ro.boundary_load(knots, p, gn, axis, side)
            assert rel(b.data.cpu().numpy(), bo) < 1e-13, (axis, side)
            assert not b.flat[..., V.npts[-1]:].any()
            b2 = fem.boundary_load(V, knots, p, gt, axis, side, plane_chunk=chunk)
            assert torch.equal(b.flat, b2.flat)
            if chunk is not None:
                b3 = fem.boundary_load(V, knots, p, gt, axis, side)
                assert rel(b3.data.cpu().numpy(), bo) < 1e-13
            r = fem.boundary_load(V, knots, p, gt, axis, side, out=acc, plane_chunk=chunk)
            assert r is acc
            total = total + bo
    assert rel(acc.data.cpu().numpy(), total) < 1e-13
    assert not acc.flat[..., V.npts[-1]:].any()
    # a constant g = 1 adds the face's mass row sums: sum of the plane = face area
    one = (lambda x, y: torch.ones_like(x * y)) if d == 3 else (lambda x: torch.ones_like(x))
    b = fem.boundary_load(V, knots, p, one, 0, 1, plane_chunk=chunk)
    assert abs(float(b.data.sum()) - 1.0) < 1e-13


def test_boundary_load_bad_values(dev):
    from poms_b200 import fem
    p, Ns = 2, (5, 6, 7)
    knots = [_knots(p, N) for N in Ns]
    V = _space([N + p for N in Ns], [p] * 3, dev)
    for g in (lambda x, y: (x * y)[:, :-1], lambda x, y: (x * y).float(), lambda x, y: (x * y).cpu(),
              lambda x, y: (x * y).cpu().numpy()):
        with pytest.raises(ValueError):
            fem.boundary_load(V, knots, p, g, 2, 0)


# ----------------------------------------------------------------------------- manufactured solutions
K3 = (1.0, 2.0, 3.0)


def _exp_solution(d):
    """u = exp(k . x) / scale: non-zero normal derivative on every face."""
    k = K3[:d]
    scale = float(np.exp(sum(k)))
    u = lambda *X: torch.exp(sum(ki * x for ki, x in zip(k, X))) / scale
    gu = lambda *X: tuple(ki * u(*X) for ki in k)
    return k, scale, u, gu


def _face_g(k, scale, axis, side, alpha, d):
    """g = du/dn + alpha u on the face x_axis = side, as a function of the other coordinates."""
    kn = k[axis] if side == 1 else -k[axis]
    fixed = float(np.exp(k[axis] * side))
    others = [k[b] for b in range(d) if b != axis]

    def g(*X):
        v = torch.exp(sum(ki * x for ki, x in zip(others, X))) * (fixed / scale)
        return (kn + alpha) * v
    return g


def _manufactured(dev, p, d, Ns, c, robin):
    from poms_b200 import fem
    from poms_b200.mg import Hierarchy, mg_pcg
    k, scale, u, gu = _exp_solution(d)
    lam = sum(ki * ki for ki in k)
    f = lambda *X: (c - lam) * u(*X)
    rows = []
    for N in Ns:
        h = Hierarchy(p, [N] * d, device=dev, c=c, robin=robin)
        lv = h.levels[0]
        b = fem.load_vector(lv.V, lv.knots, p, f, out=lv.ws("b"))
        for axis in range(d):
            for side in (0, 1):
                alpha = robin[axis][side] if robin is not None else 0.0
                fem.boundary_load(lv.V, lv.knots, p, _face_g(k, scale, axis, side, alpha, d), axis, side, out=b)
        x, info = mg_pcg(h, b, tol=1e-12, maxiter=200)
        assert info["success"], info["niter"]
        e = fem.error_norms(x, lv.knots, p, u, gu)
        rows.append((N, e["l2"], e["h1"], info["niter"]))
    return rows


MANUF = [(1, 3, (16, 32, 64)), (2, 3, (8, 16, 32)), (3, 3, (8, 16, 32)), (4, 3, (8, 16)),
         (1, 2, (64, 128, 256)), (2, 2, (32, 64, 128)), (3, 2, (16, 32, 64)), (4, 2, (8, 16)), (5, 2, (6, 12))]


@pytest.mark.parametrize("p,d,Ns", MANUF)
@pytest.mark.parametrize("case", ["neumann", "robin"])
def test_manufactured_convergence(dev, p, d, Ns, case):
    """neumann: du/dn = g on every face, c = 2.  robin: c = 0, du/dn + alpha u = g on three faces (one of
    them on the last axis), du/dn = g on the others."""
    if case == "neumann":
        c, robin = 2.0, None
    else:
        c, robin = 0.0, [(2.0, 0.0), (0.0, 5.0), (0.0, 1.0)][:d - 1] + [(0.0, 1.0)]
    rows = _manufactured(dev, p, d, Ns, c, robin)
    rows = [r for r in rows if r[1] > 1e-10]
    assert len(rows) >= 2, rows
    (N0, l0, h0, _), (N1, l1, h1, _) = rows[-2], rows[-1]
    ol2, oh1 = np.log(l0 / l1) / np.log(N1 / N0), np.log(h0 / h1) / np.log(N1 / N0)
    assert ol2 >= p + 1 - 0.25 and oh1 >= p - 0.25, (rows, ol2, oh1)


# ----------------------------------------------------------------------------- backward Euler
@pytest.mark.parametrize("d,p,N", [(2, 3, 32), (3, 3, 16)])
def test_backward_euler_heat_equation(dev, d, p, N):
    """u_t = Lap u, du/dn = 0, u0 = prod cos(pi x_a): (M / tau + K) u^{n+1} = M u^n / tau is the hierarchy
    with c = 1 / tau; the first right-hand side is int u0 phi_i / tau.  The iterates follow the discrete
    decay (1 + lambda tau)^-n u0 up to the spatial error, and the exact decay exp(-lambda t) to first order
    in tau."""
    from poms_b200 import fem
    from poms_b200.mg import Hierarchy, mg_pcg
    from poms_b200.stencil import KronSumMatrix
    lam = d * np.pi ** 2
    u0 = lambda *X: torch.cos(np.pi * X[0]) * torch.cos(np.pi * X[1]) * (torch.cos(np.pi * X[2]) if d == 3 else 1.0)

    def run(tau, steps):
        h = Hierarchy(p, [N] * d, device=dev, c=1.0 / tau)
        lv = h.levels[0]
        M = KronSumMatrix(lv.A.mass_bands)
        b = fem.load_vector(lv.V, lv.knots, p, lambda *X: u0(*X) / tau)
        errs = []
        for n in range(1, steps + 1):
            x, info = mg_pcg(h, b, tol=1e-12, maxiter=100)
            assert info["success"]
            x = x.copy()
            b = M.dot(x) * (1.0 / tau)
            disc = (1.0 + lam * tau) ** -n
            exact = np.exp(-lam * n * tau)
            e_disc = fem.error_norms(x, lv.knots, p, lambda *X: disc * u0(*X))["l2"]
            e_ex = fem.error_norms(x, lv.knots, p, lambda *X: exact * u0(*X))["l2"]
            errs.append((e_disc, e_ex))
        return errs

    norm0 = 0.5 ** (d / 2.0)                       # ||u0||_L2 on the unit cube
    e1 = run(0.01, 4)
    e2 = run(0.005, 8)
    assert max(e for e, _ in e1 + e2) < 1e-4 * norm0
    ratio = e1[-1][1] / e2[-1][1]                   # same final time 0.04
    assert 1.7 < ratio < 2.2, (e1, e2)
    assert e1[-1][1] < lam * lam * 0.04 * 0.01 * norm0
