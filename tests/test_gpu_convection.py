"""GPU: constant-velocity convection -Lap u + beta . grad u + c u through mg_gmres.

* the operator with beta against the oracle (tests/convection_oracle.py), 2-D and 3-D, p = 1..5, every epilogue
  and mat-vec path on shapes with interior and ragged tiles; the dispatch asserted: a velocity with a non-zero
  component on axis 2 or 3 makes the interior rows non-symmetric, so the 3-D kernel runs variant 0 and the 2-D
  kernel its sym = 0 form;
* mg_gmres against the oracle restatement (GMRES on the oracle operator, one V-cycle of the oracle hierarchy as
  the preconditioner): identical iteration counts, solutions to 1e-10, for three velocities, c = 0 with Robin
  faces and c = 1, the glt, glt_poly and jacobi smoothers, host and device setup;
* the device advection band against the host band;
* a manufactured solution with non-zero normal flux: L2 order p+1, H1 order p;
* determinism, h.op without beta, and mg_pcg refusing a non-symmetric hierarchy."""
import numpy as np
import pytest

import convection_oracle as co
import robin_oracle as ro
from test_gpu_nonuniform import _all_epilogues, _run_all_paths, rel, _space, _arr, tma_sym
from test_robin_reaction import _knots as _knots_kind

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


def _robin_for(beta, extra=0.0):
    """alpha = |beta_a| / 2 + extra on each inflow face (beta . n < 0), 0 on the outflow faces."""
    return [((0.5 * b + extra, 0.0) if b > 0 else (0.0, -0.5 * b + extra)) for b in beta]


BETAS3 = [(1.0, 0.0, 0.0), (10.0, -5.0, 3.0), (50.0, 20.0, 0.0)]


# ----------------------------------------------------------------------------- operator
SHAPE3 = {1: (37, 147, 297), 2: (68, 129, 260), 3: (37, 147, 297), 4: (21, 60, 200), 5: (21, 60, 200)}


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("beta", BETAS3)
def test_operator3d_all_paths_vs_oracle(dev, p, beta):
    from poms_b200.stencil import KronSumMatrix
    knots = [_knots(p, N) for N in SHAPE3[p]]
    robin = _robin_for(beta)
    A = KronSumMatrix.poisson(p, knots, c=1.0, robin=robin, beta=beta)
    Ao = co.poisson_operator(p, knots, 1.0, robin, list(beta))[0]
    rng0, rng = KronSumMatrix.poisson(p, knots)._toeplitz()[1], A._toeplitz()[1]
    assert np.array_equal(rng, rng0) and rng[5] - rng[4] > 64
    # velocity on an inner axis: non-symmetric Toeplitz rows there, the kernel takes variant 0
    assert tma_sym(A) == (beta[1] == 0.0 and beta[2] == 0.0)
    _run_all_paths(A, Ao, _space(A.npts, [p] * 3, dev), dev, seed=p)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("beta", [(1.0, 0.0), (10.0, -5.0), (0.0, 30.0)])
def test_operator2d_vs_oracle(dev, p, beta):
    from poms_b200.stencil import KronSumMatrix
    knots = [_knots(p, N) for N in (120, 500)]
    robin = _robin_for(beta)
    A = KronSumMatrix.poisson(p, knots, c=1.0, robin=robin, beta=beta)
    Ao = co.poisson_operator(p, knots, 1.0, robin, list(beta))[0]
    assert A._toeplitz()[1][3] - A._toeplitz()[1][2] > 64
    assert tma_sym(A) == (beta[1] == 0.0)               # False: the 2-D kernel runs with sym = 0
    _all_epilogues(A, Ao, _space(A.npts, [p, p], dev), dev, 3 + p, "2-D")


# ----------------------------------------------------------------------------- mg_gmres
def _compare_gmres(h, ho, beta, c, robin, dev, maxiter=400, converges=True):
    from poms_b200.mg import mg_gmres
    from poms_b200.stencil import StencilVector
    p = h.p
    assert len(h.levels) == len(ho.levels) >= 2
    for a, b in zip(h.levels[:-1], ho.levels[:-1]):
        assert abs(a.lmax - b["lmax"]) < 1e-9 * b["lmax"]
    knots = ho.levels[0]["knots"]
    Ao = co.poisson_operator(p, knots, c, robin, list(beta))[0]
    npts = h.levels[0].V.npts
    rhs = np.random.default_rng(7).standard_normal(npts)
    b = StencilVector.from_array(h.levels[0].V, rhs)
    x, info = mg_gmres(h, b, tol=1e-10, maxiter=maxiter)
    xo, io = co.mg_gmres(ho, Ao, rhs, tol=1e-10, maxiter=maxiter)
    assert info["niter"] == io["niter"], (info["niter"], io["niter"])
    assert info["success"] == io["success"] == converges, (info["success"], io["success"])
    assert rel(_arr(x), xo) < 1e-10
    if not converges:
        return info["niter"]
    r = rhs - Ao.dot(_arr(x))
    assert np.sqrt(np.vdot(r, r)) <= 1e-10 * np.linalg.norm(rhs) * (1 + 1e-9)
    return info["niter"]


GM_CASES = [(beta, c) for beta in BETAS3 for c in (0.0, 1.0)]


@pytest.mark.parametrize("smoother", ["glt", "glt_poly", "jacobi"])
@pytest.mark.parametrize("beta,c", GM_CASES)
def test_mg_gmres_vs_oracle(dev, smoother, beta, c):
    """3-D p = 3, 16^3 elements (two levels).  c = 0: the Robin faces alpha = |beta_a| / 2 (+0.5 on the faces of
    axes without velocity, so that some alpha > 0 there too) make the operator definite."""
    from poms_b200.mg import Hierarchy
    p, N = 3, [16, 16, 16]
    robin = _robin_for(beta, 0.0) if c == 1.0 else [r if b != 0.0 else (0.5, 0.0)
                                                      for r, b in zip(_robin_for(beta), beta)]
    h = Hierarchy(p, N, device=dev, smoother=smoother, c=c, robin=robin, beta=beta)
    ho = ro.MGHierarchy(p, N, smoother=smoother, c=c, robin=robin)
    # The Jacobi-Chebyshev V-cycle is the weakest preconditioner: about 200 (beta = (1, 0, 0)) and 440
    # (beta = (10, -5, 3)) iterations.  At beta = (50, 20, 0) GMRES(30) stagnates with it (no convergence in
    # 3000 iterations, on the GPU and in the oracle alike): there the first 300 iterations are compared.
    stagnates = smoother == "jacobi" and beta[0] == 50.0
    n = _compare_gmres(h, ho, beta, c, robin, dev, maxiter=300 if stagnates else 600, converges=not stagnates)
    print("smoother", smoother, "beta", beta, "c", c, "GMRES iterations", n)


@pytest.mark.parametrize("beta", [(10.0, -5.0), (1.0, 0.0)])
def test_mg_gmres_2d_vs_oracle(dev, beta):
    from poms_b200.mg import Hierarchy
    p, N, robin = 2, [32, 24], _robin_for(beta, 1.0)
    h = Hierarchy(p, N, device=dev, c=0.0, robin=robin, beta=beta)
    _compare_gmres(h, ro.MGHierarchy(p, N, c=0.0, robin=robin), beta, 0.0, robin, dev)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_device_advection_band_vs_host(dev, p):
    from poms_b200 import bsplines as bs, setup_device as sd
    for N, kind in [(8, "uniform"), (200, "uniform"), (23, "graded")]:
        T = _knots_kind(p, N, kind == "graded")
        with sd.device_setup(True, dev):
            Gd = sd.assemble_1d_advection(p, T)
        Gh = bs.assemble_1d_advection(p, T)
        assert np.abs(Gd - Gh).max() <= 1e-14 * np.abs(Gh).max(), (N, kind)
        if kind == "uniform" and N > 4 * p + 1:
            assert all(np.array_equal(Gd[i], Gd[(N + p) // 2]) for i in range(2 * p, N + p - 2 * p))


@pytest.mark.parametrize("beta,c", [((10.0, -5.0, 3.0), 0.0), ((50.0, 20.0, 0.0), 1.0)])
def test_mg_gmres_device_setup_vs_oracle(dev, beta, c):
    from poms_b200.mg import Hierarchy
    p, N = 3, [16, 16, 16]
    robin = [r if b != 0.0 else (0.5, 0.0) for r, b in zip(_robin_for(beta), beta)]
    h = Hierarchy(p, N, device=dev, c=c, robin=robin, beta=beta, setup="device")
    hh = Hierarchy(p, N, device=dev, c=c, robin=robin, beta=beta)
    for x, y in zip(h.op.Ks + h.op.Ms, hh.op.Ks + hh.op.Ms):
        assert np.abs(x - y).max() <= 1e-13 * np.abs(y).max()
    _compare_gmres(h, ro.MGHierarchy(p, N, c=c, robin=robin), beta, c, robin, dev, maxiter=600)


# ----------------------------------------------------------------------------- manufactured solution
K3 = (1.0, 2.0, 3.0)


def _manufactured(dev, p, d, Ns, beta, c, robin):
    """u = exp(k . x) / scale: f = (c - |k|^2 + beta . k) u, and g = du/dn + alpha u on every face (non-zero
    normal flux everywhere)."""
    from poms_b200 import fem
    from poms_b200.mg import Hierarchy, mg_gmres
    from test_gpu_robin_reaction import _face_g
    k = K3[:d]
    scale = float(np.exp(sum(k)))
    u = lambda *X: torch.exp(sum(ki * x for ki, x in zip(k, X))) / scale
    gu = lambda *X: tuple(ki * u(*X) for ki in k)
    coef = c - sum(ki * ki for ki in k) + sum(b * ki for b, ki in zip(beta, k))
    f = lambda *X: coef * u(*X)
    rows = []
    for N in Ns:
        h = Hierarchy(p, [N] * d, device=dev, c=c, robin=robin, beta=beta)
        lv = h.levels[0]
        b = fem.load_vector(lv.V, lv.knots, p, f, out=lv.ws("b"))
        for axis in range(d):
            for side in (0, 1):
                fem.boundary_load(lv.V, lv.knots, p, _face_g(k, scale, axis, side, robin[axis][side], d), axis, side,
                                  out=b)
        x, info = mg_gmres(h, b, tol=1e-12, maxiter=600)
        assert info["success"], info["niter"]
        e = fem.error_norms(x, lv.knots, p, u, gu)
        rows.append((N, e["l2"], e["h1"], info["niter"]))
    return rows


MANUF = [(2, 3, (8, 16, 32)), (3, 3, (8, 16, 32)), (1, 2, (64, 128, 256)), (3, 2, (16, 32, 64)), (4, 2, (8, 16, 32))]


@pytest.mark.parametrize("p,d,Ns", MANUF)
@pytest.mark.parametrize("c", [0.0, 1.0])
def test_manufactured_convergence(dev, p, d, Ns, c):
    beta = (4.0, -2.0, 1.0)[:d]
    robin = _robin_for(beta, 1.0)
    rows = _manufactured(dev, p, d, Ns, beta, c, robin)
    rows = [r for r in rows if r[1] > 1e-10]
    assert len(rows) >= 2, rows
    (N0, l0, h0, _), (N1, l1, h1, _) = rows[-2], rows[-1]
    ol2, oh1 = np.log(l0 / l1) / np.log(N1 / N0), np.log(h0 / h1) / np.log(N1 / N0)
    assert ol2 >= p + 1 - 0.25 and oh1 >= p - 0.25, (rows, ol2, oh1)


# ----------------------------------------------------------------------------- determinism, interface
def test_mg_gmres_deterministic_and_interface(dev):
    from poms_b200.mg import Hierarchy, mg_gmres, mg_pcg
    from poms_b200.stencil import StencilVector
    beta = (10.0, -5.0, 3.0)
    h = Hierarchy(3, [32, 32, 32], device=dev, c=1.0, robin=_robin_for(beta), beta=beta)
    assert h.op is not h.levels[0].A and h.op.Ks[0].shape == h.levels[0].A.Ks[0].shape
    b = StencilVector(h.levels[0].V)
    b.data.copy_(torch.rand(b.data.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64))
    x1, i1 = mg_gmres(h, b, tol=1e-10)
    x2, i2 = mg_gmres(h, b, tol=1e-10)
    assert i1["niter"] == i2["niter"] and i1["history"] == i2["history"]
    assert torch.equal(x1.flat, x2.flat)
    with pytest.raises(ValueError):
        mg_pcg(h, b)
    # without beta: h.op is the fine level's operator, and mg_gmres solves the symmetric problem too
    h0 = Hierarchy(3, [16, 16, 16], device=dev)
    assert h0.op is h0.levels[0].A and h0.beta is None
    b0 = StencilVector(h0.levels[0].V)
    b0.data.fill_(1.0)
    xg, ig = mg_gmres(h0, b0, tol=1e-10)
    xc, ic = mg_pcg(h0, b0, tol=1e-10)
    assert ig["success"] and rel(_arr(xg), _arr(xc)) < 1e-8
