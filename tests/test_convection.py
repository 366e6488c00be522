"""Constant-velocity convection -Lap u + beta . grad u + c u with du/dn + alpha u = g (CPU).

The 1-D advection band against scipy BSpline quadrature (uniform, graded and C0 knots), its identity
G + G^T = E_hi - E_lo and its bit-identical interior rows; KronSumMatrix.poisson(beta=) against a dense scipy
assembly; the lambda_min formula of the symmetric part against dense eigenvalues (both eigen paths); every
ValueError; beta=None bit-identical to the operator without it; the oracle restatement of mg_gmres with
iteration counts that do not grow with the grid; the device assembly kernel compiled for the host under
ASan / TSan."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
from scipy.interpolate import BSpline
from scipy.linalg import eigh

from conftest import ROOT
import convection_oracle as co
import robin_oracle as ro
from oracle import poms_oracle as po
from poms_b200 import bsplines as bs
from poms_b200.stencil import KronSumMatrix, symmetric_part_lmin, _gen_eig_min

EMU = os.path.join(ROOT, "tests", "host_emu")
FULL = os.environ.get("POMS_EMU_FULL") == "1"


def _knots(p, N, kind="uniform"):
    if kind == "c0":                    # one interior breakpoint of multiplicity p
        br = np.arange(1, N) / N
        inner = np.sort(np.concatenate([br, np.full(p - 1, br[len(br) // 2])]))
        return np.concatenate([np.zeros(p + 1), inner, np.ones(p + 1)])
    T = bs.make_open_knots(p, N + p)
    if kind == "graded":
        T[p + 1:N + p] = T[p + 1:N + p] ** 1.5
    return T


def _scipy_axis(T, p):
    """Dense mass, stiffness and advection G[i, j] = int phi_j' phi_i from scipy BSpline with a (p+2)-point
    Gauss rule per element."""
    n = len(T) - p - 1
    u, w = np.polynomial.legendre.leggauss(p + 2)
    br = np.unique(T)
    x = np.concatenate([0.5 * (a + b) + 0.5 * (b - a) * u for a, b in zip(br[:-1], br[1:])])
    wq = np.concatenate([0.5 * (b - a) * w for a, b in zip(br[:-1], br[1:])])
    sp = [BSpline(T, np.eye(n)[i], p) for i in range(n)]
    B = np.array([s(x) for s in sp])
    D = np.array([s.derivative()(x) for s in sp])
    return (B * wq) @ B.T, (D * wq) @ D.T, (B * wq) @ D.T


def _kron(mats):
    out = np.ones((1, 1))
    for m in mats:
        out = np.kron(out, m)
    return out


def _dense_scipy(p, knots, c, robin, beta):
    ax = [_scipy_axis(T, p) for T in knots]
    d = len(ax)
    A = c * _kron([M for M, _, _ in ax])
    for a in range(d):
        Ka = ax[a][1] + beta[a] * ax[a][2]
        n = Ka.shape[0]
        if robin is not None:
            Ka = Ka.copy()
            Ka[0, 0] += robin[a][0]
            Ka[n - 1, n - 1] += robin[a][1]
        A = A + _kron([Ka if b == a else ax[b][0] for b in range(d)])
    return A


# ------------------------------------------------------------------------------------- 1-D band
@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("kind", ["uniform", "graded", "c0"])
def test_advection_band_vs_scipy(p, kind):
    T = _knots(p, 11, kind)
    n = len(T) - p - 1
    ref = _scipy_axis(T, p)[2]
    G = bs.assemble_1d_advection(p, T)
    assert G.shape == (n, 2 * p + 1)
    Gd = bs.band_to_dense(G)
    assert np.abs(Gd - ref).max() < 1e-13 * np.abs(ref).max()
    assert np.abs(co.advection_1d(p, T) - ref).max() < 1e-13 * np.abs(ref).max()
    # integration by parts on an open knot vector: G + G^T = e_{n-1} e_{n-1}^T - e_0 e_0^T
    E = np.zeros((n, n))
    E[0, 0], E[-1, -1] = -1.0, 1.0
    assert np.abs(Gd + Gd.T - E).max() < 1e-14 * max(1.0, np.abs(Gd).max())
    # out-of-matrix band entries are zero
    for k in range(-p, p + 1):
        i = np.arange(n)
        assert not G[(i + k < 0) | (i + k >= n), k + p].any()


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_advection_band_toeplitz_interior_bit_identical(p):
    N = 40
    T = _knots(p, N)
    n = N + p
    G = bs.assemble_1d_advection(p, T)
    assert all(np.array_equal(G[i], G[n // 2]) for i in range(2 * p, n - 2 * p))
    raw = bs.assemble_1d_advection(p, T, toeplitz_interior=False)
    assert np.abs(raw - G).max() < 1e-13 * np.abs(G).max()
    # antisymmetric Toeplitz row: G[i, p+k] = -G[i, p-k]
    row = G[n // 2]
    assert np.abs(row + row[::-1]).max() < 1e-13 * np.abs(row).max()
    # graded knots: nothing is overwritten
    Tg = _knots(p, N, "graded")
    assert np.array_equal(bs.assemble_1d_advection(p, Tg), bs.assemble_1d_advection(p, Tg, toeplitz_interior=False))


# ------------------------------------------------------------------------------------- operator
BETAS = {2: [(1.0, 0.0), (10.0, -5.0), (-3.0, 40.0)], 3: [(1.0, 0.0, 0.0), (10.0, -5.0, 3.0), (50.0, 20.0, 0.0)]}


def _robin_for(beta, extra=0.0):
    """alpha = |beta_a| / 2 + extra on each inflow face (beta . n < 0), 0 on the outflow faces."""
    return [((0.5 * b + extra, 0.0) if b > 0 else (0.0, -0.5 * b + extra)) for b in beta]


@pytest.mark.parametrize("p", [1, 2, 3, 5])
@pytest.mark.parametrize("d", [2, 3])
def test_poisson_beta_vs_dense_scipy(p, d):
    Ns = (7, 5, 6)[:d] if d == 3 else (9, 8)
    knots = [_knots(p, N, "graded" if a == 0 else "uniform") for a, N in enumerate(Ns)]
    for beta in BETAS[d]:
        for c, robin in ((1.0, None), (0.0, _robin_for(beta, 1.0)), (2.5, _robin_for(beta))):
            if robin is None and max(abs(b) for b in beta) > 1.0:
                continue                        # indefinite without inflow terms (see the ValueError test)
            A = KronSumMatrix.poisson(p, knots, c=c, robin=robin, beta=beta)
            ref = _dense_scipy(p, knots, c, robin, beta)
            dense = sum(_kron([bs.band_to_dense(A.Ks[b] if b == a else A.Ms[b]) for b in range(d)]) for a in range(d))
            assert np.abs(dense - ref).max() < 1e-12 * np.abs(ref).max(), (beta, c)
            Ao = co.poisson_operator(p, knots, c, robin, beta)[0].tocsr().toarray()
            assert np.abs(Ao - ref).max() < 1e-12 * np.abs(ref).max(), (beta, c)


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_beta_none_bit_identical(p):
    """beta=None (and an all-zero beta) build exactly the bands, mass bands and Toeplitz ranges of the operator
    without a convection term."""
    knots = [_knots(p, 40), _knots(p, 12, "graded"), _knots(p, 33)]
    robin = [(1.0, 0.0), (0.0, 0.0), (0.0, 3.0)]
    for c, rb in ((1.0, None), (0.0, robin)):
        ref = KronSumMatrix.poisson(p, knots, c=c, robin=rb)
        for A in (KronSumMatrix.poisson(p, knots, c=c, robin=rb, beta=None),
                  KronSumMatrix.poisson(p, knots, c=c, robin=rb, beta=[0.0, 0, -0.0])):
            for a in range(3):
                assert np.array_equal(A.Ks[a], ref.Ks[a]) and np.array_equal(A.Ms[a], ref.Ms[a])
                assert np.array_equal(A.mass_bands[a], ref.mass_bands[a])
            assert all(np.array_equal(x, y) for x, y in zip(A._toeplitz(), ref._toeplitz()))


def test_convection_keeps_toeplitz_ranges():
    """beta_a G_a has bit-identical interior rows on uniform knots: the Toeplitz ranges (the constant-bank path
    of the mat-vec kernels) stay those of the symmetric operator, and the interior rows of K_a + beta_a G_a are
    no longer symmetric when beta_a != 0."""
    p = 3
    knots = [_knots(p, N) for N in (40, 36, 50)]
    rng0 = KronSumMatrix.poisson(p, knots)._toeplitz()[1]
    for beta in BETAS[3]:
        A = KronSumMatrix.poisson(p, knots, robin=_robin_for(beta), beta=beta)
        coef, rng = A._toeplitz()
        assert np.array_equal(rng, rng0)
        for a in range(3):
            k = coef[a, 1]
            assert (np.abs(k - k[::-1]).max() > 1e-3 * np.abs(k).max()) == (beta[a] != 0.0)


# ------------------------------------------------------------------------------------- well-posedness
@pytest.mark.parametrize("p,Ns", [(1, (8, 7)), (2, (6, 7)), (3, (5, 6, 4)), (2, (4, 5, 6))])
def test_lmin_formula_vs_dense_symmetric_part(p, Ns):
    d = len(Ns)
    knots = [_knots(p, N, "graded" if a == 1 else "uniform") for a, N in enumerate(Ns)]
    Mbig = _kron([bs.band_to_dense(bs.assemble_1d_bands(p, T)[0]) for T in knots])
    cases = [(1.0, None, [1.0] + [0.0] * (d - 1)), (0.5, None, [3.0] * d), (0.0, _robin_for([4.0] * d), [4.0] * d),
             (0.1, [(0.0, 0.0)] * d, [-2.0] + [0.0] * (d - 1)), (0.0, [(2.0, 0.0)] * d, [0.0] * d)]
    for c, robin, beta in cases:
        _, Mb, Kb = ro.poisson_operator(p, knots, c, robin)
        lam = symmetric_part_lmin(Kb, Mb, c, beta, [1.0] * d)
        A = _dense_scipy(p, knots, c, robin, beta)
        ref = eigh(0.5 * (A + A.T), Mbig, eigvals_only=True)[0]
        assert abs(lam - ref) < 1e-9 * max(1.0, abs(ref)), (c, robin, beta, lam, ref)


@pytest.mark.parametrize("p", [1, 3, 5])
def test_lmin_sparse_path_vs_dense(p):
    """n > 1500: shift-invert Lanczos from the trace-inequality bound agrees with dense LAPACK."""
    N = 1600
    T = _knots(p, N)
    M, K = bs.assemble_1d_bands(p, T)
    # (the dense reference itself is accurate to ~1e-7 on these pencils: M is ill-conditioned at p = 5)
    for beta, lo, hi in ((0.0, 1.0, 0.0), (3.0, 0.0, 0.0), (-40.0, 0.0, 25.0), (200.0, 1.0, 0.0)):
        S = K.copy()
        S[0, p] += lo - 0.5 * beta
        S[-1, p] += hi + 0.5 * beta
        bound = -(0.25 * beta * beta + 0.5 * abs(beta))
        got = _gen_eig_min(S, M, bound)
        ref = eigh(bs.band_to_dense(S), bs.band_to_dense(M), eigvals_only=True, subset_by_index=[0, 0])[0]
        assert bound <= ref and abs(got - ref) < 1e-6 * max(1.0, abs(ref)), (beta, got, ref)


BAD_BETA = [dict(beta=[1.0]), dict(beta=[1.0, 2.0, 3.0]), dict(beta=[1.0, float("nan")]),
            dict(beta=[float("inf"), 0.0]), dict(beta=["a", 0.0]), dict(beta=3.0),
            # indefinite symmetric part: small c, large beta, an inflow face with alpha = 0
            dict(c=1e-3, beta=[1.0, 0.0]), dict(c=1.0, beta=[40.0, 0.0]),
            dict(c=0.0, robin=[(0.0, 5.0), (0.0, 0.0)], beta=[6.0, 0.0]),
            dict(c=1.0, robin=[(15.0, 0.0), (0.0, 0.0)], beta=[40.0, 0.0]),
            # the rule of the symmetric operator stays in force
            dict(c=0.0, beta=[1.0, 0.0]), dict(c=-1.0, beta=[0.0, 0.0])]


@pytest.mark.parametrize("kw", BAD_BETA)
def test_bad_beta_raise(kw):
    from poms_b200.mg import Hierarchy
    knots = [_knots(2, 8), _knots(2, 8)]
    with pytest.raises(ValueError):
        KronSumMatrix.poisson(2, knots, **kw)
    with pytest.raises(ValueError):
        Hierarchy(2, [8, 8], device="cpu", **kw)


def test_inflow_alpha_makes_it_well_posed():
    """The same velocities are accepted once the inflow faces carry alpha >= |beta_a| / 2, even with c = 0."""
    knots = [_knots(2, 8), _knots(2, 8)]
    for beta in ([40.0, 0.0], [2.0, -7.0], [-1.0, 1.0]):
        A = KronSumMatrix.poisson(2, knots, c=0.0, robin=_robin_for(beta, 0.1), beta=beta)
        assert A.Ks[0].shape == (10, 5)


# ------------------------------------------------------------------------------------- oracle mg_gmres
# 3-D p = 3, c = 1, alpha = |beta_a| / 2 on the inflow faces, a seeded random right-hand side, tol 1e-10,
# restart 30, glt smoother, Nc = 4 (so that N = 8 has two levels too).  Recorded GMRES iteration counts at
# N = 8, 16, 32, 64:
#   beta (1, 0, 0)      32, 32, 31, 30     (MG-PCG on the symmetric problem: 28 at N = 16 and 32)
#   beta (10, -5, 3)    70, 68, 62, 59
# The count depends on beta, not on h: it never grows with N.  It falls slowly at the larger velocity, because
# the coarse grids carry the larger cell Peclet numbers.  (beta = (50, 20, 0) needs 260 to 300 iterations with
# restart 30; it runs on the GPU only.)
GMRES_COUNTS = {(1.0, 0.0, 0.0): [32, 32, 31, 30], (10.0, -5.0, 3.0): [70, 68, 62, 59]}


@pytest.mark.parametrize("beta", list(GMRES_COUNTS))
def test_oracle_mg_gmres_counts_independent_of_h(beta):
    p, c = 3, 1.0
    robin = _robin_for(beta)
    counts = []
    for N in (8, 16, 32, 64):
        h = ro.MGHierarchy(p, [N] * 3, Nc=4, c=c, robin=robin)
        assert len(h.levels) >= 2
        knots = [po.make_open_knots(p, N + p)] * 3
        A = co.poisson_operator(p, knots, c, robin, list(beta))[0]
        b = np.random.default_rng(7).standard_normal(A.npts)
        x, info = co.mg_gmres(h, A, b, tol=1e-10)
        assert info["success"]
        r = b - A.dot(x)
        assert np.sqrt(np.vdot(r, r)) <= 1e-10 * np.sqrt(np.vdot(b, b))
        counts.append(info["niter"])
    print("beta", beta, "GMRES iterations at N = 8, 16, 32, 64:", counts)
    assert all(abs(x - y) <= 2 for x, y in zip(counts, GMRES_COUNTS[beta])), counts
    assert all(f <= c_ + 2 for c_, f in zip(counts[:-1], counts[1:])), counts     # no growth with N
    if beta == (1.0, 0.0, 0.0):
        assert max(counts) - min(counts) <= 2, counts


# ------------------------------------------------------------------------------------- host emulation
@pytest.fixture(scope="module")
def advection_exes(tmp_path_factory):
    """emu_advection under {ASan, TSan}: the section of poms_setup.cu that make_emu_source cuts out."""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    sys.path.insert(0, EMU)
    import make_emu_source
    d = tmp_path_factory.mktemp("emu_advection")
    src, _ = make_emu_source.setup_section()
    (d / "setup_emu.cuh").write_text(src)
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    procs = {}
    for name, flags in (("asan", ["-fsanitize=address", "-fno-omit-frame-pointer"]), ("tsan", ["-fsanitize=thread"])):
        out = str(d / ("emu_advection_" + name))
        procs[name] = (out, subprocess.Popen(
            [gxx, "-std=c++17", "-O0", "-g"] + flags + ["-I" + EMU, "-I" + str(d), "-I" + os.path.join(ROOT, "include"),
                                                         "-I" + cuda_inc, os.path.join(EMU, "emu_advection.cpp"),
                                                         "-o", out, "-lpthread"],
            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    res = {}
    for name, (out, pr) in procs.items():
        log = pr.communicate()[0]
        assert pr.returncode == 0, log[-3000:]
        probe = subprocess.run([out], capture_output=True, text=True)
        if probe.returncode == 2 and "FATAL" not in probe.stderr:
            res[name] = out
    return res


def _run_advection(exe, tmp, T, p):
    n = len(T) - p - 1
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:2] = n, p
    u, w = np.polynomial.legendre.leggauss(p + 1)
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        for a in (T, u, w):
            a = np.ascontiguousarray(a, dtype=np.float64)
            np.array([a.size], dtype=np.int64).tofile(f)
            a.tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:], dtype=np.float64).reshape(n, 2 * p + 1)


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_advection_kernel_emulated(advection_exes, tmp_path, san, p):
    if not FULL and not ((san == "asan" and p in (1, 3, 5)) or (san == "tsan" and p == 3)):
        pytest.skip("not in the core set (POMS_EMU_FULL=1 runs every case under both sanitizers)")
    if san not in advection_exes:
        pytest.skip("emu_advection (%s) cannot start in this environment" % san)
    exe = advection_exes[san]
    for N, kind in [(8, "uniform"), (37, "uniform"), (23, "graded"), (19, "c0")]:
        T = _knots(p, N, kind)
        Gh = bs.assemble_1d_advection(p, T, toeplitz_interior=False)
        Gd = _run_advection(exe, tmp_path, T, p)
        assert np.abs(Gd - Gh).max() <= 1e-13 * np.abs(Gh).max(), (N, kind)
