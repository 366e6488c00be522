"""GPU parity on inputs the benchmark never produces but users do: graded, boundary-layer, mirror-graded and
jittered knot vectors (the Toeplitz interior range of the bands collapses to the middle row and the TMA
mat-vec takes other branches: variant 0 when the interior rows are not symmetric, the non-Toeplitz plane
loop of variant 1 when axis 1 is graded), degrees 1 and 5 of the 3-D kernels with interior tiles,
synthetic Toeplitz ranges, plane sub-range launches, transfers between non-uniform nested knot vectors,
the dense fp64 tensor-core contraction of the coarse solve at the sizes the hierarchy builds, and solves
on graded meshes whose error is measured against the exact solution.

Every case asserts the dispatch it targets (Toeplitz ranges, the kernel's symmetry predicate, the transfer
kind after the call, the dense mode), so that a later change of the dispatch cannot quietly turn a case
into a copy of one that `test_gpu_benchpath.py` already runs.  References are the CPU oracle
(`oracle.poms_oracle`, its own dense assembly and Boehm insertion matrices) or numpy in long double."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


# ----------------------------------------------------------------------------- knot families
def _clamped(p, interior):
    return np.concatenate([np.zeros(p + 1), np.asarray(interior, float), np.ones(p + 1)])


def uniform(p, N):
    from poms_b200 import bsplines as bs
    return bs.make_open_knots(p, N + p)


def power(p, N, g=1.5):
    """N elements, interior knots t -> t^g (the grading of tests/test_fem.py)."""
    return _clamped(p, (np.arange(1, N) / N) ** g)


def blayer(p, N, m=3):
    """N - 2 uniform elements in the middle, the first and last split into m + 1 geometrically halved ones."""
    h = 1.0 / N
    ends = h * 0.5 ** np.arange(m, 0, -1)
    return _clamped(p, np.concatenate([ends, np.arange(1, N) * h, 1.0 - ends[::-1]]))


def cosine(p, N):
    """N elements, t -> (1 - cos(pi t)) / 2: mirror-symmetric, finest at both ends."""
    return _clamped(p, 0.5 * (1.0 - np.cos(np.pi * np.arange(1, N) / N)))


def jitter(p, N, eps=1e-12):
    """Uniform interior knots moved by up to eps (seeded): not uniform to `_is_uniform_open`, interior rows
    equal to ~1e-11 only."""
    t = np.arange(1, N) / N
    return _clamped(p, t + eps * np.random.default_rng(N).uniform(-1.0, 1.0, t.size))


FAMILIES = {"u": uniform, "pow": power, "bl": blayer, "cos": cosine, "jit": jitter}


def family_knots(kind, p, N):
    """Knot vector of `kind` with about N elements.  cosine: N is made such that the number of basis
    functions is odd, so that the middle row is its own mirror image (symmetric to rounding)."""
    if kind == "cos" and (N + p) % 2 == 0:
        N += 1
    return FAMILIES[kind](p, N)


# ----------------------------------------------------------------------------- dispatch predicates
SYM_TOL = 1e-13        # poms_matvec3d_tma.cuh try_matvec3d_tma / poms_matvec2d_tma.cuh: `sym`


def tma_sym(A):
    """The kernels' symmetry test, restated: the Toeplitz rows of the M and K bands of every axis but the
    first are symmetric to SYM_TOL relative (sum form; the 3-D single product is always 'symmetric').
    3-D: False selects the round-1 TMA kernel (variant 0).  2-D: False selects the g.sym = 0 sum form."""
    from poms_b200.stencil import FORM_SUM
    if A.form != FORM_SUM:
        return A.ndim == 3
    coef = A._toeplitz()[0]
    for a in range(1, A.ndim):
        for r in coef[a]:
            if not np.all(np.abs(r - r[::-1]) <= SYM_TOL * np.abs(r).max()):
                return False
    return True


def range_ok(kind, p, n, lo, hi):
    """Is [lo, hi) what KronSumMatrix._toeplitz reports for one axis of `kind` with n basis functions?
    Uniform: at least the rows 2p .. n-2p-1 that assemble_1d_bands makes bit-identical (a boundary row
    may equal them by chance); every other family: the middle row alone."""
    if kind == "u" and n > 4 * p + 1:
        return lo <= 2 * p and hi >= n - 2 * p and hi - lo <= n - 2 * p
    return (lo, hi) == (n // 2, n // 2 + 1)


def expected_sym(kinds, p, npts):
    """Symmetry predicate expected for per-axis knot kinds: uniform rows are symmetric to rounding, and so
    are the middle rows of a boundary layer (uniform there) and of a cosine grading with an odd number of
    functions; power-graded rows are asymmetric by ~1e-2, jittered ones by ~1e-11."""
    return all(k in ("u", "bl") or (k == "cos" and n % 2 == 1) for k, n in zip(kinds[1:], npts[1:]))


def check_dispatch(A, kinds, p):
    rng = A._toeplitz()[1]
    for a, (k, n) in enumerate(zip(kinds, A.npts)):
        assert range_ok(k, p, n, *rng[2 * a:2 * a + 2]), (a, k, rng)
    assert tma_sym(A) == expected_sym(kinds, p, A.npts)


# ----------------------------------------------------------------------------- small helpers
def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _space(npts, pads, dev):
    from poms_b200.stencil import StencilVectorSpace
    return StencilVectorSpace(list(npts), list(pads), [False] * len(npts), device=dev)


def _vec(V, arr):
    from poms_b200.stencil import StencilVector
    return StencilVector.from_array(V, arr)


def _arr(v):
    return v.toarray().reshape(v.space.npts)


def _operator(p, knots):
    from poms_b200.stencil import KronSumMatrix
    from oracle import poms_oracle as po
    return KronSumMatrix.poisson(p, knots), po.poisson_operator(p, knots)[0]


def _all_epilogues(A, Ao, V, dev, seed, mode):
    """Every epilogue and fused dot of A against the oracle operator, at the tolerances of
    test_gpu_benchpath.test_toeplitz_operator_all_epilogues_vs_oracle; returns the STORE result."""
    from poms_b200.stencil import (StencilVector, DeviceContext, EPI_STORE, EPI_RESID, EPI_JACOBI,
                                   EPI_DINV, EPI_AXPY)
    rng = np.random.default_rng(seed)
    Xh, Bh = rng.standard_normal(V.npts), rng.standard_normal(V.npts)
    X, B = _vec(V, Xh), _vec(V, Bh)
    ctx = DeviceContext.get(dev)
    Yo = Ao.dot(Xh)
    D = Ao.diagonal()
    sc = np.abs(Yo).max()
    Y = StencilVector(V)
    A.apply(X, Y, EPI_STORE, dot_ptr=ctx.sptr(10))
    store = _arr(Y)
    assert rel(store, Yo) < 1e-13, mode
    assert abs(ctx.scal[10].item() - np.vdot(Xh, Yo)) < 1e-12 * np.vdot(np.abs(Xh), np.abs(Yo)), mode
    A.apply(X, Y, EPI_RESID, b=B, dot_ptr=ctx.sptr(11))
    Ro = Bh - Yo
    assert np.abs(_arr(Y) - Ro).max() < 1e-13 * sc, mode
    assert abs(ctx.scal[11].item() - np.vdot(Ro, Ro)) < 1e-12 * np.vdot(Ro, Ro), mode
    om = 0.61
    dr = om * Ro / D
    A.apply(X, Y, EPI_JACOBI, b=B, omega=om, dot_ptr=ctx.sptr(12))
    assert np.abs(_arr(Y) - (Xh + dr)).max() < 1e-12 * np.abs(Xh + dr).max(), mode
    assert abs(ctx.scal[12].item() - np.vdot(dr, dr)) < 1e-11 * np.vdot(dr, dr), mode
    A.apply(X, Y, EPI_DINV, b=B, omega=1.0)
    assert np.abs(_arr(Y) - Ro / D).max() < 1e-12 * np.abs(Ro / D).max(), mode
    A.apply(X, Y, EPI_AXPY, b=B, omega=om)
    assert np.abs(_arr(Y) - (Bh + om * Yo)).max() < 1e-13 * (sc + np.abs(Bh).max()), mode
    A.apply(X, Y, EPI_AXPY, b=None, omega=om)
    assert np.abs(_arr(Y) - om * Yo).max() < 1e-13 * sc, mode
    if V.ld != V.local_shape[-1]:
        assert float(Y.flat[..., V.local_shape[-1]:].abs().max()) == 0.0, mode
    return store


def _run_all_paths(A, Ao, V, dev, seed):
    """Variant 1 (v3), variant 0 (round-1 TMA kernel) and the generic kernel: every epilogue of each
    against the oracle, and the three STORE results against each other."""
    from poms_b200 import _lib
    L = _lib.lib()
    out = {}
    try:
        for mode in ("v1", "v0", "generic"):
            L.poms_set_matvec3d_variant(0 if mode == "v0" else 1)
            L.poms_set_force_generic(1 if mode == "generic" else 0)
            out[mode] = _all_epilogues(A, Ao, V, dev, seed, mode)
    finally:
        L.poms_set_force_generic(0)
        L.poms_set_matvec3d_variant(1)
    sc = np.abs(out["v1"]).max()
    assert np.abs(out["v0"] - out["v1"]).max() < 1e-13 * sc
    assert np.abs(out["generic"] - out["v1"]).max() < 1e-13 * sc
    return out


# ----------------------------------------------------------------------------- 1. operator
# N elements per axis: interior and ragged tiles in both tile axes (64 columns, 16 rows) and several
# chunks along axis 1; smaller at p = 4, 5 (the oracle's dense assembly is the cost)
SHAPE3 = {1: (37, 147, 297), 2: (68, 129, 260), 3: (37, 147, 297), 4: (21, 60, 200), 5: (21, 60, 200)}
GRADED3 = {"g1": ("pow", "u", "u"), "g2": ("u", "pow", "u"), "g3": ("u", "u", "pow"),
           "all": ("pow", "pow", "pow"), "blayer": ("bl", "bl", "bl"), "cosine": ("cos", "cos", "cos"),
           "jitter": ("jit", "jit", "jit")}
OP3_CASES = [(name, p) for name in GRADED3 for p in range(1, 6)] + [("uniform", 1), ("uniform", 5)]


@pytest.mark.parametrize("name,p", OP3_CASES)
def test_operator3d_nonuniform_all_paths_vs_oracle(dev, name, p):
    kinds = GRADED3.get(name, ("u", "u", "u"))
    knots = [family_knots(k, p, N) for k, N in zip(kinds, SHAPE3[p])]
    A, Ao = _operator(p, knots)
    check_dispatch(A, kinds, p)
    if name == "uniform":
        lo, hi = A._toeplitz()[1][4:6]
        assert hi - lo > 64, "the shape must contain Toeplitz-interior tiles"
    V = _space(A.npts, [p] * 3, dev)
    _run_all_paths(A, Ao, V, dev, seed=p)


GRADED2 = {"g1": ("pow", "u"), "g2": ("u", "pow"), "both": ("pow", "pow")}


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("name", list(GRADED2))
def test_operator2d_graded_vs_oracle(dev, name, p):
    """Graded axis 2 switches the 2-D TMA kernel to its g.sym = 0 sum form; graded axis 1 leaves no
    Toeplitz rows along the march."""
    kinds = GRADED2[name]
    knots = [family_knots(k, p, N) for k, N in zip(kinds, (120, 500))]
    A, Ao = _operator(p, knots)
    check_dispatch(A, kinds, p)
    assert tma_sym(A) == (kinds[1] == "u")
    _all_epilogues(A, Ao, _space(A.npts, [p, p], dev), dev, 3 + p, "2-D")


def _synthetic_ranges(n, p):
    """Toeplitz ranges inside the bit-identical rows [2p, n - 2p) of a uniform operator that start and end
    off the 2p margins and off tile boundaries: lo >> 2p; hi - lo shorter than a tile; empty."""
    return {"deep": [(2 * p + 9, n[0] - 2 * p - 5), (2 * p + 19, n[1] - 2 * p - 6), (2 * p + 37, n[2] - 2 * p - 11)],
            "short": [(2 * p + 3, 2 * p + 8), (21, 30), (70, 101)],
            "empty": [(n[0] // 2,) * 2, (n[1] // 2,) * 2, (n[2] // 2,) * 2],
            "asym": [(2 * p + 9, n[0] - 2 * p - 5), (2 * p + 19, n[1] - 2 * p - 6), (2 * p + 37, n[2] - 2 * p - 11)]}


SYNTH_N = (60, 60, 200)


def perturb_outside(bands, lo, hi, seed):
    """Copies of 1-D bands whose rows outside [lo, hi) are scaled by 1 + 1e-3 u (u uniform in [-1, 1]):
    the rows a kernel must take from memory then differ from the constant-bank row, so a row put on the
    wrong side of a range boundary changes the result."""
    rng = np.random.default_rng(seed)
    out = []
    for b in bands:
        b = b.copy()
        f = 1.0 + 1e-3 * rng.uniform(-1.0, 1.0, b.shape)
        f[lo:hi] = 1.0
        out.append(b * f)
    return out


@pytest.mark.parametrize("which", ["deep", "short", "empty", "asym"])
@pytest.mark.parametrize("p", [1, 2, 3, 5])
def test_operator3d_synthetic_toeplitz_ranges(dev, p, which):
    """The kernels take rows [lo, hi) of each axis from the constant bank and the others from memory:
    ranges that begin and end anywhere (the slab sub-problems shift them at run time) isolate the column
    pair / plane-range arithmetic of the v3 kernel (tl / th / nb, toep2_cta, toep1) and of variant 0.
    Rows outside the ranges are perturbed (perturb_outside), rows inside are the uniform middle row; "asym":
    the rows inside are one row made asymmetric by 1e-3, which the symmetry test must send to variant 0
    (the pair sums of variant 1 would use the mean of its two halves)."""
    from poms_b200.stencil import KronSumMatrix
    from oracle import poms_oracle as po
    U = KronSumMatrix.poisson(p, [uniform(p, N) for N in SYNTH_N])
    coef, full = U._toeplitz()
    ranges = _synthetic_ranges(U.npts, p)[which]
    rng = np.array([v for r in ranges for v in r], dtype=np.int32)
    assert np.all(rng[0::2] >= full[0::2]) and np.all(rng[1::2] <= full[1::2]) and np.all(rng[1::2] >= rng[0::2])
    Ms, Ks = [], []
    for a, (lo, hi) in enumerate(ranges):
        m, k = perturb_outside([U.Ms[a], U.Ks[a]], lo, hi, seed=10 * p + a)
        if which == "asym":
            coef = coef.copy()
            coef[a] *= 1.0 + 1e-3 * np.linspace(-1.0, 1.0, coef.shape[-1])
            m[lo:hi], k[lo:hi] = coef[a, 0], coef[a, 1]
        Ms.append(m)
        Ks.append(k)
    A = KronSumMatrix(Ms, Ks)
    A._toep = (coef, rng)
    assert tma_sym(A) == (which != "asym")
    Ao = po.KronSumOperator([(Ks[0], Ms[1], Ms[2]), (Ms[0], Ks[1], Ms[2]), (Ms[0], Ms[1], Ks[2])])
    _run_all_paths(A, Ao, _space(A.npts, [p] * 3, dev), dev, seed=17 + p)


@pytest.mark.parametrize("p", [2, 3])
def test_plane_subrange_launches_match_full_launch(dev, p):
    """The slab-overlap path of KronSumMatrix.apply on one device: output planes [0, P), [P, n1 - P) and
    [n1 - P, n1) as three launches of the same kernel on shifted pointers (the planes outside each range
    are its ghost planes), with a graded axis 1.  Each point's sum runs over the same terms in the same
    order whatever the launch, so the union must be bit-identical to one full launch."""
    from poms_b200 import _lib
    from poms_b200.stencil import StencilVector, DeviceContext, EPI_STORE, EPI_RESID, EPI_AXPY
    kinds = ("pow", "u", "u")
    knots = [family_knots(k, p, N) for k, N in zip(kinds, (60, 40, 150))]
    A, Ao = _operator(p, knots)
    check_dispatch(A, kinds, p)
    V = _space(A.npts, [p] * 3, dev)
    rng = np.random.default_rng(p)
    X, B = _vec(V, rng.standard_normal(V.npts)), _vec(V, rng.standard_normal(V.npts))
    L = _lib.lib()
    ctx = DeviceContext.get(dev)
    m, k = A._bands(V)
    kp = [t.data_ptr() if t is not None else None for t in k]
    n1, P = V.local_shape[0], A.P
    for epi, bv in ((EPI_STORE, None), (EPI_RESID, B), (EPI_AXPY, B)):
        bp = bv.ptr if bv is not None else None
        full, parts = StencilVector(V), StencilVector(V)
        A._launch(L, V, X, full, bp, m, kp, epi, 0.7, None, ctx)
        for z0, z1 in ((0, P), (P, n1 - P), (n1 - P, n1)):
            A._launch(L, V, X, parts, bp, m, kp, epi, 0.7, None, ctx, z0, z1)
        assert torch.equal(parts.flat, full.flat), epi
        if epi == EPI_STORE:
            assert rel(_arr(full), Ao.dot(_arr(X))) < 1e-13


# ----------------------------------------------------------------------------- 2. transfers
def _nested(kind, p):
    """(Tc, Tf) per axis for a kind of nesting between non-uniform knot vectors."""
    from poms_b200.mg import fine_knots
    out = []
    for N in (18, 20, 70):
        if kind == "graded":
            Tc = power(p, N)
        elif kind == "blayer":
            Tc = blayer(p, N)
        else:
            Tc = uniform(p, N)
        u = np.unique(Tc)
        mids = 0.5 * (u[1:] + u[:-1])
        if kind == "local":
            mids = np.concatenate([mids[:3], mids[-3:]])         # refine the first and last 3 elements only
        out.append((Tc, fine_knots(Tc, mids)))
    return out


@pytest.mark.parametrize("kind", ["graded", "local", "blayer"])
@pytest.mark.parametrize("p", [1, 3, 5])
def test_transfer_nonuniform_nested_vs_oracle(dev, p, kind):
    from poms_b200.mg import Transfer
    from oracle import poms_oracle as po
    axes = _nested(kind, p)
    Tc, Tf = [a[0] for a in axes], [a[1] for a in axes]
    nc, nf = [len(T) - p - 1 for T in Tc], [len(T) - p - 1 for T in Tf]
    Vf, Vc = _space(nf, [p] * 3, dev), _space(nc, [p] * 3, dev)
    tr = Transfer(Tc, Tf, p, dev)
    P1s = [po.insertion_matrix(po.knots_to_insert(Tf[a], nf[a], p, Tc[a], nc[a], p), nc[a], p, Tc[a])
           for a in range(3)]
    for a in range(3):
        assert P1s[a].shape == (nf[a], nc[a])
    if kind != "local" and p > 1:
        # not the uniform 2:1 pattern: the rows differ from those of the uniform coarse grid (at p = 1 a
        # midpoint insertion gives the weights 1, 1/2, 1/2 whatever the element lengths)
        from poms_b200 import bsplines as bs
        st_u, cf_u, _ = bs.knot_insertion_rows(uniform(p, 70), uniform(p, 140), p)
        st, cf, _ = tr.P1_rows[2]
        assert cf.shape != cf_u.shape or np.abs(cf - cf_u).max() > 1e-3
    rng = np.random.default_rng(11 + p)
    rf, ec, xf = rng.standard_normal(nf), rng.standard_normal(nc), rng.standard_normal(nf)
    same_w = len({op.W for op in tr.R}) == 1 and len({op.W for op in tr.P}) == 1
    ran = []
    for k in ("v1", "v2", None):
        if k == "v2" and not same_w:
            continue                   # v2 needs one row width on all axes
        if kind == "local" and k is not None:
            # the one-pass tiles are sized for about two fine points per coarse point; on an axis refined
            # only locally (n_f ~ n_c) a tile may need more coarse points than it stages, and the kernel
            # then declines (negative status) instead of computing.  Call it directly: each operation
            # either declines or is exact.
            from poms_b200.mg import _fused_restrict, _fused_prolong
            rc = _vec(Vc, np.zeros(nc))
            if _fused_restrict(tr.R, _vec(Vf, rf).flat, tuple(nf), Vf.ld, rc.flat, tuple(nc), Vc.ld,
                               v2=(k == "v2")):
                assert rel(_arr(rc), po.restrict(P1s, rf)) < 1e-13, k
                ran.append(k + " restrict")
            x = _vec(Vf, xf)
            if _fused_prolong(tr.P, _vec(Vc, ec).flat, tuple(nc), Vc.ld, x.flat, tuple(nf), Vf.ld, True,
                              v2=(k == "v2")):
                assert rel(_arr(x), xf + po.prolong(P1s, ec)) < 1e-13, k
                ran.append(k + " prolong")
            continue
        tr.fused, tr.fused_max = k == "v1", (10 ** 12 if k == "v1" else -1)
        tr.fused_v2, tr.v2_min = k == "v2", 0
        assert tr._want_fused(Vf.npts, "restrict") == tr._want_fused(Vf.npts, "prolong") == k
        assert rel(_arr(tr.restrict(_vec(Vf, rf), Vc)), po.restrict(P1s, rf)) < 1e-13, k
        x = _vec(Vf, xf)
        tr.prolong_add(_vec(Vc, ec), x)
        assert rel(_arr(x), xf + po.prolong(P1s, ec)) < 1e-13, k
        assert tr._want_fused(Vf.npts, "restrict") == tr._want_fused(Vf.npts, "prolong") == k, \
            "silent fall-back to the gathers"
        ran.append(k)
    print("%s p=%d: %s" % (kind, p, ran))
    if kind in ("graded", "blayer"):
        assert "v2" in ran, "v2 must run on rows that are not the uniform 2:1 pattern"


# ----------------------------------------------------------------------------- 3. coarse solve
DENSE_N = [1, 4, 31, 32, 33, 63, 64, 65, 131, 259]


def _odd_ld(n):
    return n + 1 if n % 2 == 0 else n + 2


def _dense_case(dev, n_in, n_out, axis, seed):
    """One contraction out = Q along `axis` through _AxisOp(dense=True) on pitched arrays with an odd
    row pitch and outer extents that are not multiples of 64; returns the max error over the bound
    n_in eps sum_j |Q_ij| |x_j| (the standard bound of a length-n_in fp64 dot product)."""
    from poms_b200.mg import _AxisOp
    rng = np.random.default_rng(seed)
    shape = [37, 23, 29]
    shape[axis] = n_in
    Q = rng.standard_normal((n_out, n_in))
    op = _AxisOp(np.zeros(n_out, np.int32), Q, n_in, dev, dense=True)
    assert op.dense
    x = rng.standard_normal(shape)
    ld_in = _odd_ld(shape[2])
    ld_out = _odd_ld(n_out) if axis == 2 else ld_in
    src = torch.zeros(tuple(shape[:2]) + (ld_in,), dtype=torch.float64, device=dev)
    src[:, :, :shape[2]] = torch.as_tensor(x, device=dev)
    out_shape = list(shape)
    out_shape[axis] = n_out
    dst = torch.zeros(tuple(out_shape[:2]) + (ld_out,), dtype=torch.float64, device=dev)
    op.apply(src, dst, tuple(shape), ld_in, ld_out, axis)
    y = dst[:, :, :out_shape[2]].cpu().numpy()
    xl, Ql = x.astype(np.longdouble), Q.astype(np.longdouble)
    sub = "ij,jbc->ibc" if axis == 0 else ("ij,ajc->aic" if axis == 1 else "ij,abj->abi")
    ref = np.einsum(sub, Ql, xl)
    bound = n_in * EPS * np.einsum(sub, np.abs(Ql), np.abs(xl))
    return float(np.max(np.abs(y - ref) / bound))


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_dense_dmma_contraction_vs_longdouble(dev, monkeypatch, axis):
    """poms_axis_dense_dmma (the eigenbasis contractions of CoarseSolver) at every K-chunk / tile edge
    up to the 8-GPU replicated coarse grid (259), square and rectangular Q; the gather kernel
    (POMS_B200_DENSE=gather) must meet the same bound, so the two agree to within twice of it."""
    from poms_b200 import mg
    sizes = [(n, n) for n in DENSE_N] + [(130, 11), (67, 131), (33, 65)]
    for mode in ("dmma", "gather"):
        monkeypatch.setenv("POMS_B200_DENSE", mode)
        assert mg._dense_mode() == mode
        for n_in, n_out in sizes:
            err = _dense_case(dev, n_in, n_out, axis, seed=n_in * 7 + n_out)
            assert err <= 1.0, (mode, n_in, n_out, err)


def _fd_oracle(p, knots, b):
    """x = A^-1 b by the oracle's eigenpair solve (scipy eigh of the oracle's own assembly), the 1-D
    condition numbers cond(M_a) and an estimate of ||A||_2 from the 1-D factors."""
    from scipy.linalg import eigh
    from oracle import poms_oracle as po
    Ao, Mb, Kb = po.poisson_operator(p, knots)
    d = len(knots)
    Qs, D, condM, nM, nK = [], 1.0, [], [], []
    for a in range(d):
        Md, Kd = po.band_to_dense(Mb[a]), po.band_to_dense(Kb[a])
        w, Q = eigh(0.5 * (Kd + Kd.T), 0.5 * (Md + Md.T))
        Qs.append(Q)
        shp = [1] * d
        shp[a] = len(w)
        D = D + w.reshape(shp)
        condM.append(np.linalg.cond(Md))
        nM.append(np.linalg.norm(Md, 2))
        nK.append(np.linalg.norm(Kd, 2))
    z = b
    for a, Q in enumerate(Qs):
        z = np.moveaxis(np.tensordot(Q.T, z, axes=(1, a)), 0, a)
    z = z / D
    for a, Q in enumerate(Qs):
        z = np.moveaxis(np.tensordot(Q, z, axes=(1, a)), 0, a)
    normA = np.prod(nM) + sum(nK[a] * np.prod([nM[c] for c in range(d) if c != a]) for a in range(d))
    return Ao, z, condM, normA


COARSE = [(3, (35, 35, 35)), (3, (67, 67, 67)), (3, (131, 131, 131)), (3, (259, 35, 35)), (3, (131, 35, 67)),
          (5, (69, 133))]


@pytest.mark.parametrize("setup", ["host", "device"])
@pytest.mark.parametrize("grading", ["uniform", "graded"])
@pytest.mark.parametrize("p,npts", COARSE)
def test_coarse_solver_real_sizes(dev, p, npts, grading, setup):
    """CoarseSolver on the coarse grids the hierarchy builds (C3 35^3 and 67^3, C5 131^3, the 8-GPU
    replicated 259 x 35 x 35, an anisotropic grid, a 2-D C4-like grid): the residual against the oracle
    operator is at rounding level of ||A|| ||x||, and x agrees with the oracle's eigenpair solve to a
    tolerance scaled by the 1-D condition numbers of the mass matrices (the eigenbases are M-orthonormal,
    ||Q||^2 = 1 / lambda_min(M))."""
    from poms_b200 import setup_device as sd
    from poms_b200.stencil import KronSumMatrix
    from poms_b200.mg import CoarseSolver
    kn = (lambda n: power(p, n - p)) if grading == "graded" else (lambda n: uniform(p, n - p))
    knots = [kn(n) for n in npts]
    A = KronSumMatrix.poisson(p, knots)
    if setup == "device":
        with sd.device_setup(True, dev):
            cs = CoarseSolver(A, dev)
    else:
        cs = CoarseSolver(A, dev)
    for op in cs.Q + cs.Qt:
        assert op.dense                    # the tensor-core contraction, not a W = n gather
    V = _space(npts, [p] * len(npts), dev)
    b = np.random.default_rng(sum(npts)).standard_normal(npts)
    x = _arr(cs.solve(_vec(V, b)))
    Ao, xo, condM, normA = _fd_oracle(p, knots, b)
    r = b - Ao.dot(x)
    res = np.linalg.norm(r) / (normA * np.linalg.norm(x))
    assert res < 2 * max(npts) * EPS, res
    tol = 8 * EPS * sum(n * c for n, c in zip(npts, condM))
    err = rel(x, xo)
    assert err < tol, (err, tol)


# ----------------------------------------------------------------------------- 4. graded-mesh solves
def _manufactured(d):
    pi = np.pi
    u = lambda *X: torch.cos(pi * X[0]) * (torch.cos(pi * X[1]) if d == 2 else torch.cos(pi * X[1]) * torch.cos(pi * X[2]))
    f = lambda *X: (1.0 + d * pi * pi) * u(*X)

    def gu(*X):
        c = [torch.cos(pi * t) for t in X]
        s = [-pi * torch.sin(pi * t) for t in X]
        res = []
        for a in range(d):
            out = None
            for b_ in range(d):
                v = s[b_] if a == b_ else c[b_]
                out = v if out is None else out * v
            res.append(out)
        return tuple(res)
    return u, f, gu


@pytest.mark.parametrize("p,d,Ns", [(2, 3, (8, 16, 32)), (3, 3, (8, 16, 32)), (5, 2, (8, 16, 32, 64))])
def test_graded_mesh_solve_converges(dev, p, d, Ns):
    """u = prod cos(pi x_a) (natural boundary condition) from f = (1 + d pi^2) u on power-graded meshes,
    solved exactly by fast diagonalisation (CoarseSolver: a Kronecker sum needs no iteration), so that
    nothing is taken from the mat-vec but the residual check; the errors come from the quadrature of
    fem.error_norms against u and grad u.  Orders as in test_fem.test_manufactured_convergence."""
    from poms_b200 import fem
    from poms_b200.stencil import KronSumMatrix, StencilVector, EPI_RESID
    from poms_b200.mg import CoarseSolver
    u, f, gu = _manufactured(d)
    rows = []
    for N in Ns:
        knots = [power(p, N)] * d
        A = KronSumMatrix.poisson(p, knots)
        kinds = ("pow",) * d
        check_dispatch(A, kinds, p)
        V = _space(A.npts, [p] * d, dev)
        b = fem.load_vector(V, knots, p, f)
        x = CoarseSolver(A, dev).solve(b)
        r = StencilVector(V)
        A.apply(x, r, EPI_RESID, b=b)
        # fast diagonalisation is not backward stable to eps: its residual grows with the conditioning of
        # the mass matrices and the stiffness spread (numpy / scipy in fp64 leave 1.1e-12 ||b|| for a random
        # b at 2-D p = 5, N = 64 on this grading), so 2-D p = 5 gets a decade more than the 3-D cases
        tol = 1e-12 if d == 3 else 1e-11
        assert np.sqrt(r.dot(r)) <= tol * np.sqrt(b.dot(b))
        e = fem.error_norms(x, knots, p, u, gu)
        rows.append((N, e["l2"], e["h1"]))
    rows = [rw for rw in rows if rw[1] > 1e-10]
    assert len(rows) >= 2, rows
    (N0, l0, h0), (N1, l1, h1) = rows[-2], rows[-1]
    ol2, oh1 = np.log(l0 / l1) / np.log(N1 / N0), np.log(h0 / h1) / np.log(N1 / N0)
    assert ol2 >= p + 1 - 0.25 and oh1 >= p - 0.25, (rows, ol2, oh1)


def test_mg_pcg_3d_p5_vs_oracle(dev):
    """The degree-5 instantiations of the 3-D kernels inside a full V-cycle (no 3-D p = 5 solve is
    tested elsewhere), with the assertions of test_gpu_parity.test_mg_pcg_vs_oracle."""
    from poms_b200.mg import Hierarchy, mg_pcg
    from poms_b200.stencil import StencilVector
    from oracle import poms_oracle as po
    p, N = 5, [24, 24, 24]
    h = Hierarchy(p, N, device=dev, smoother="glt", nu=1)
    ho = po.MGHierarchy(p, N, smoother="glt", nu=1)
    assert len(h.levels) == len(ho.levels) >= 2
    for a, b_ in zip(h.levels[:-1], ho.levels[:-1]):
        assert abs(a.lmax - b_["lmax"]) < 1e-9 * b_["lmax"]
    b = StencilVector(h.levels[0].V)
    b.data.fill_(1.0)
    x, info = mg_pcg(h, b, tol=1e-10, maxiter=100)
    xo, io = ho.mg_pcg(np.ones(h.levels[0].V.npts), tol=1e-10, maxiter=100)
    assert info["niter"] == io["niter"] and info["success"] and io["success"]
    assert np.allclose(info["history"], io["history"], rtol=1e-6)
    assert np.allclose(info["history"][:5], io["history"][:5], rtol=1e-10)
    assert rel(_arr(x), xo) < 1e-9
    assert info["res_norm"] <= 1e-10 * info["res_norm0"]
