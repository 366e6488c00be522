"""Host-side dispatch of the mat-vec kernels on the knot families of tests/test_gpu_nonuniform.py: the
Toeplitz interior ranges `KronSumMatrix._toeplitz` hands to the TMA kernels and the symmetry predicate
that picks the kernel variant (restated from poms_matvec3d_tma.cuh / poms_matvec2d_tma.cuh), pinned per
family and degree, and for the exact inputs of every GPU case there, so that a change of the host code
that moves a case onto another branch fails here first."""
import numpy as np
import pytest

import test_gpu_nonuniform as nu
from poms_b200 import bsplines as bs
from poms_b200.stencil import KronSumMatrix


def _asym(row):
    return np.abs(row - row[::-1]).max() / np.abs(row).max()


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("kind", ["u", "pow", "bl", "cos", "jit"])
def test_family_ranges_and_symmetry(kind, p):
    knots = nu.family_knots(kind, p, 40)
    n = len(knots) - p - 1
    assert bs._is_uniform_open(knots, p) == (kind == "u")
    A = KronSumMatrix.poisson(p, [knots] * 3)
    coef, rng = A._toeplitz()
    assert list(rng) == list(rng[:2]) * 3 and nu.range_ok(kind, p, n, *rng[:2])
    # the middle row's asymmetry decides the branch: ~1e-2 (power), ~1e-11 (jitter) above the kernels'
    # 1e-13, rounding level (uniform, boundary layer, cosine with an odd number of functions) below it
    a = max(_asym(coef[ax, j]) for ax in (1, 2) for j in (0, 1))
    if kind == "pow":
        assert a > 1e-3
    elif kind == "jit":
        assert 1e-12 < a < 1e-9
    else:
        assert a < 2e-14
    assert nu.tma_sym(A) == (kind not in ("pow", "jit")) == nu.expected_sym((kind,) * 3, p, A.npts)
    # the same predicate with the threshold restated literally from the kernels
    sym = all(np.all(np.abs(r - r[::-1]) <= 1e-13 * np.abs(r).max()) for ax in (1, 2) for r in coef[ax])
    assert sym == nu.tma_sym(A)
    # a single Kronecker product is never sent to variant 0 by the predicate
    assert nu.tma_sym(KronSumMatrix(A.Ms))


def test_cosine_parity_decides_symmetry():
    """An even number of functions puts the mirror image of the middle row one row away: asymmetric."""
    for p in (2, 4):
        T = nu.cosine(p, 40)                   # n = 40 + p even
        A = KronSumMatrix.poisson(p, [T] * 3)
        assert not nu.tma_sym(A)
        assert nu.tma_sym(KronSumMatrix.poisson(p, [nu.family_knots("cos", p, 40)] * 3))


@pytest.mark.parametrize("name,p", nu.OP3_CASES)
def test_gpu_operator_cases_take_their_branch(name, p):
    kinds = nu.GRADED3.get(name, ("u", "u", "u"))
    knots = [nu.family_knots(k, p, N) for k, N in zip(kinds, nu.SHAPE3[p])]
    A = KronSumMatrix.poisson(p, knots)
    nu.check_dispatch(A, kinds, p)
    rng = A._toeplitz()[1]
    if name == "uniform":
        assert rng[5] - rng[4] > 64
    else:
        assert any(rng[2 * a + 1] - rng[2 * a] == 1 for a in range(3))


@pytest.mark.parametrize("name", list(nu.GRADED2))
def test_gpu_2d_cases_take_their_branch(name):
    kinds = nu.GRADED2[name]
    for p in range(1, 6):
        A = KronSumMatrix.poisson(p, [nu.family_knots(k, p, N) for k, N in zip(kinds, (120, 500))])
        nu.check_dispatch(A, kinds, p)
        assert nu.tma_sym(A) == (kinds[1] == "u")


@pytest.mark.parametrize("p", [1, 3, 5])
def test_synthetic_ranges_stay_inside_identical_rows(p):
    """The synthetic ranges of the GPU test lie inside the bit-identical rows of the uniform bands, begin
    past the 2p boundary rows, and off the 64-column / 16-row tile edges."""
    A = KronSumMatrix.poisson(p, [nu.uniform(p, N) for N in nu.SYNTH_N])
    full = A._toeplitz()[1]
    for which, r in nu._synthetic_ranges(A.npts, p).items():
        for a, (lo, hi) in enumerate(r):
            assert full[2 * a] <= lo <= hi <= full[2 * a + 1], (which, a)
            if which != "empty":
                assert lo > 2 * p and hi < A.npts[a] - 2 * p
            if which == "short":
                assert hi - lo < (64 if a == 2 else 16)
        if which == "deep":
            assert all(lo % 16 and hi % 16 for lo, hi in r)
