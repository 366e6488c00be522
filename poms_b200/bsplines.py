"""Host-side 1-D B-spline setup (O(n p^2) work, runs once per level; SURVEY.md section 8f-2).

What the reference gets from the third-party `spl` package (absent from its tree):
`make_open_knots`, `matrix_multi_stages`, `collocation_cardinal_splines`
(/root/reference/sources/mg_jac.py:28-29,67; mg_glt.py:115-116) and the 1-D integrals
accumulated by `assembly_1d` (/root/reference/sources/matrix_assembler.py:10-77).  Everything
here returns small NumPy arrays that the device wrappers in stencil.py upload once.

Band convention: (n, 2p+1) array, band[i, k] = A[i, i+k-p]
(/root/reference/pyccel/pyccel_functions.py:15,19).
"""
import numpy as np

__all__ = ["make_open_knots", "assemble_1d_bands", "assemble_1d_advection", "knot_insertion_rows", "rows_transpose",
           "glt_band", "cardinal_bspline_values", "band_to_lapack", "band_lu", "pad_band",
           "band_to_dense", "dense_to_band"]


def make_open_knots(p, n):
    """Clamped uniform knot vector with n basis functions of degree p (length n+p+1).
    Interior knots are the correctly rounded i/(n-p): nested meshes share them bit for bit,
    which `knots_to_insert` relies on (/root/reference/sources/multilevels.py:22)."""
    N = n - p
    if N < 1:
        raise ValueError("need at least one element: n > p")
    T = np.zeros(n + p + 1)
    T[p + 1:n] = np.arange(1, N, dtype=float) / N
    T[n:] = 1.0
    return T


def _all_basis(T, p, spans, x):
    """Values and first derivatives of the p+1 non-zero degree-p B-splines at points
    x[e, g] lying in knot span spans[e].  Vectorised de Boor triangle over all elements.
    Returns (vals, ders) of shape (ne, p+1, nq)."""
    ne, nq = x.shape
    left = np.zeros((p + 1, ne, nq))
    right = np.zeros((p + 1, ne, nq))
    N = np.zeros((p + 1, ne, nq))
    Nprev = None
    N[0] = 1.0
    for d in range(1, p + 1):
        left[d] = x - T[spans + 1 - d][:, None]
        right[d] = T[spans + d][:, None] - x
        if d == p:
            Nprev = N.copy()  # degree p-1 values (first p entries)
        saved = np.zeros((ne, nq))
        for r in range(d):
            den = right[r + 1] + left[d - r]
            tmp = N[r] / den
            N[r] = saved + right[r + 1] * tmp
            saved = left[d - r] * tmp
        N[d] = saved
    vals = np.moveaxis(N, 0, 1)
    ders = np.zeros_like(N)
    if p >= 1:
        if p == 1:
            Nprev = np.zeros_like(N)
            Nprev[0] = 1.0
        for j in range(p + 1):
            i = spans - p + j  # global index of the j-th local function
            if j >= 1:
                den = (T[i + p] - T[i])[:, None]
                ders[j] += p * Nprev[j - 1] / den
            if j <= p - 1:
                den = (T[i + p + 1] - T[i + 1])[:, None]
                ders[j] -= p * Nprev[j] / den
    return vals, np.moveaxis(ders, 0, 1)


def assemble_1d_bands(p, T, toeplitz_interior=True):
    """1-D mass and stiffness bands (n, 2p+1) on knot vector T, Gauss-Legendre with p+1
    points per element (exact): the v_m / v_s integrals of
    /root/reference/sources/matrix_assembler.py:59-74."""
    T = np.asarray(T, dtype=float)
    n = len(T) - p - 1
    spans = np.array([k for k in range(p, n) if T[k + 1] > T[k]], dtype=np.int64)
    a, b = T[spans], T[spans + 1]
    u, w = np.polynomial.legendre.leggauss(p + 1)
    x = 0.5 * (a + b)[:, None] + 0.5 * (b - a)[:, None] * u[None, :]
    wq = 0.5 * (b - a)[:, None] * w[None, :]
    v, dv = _all_basis(T, p, spans, x)
    Me = np.einsum("eiq,ejq,eq->eij", v, v, wq)
    Ke = np.einsum("eiq,ejq,eq->eij", dv, dv, wq)
    M = np.zeros((n, 2 * p + 1))
    K = np.zeros((n, 2 * p + 1))
    for il in range(p + 1):
        rows = spans - p + il
        for jl in range(p + 1):
            np.add.at(M, (rows, jl - il + p), Me[:, il, jl])
            np.add.at(K, (rows, jl - il + p), Ke[:, il, jl])
    if toeplitz_interior and n > 4 * p + 1 and _is_uniform_open(T, p):
        # On a uniform open knot vector the functions p .. n-1-p are translates of one B-spline, so
        # rows 2p .. n-2p-1 are mathematically identical; quadrature at different abscissae leaves
        # them equal only to ~1 ulp.  Make them bit-identical (copy the middle row): the kernels
        # can then take interior coefficients from the constant bank instead of memory.
        mid = n // 2
        M[2 * p:n - 2 * p] = M[mid]
        K[2 * p:n - 2 * p] = K[mid]
    return M, K


def assemble_1d_advection(p, T, toeplitz_interior=True):
    """1-D advection band G (n, 2p+1), G[i, k] = int phi_{i+k-p}' phi_i, with the Gauss rule of
    `assemble_1d_bands` (exact: the integrand has degree 2p-1).  G is not symmetric; integration by parts
    gives G + G^T = e_{n-1} e_{n-1}^T - e_0 e_0^T on an open knot vector.  On uniform open knots rows
    2p .. n-2p-1 are made bit-identical to the middle row, as in `assemble_1d_bands`."""
    T = np.asarray(T, dtype=float)
    n = len(T) - p - 1
    spans = np.array([k for k in range(p, n) if T[k + 1] > T[k]], dtype=np.int64)
    a, b = T[spans], T[spans + 1]
    u, w = np.polynomial.legendre.leggauss(p + 1)
    x = 0.5 * (a + b)[:, None] + 0.5 * (b - a)[:, None] * u[None, :]
    wq = 0.5 * (b - a)[:, None] * w[None, :]
    v, dv = _all_basis(T, p, spans, x)
    Ge = np.einsum("eiq,ejq,eq->eij", v, dv, wq)          # Ge[e, il, jl] = int phi_jl' phi_il
    G = np.zeros((n, 2 * p + 1))
    for il in range(p + 1):
        rows = spans - p + il
        for jl in range(p + 1):
            np.add.at(G, (rows, jl - il + p), Ge[:, il, jl])
    if toeplitz_interior and n > 4 * p + 1 and _is_uniform_open(T, p):
        G[2 * p:n - 2 * p] = G[n // 2]
    return G


def quadrature_tables(T, p):
    """Per-element Gauss-Legendre tables of the (p+1)-point rule of `assemble_1d_bands` on the non-empty
    knot spans of T: points x (ne, p+1), weights w (ne, p+1), basis values v and first derivatives d
    (ne, p+1 functions, p+1 points) and the index `first` (ne,) of each element's first basis function."""
    T = np.asarray(T, dtype=float)
    n = len(T) - p - 1
    spans = np.array([k for k in range(p, n) if T[k + 1] > T[k]], dtype=np.int64)
    a, b = T[spans], T[spans + 1]
    u, w = np.polynomial.legendre.leggauss(p + 1)
    x = 0.5 * (a + b)[:, None] + 0.5 * (b - a)[:, None] * u[None, :]
    wq = 0.5 * (b - a)[:, None] * w[None, :]
    v, dv = _all_basis(T, p, spans, x)
    return {"n": n, "x": x, "w": wq, "v": v, "d": dv, "first": spans - p}


def _is_uniform_open(T, p):
    """True if T is a clamped knot vector with equally spaced simple interior knots."""
    n = len(T) - p - 1
    if np.any(T[:p + 1] != T[0]) or np.any(T[n:] != T[-1]):
        return False
    h = np.diff(T[p:n + 1])
    return bool(np.all(h > 0) and np.max(np.abs(h - h.mean())) <= 8 * np.finfo(float).eps * abs(T[-1] - T[0]))


def knot_insertion_rows(Tc, Tf, p):
    """Knot-insertion (prolongation) matrix P1 of shape (n_f, n_c) between nested knot
    vectors Tc subset Tf, in row-compressed form: (start, coef) with
    P1[i, start[i] + w] = coef[i, w], w = 0..p.  Same matrix as
    `matrix_multi_stages(ts, nc, p, Tc)` (/root/reference/sources/mg_jac.py:67), built with
    the Oslo recursion (discrete B-splines) in O(n_f p^2) instead of a product of n_f - n_c
    dense Boehm matrices."""
    Tc = np.asarray(Tc, dtype=float)
    Tf = np.asarray(Tf, dtype=float)
    nc = len(Tc) - p - 1
    nf = len(Tf) - p - 1
    i = np.arange(nf)
    # coarse span mu of each fine knot Tf[i]: Tc[mu] <= Tf[i] < Tc[mu+1], clamped to [p, nc-1]
    mu = np.clip(np.searchsorted(Tc, Tf[:nf], side="right") - 1, p, nc - 1)
    # alpha[w] <-> coarse index j = mu - k + w at recursion level k (k+1 entries)
    alpha = np.zeros((p + 1, nf))
    alpha[0] = 1.0
    for k in range(1, p + 1):
        new = np.zeros((p + 1, nf))
        tau = Tf[i + k]
        for w in range(k + 1):
            j = mu - k + w
            acc = np.zeros(nf)
            if w >= 1:  # alpha_{j,k-1} is old entry w-1
                den = Tc[j + k] - Tc[j]
                ok = den > 0
                t = np.zeros(nf)
                t[ok] = (tau[ok] - Tc[j][ok]) / den[ok]
                acc += t * alpha[w - 1]
            if w <= k - 1:  # alpha_{j+1,k-1} is old entry w
                den = Tc[j + k + 1] - Tc[j + 1]
                ok = den > 0
                t = np.zeros(nf)
                t[ok] = (Tc[j + k + 1][ok] - tau[ok]) / den[ok]
                acc += t * alpha[w]
            new[w] = acc
        alpha = new
    start = (mu - p).astype(np.int32)
    coef = np.ascontiguousarray(alpha.T)
    return start, coef, nc


def rows_transpose(start, coef, n_cols):
    """Row-compressed form of the transpose (restriction R1 = P1^T,
    /root/reference/sources/mg_jac.py:68): returns (start_t, coef_t) with
    R1[j, start_t[j] + w] = coef_t[j, w]."""
    n_rows, W = coef.shape
    lo = np.full(n_cols, n_rows, dtype=np.int64)
    hi = np.full(n_cols, -1, dtype=np.int64)
    for w in range(W):
        j = start + w
        nz = coef[:, w] != 0.0
        ii = np.nonzero(nz)[0]
        np.minimum.at(lo, j[ii], ii)
        np.maximum.at(hi, j[ii], ii)
    empty = hi < lo
    lo[empty] = 0
    hi[empty] = 0
    Wt = int((hi - lo).max()) + 1
    coef_t = np.zeros((n_cols, Wt))
    for w in range(W):
        j = start + w
        nz = coef[:, w] != 0.0
        ii = np.nonzero(nz)[0]
        coef_t[j[ii], ii - lo[j[ii]]] = coef[ii, w]
    return lo.astype(np.int32), coef_t


def rows_to_dense(start, coef, n_cols):
    n_rows, W = coef.shape
    A = np.zeros((n_rows, n_cols))
    for w in range(W):
        j = start + w
        ok = (j >= 0) & (j < n_cols)
        A[np.nonzero(ok)[0], j[ok]] += coef[ok, w]
    return A


def dense_to_rows(A):
    """Row-compressed (start, coef) form of a dense matrix (general transfer operators such
    as the reference's direct fine -> nc jump, whose columns are wide)."""
    n_rows, n_cols = A.shape
    lo = np.zeros(n_rows, dtype=np.int32)
    width = 1
    nzr = [np.nonzero(A[i])[0] for i in range(n_rows)]
    for i, nz in enumerate(nzr):
        if len(nz):
            lo[i] = nz[0]
            width = max(width, nz[-1] - nz[0] + 1)
    coef = np.zeros((n_rows, width))
    for i in range(n_rows):
        hi = min(n_cols, lo[i] + width)
        coef[i, :hi - lo[i]] = A[i, lo[i]:hi]
    return lo, coef


def cardinal_bspline_values(q):
    """phi_q at its interior abscissae (q+1)/2 + k, |k| <= q//2 + ...: the symmetric stencil
    of the cardinal B-spline of degree q (integer points for odd q, midpoints for even q)."""
    # phi_q(x) = sum_{j=0}^{q+1} (-1)^j C(q+1, j) (x-j)_+^q / q!
    from math import comb, factorial
    half = (q + 1) // 2
    ks = np.arange(-half, half + 1)
    x = (q + 1) / 2.0 + ks
    v = np.zeros(len(ks))
    for j in range(q + 2):
        v += (-1) ** j * comb(q + 1, j) * np.maximum(x - j, 0.0) ** q
    v /= factorial(q)
    v[np.abs(v) < 1e-15] = 0.0
    return ks, v


def glt_band(p, n, degree=None):
    """Symmetric Toeplitz band t_k = phi_q((q+1)/2 + k) (q = `degree`, default p) stored with
    half-bandwidth p: the band `array_to_mat_stencil(n, p, collocation_cardinal_splines(p, n))`
    hands to pcg_glt (/root/reference/sources/mg_glt.py:115-118).  The third-party
    `collocation_cardinal_splines` is UNPINNED; see DESIGN.md."""
    q = p if degree is None else degree
    ks, v = cardinal_bspline_values(q)
    band = np.zeros((n, 2 * p + 1))
    for k, val in zip(ks, v):
        if abs(k) <= p and val != 0.0:
            i = np.arange(max(0, -k), min(n, n - k))
            band[i, k + p] = val
    return band


def band_to_dense(band):
    n, w = band.shape
    p = (w - 1) // 2
    A = np.zeros((n, n))
    for k in range(-p, p + 1):
        i = np.arange(max(0, -k), min(n, n - k))
        A[i, i + k] = band[i, k + p]
    return A


def dense_to_band(A, p):
    n = A.shape[0]
    band = np.zeros((n, 2 * p + 1))
    for k in range(-p, p + 1):
        i = np.arange(max(0, -k), min(n, n - k))
        band[i, k + p] = A[i, i + k]
    return band


def pad_band(band, P):
    """Embed an (n, 2p+1) band into half-bandwidth P >= p (zero outer diagonals)."""
    n, w = band.shape
    p = (w - 1) // 2
    if p == P:
        return np.ascontiguousarray(band, dtype=np.float64)
    if p > P:
        raise ValueError("cannot shrink a band")
    out = np.zeros((n, 2 * P + 1))
    out[:, P - p:P + p + 1] = band
    return out


def band_to_lapack(band):
    """(n, 2p+1) band -> LAPACK general band storage for dgbtrf, shape (3p+1, n):
    AB[kl+ku+i-j, j] = A[i, j] (/root/reference/sources/tests/test_kron_solve_bnd.py:30-42)."""
    n, w = band.shape
    p = (w - 1) // 2
    ab = np.zeros((3 * p + 1, n))
    for k in range(-p, p + 1):
        i = np.arange(max(0, -k), min(n, n - k))
        ab[2 * p - k, i + k] = band[i, k + p]
    return ab, p, p


def band_lu(band):
    """dgbtrf of a band matrix -> (lu_band, kl, ku, ipiv): the `[A_bnd, la, ua, A_piv]` list
    kron_solve_bnd_par takes (/root/reference/sources/kron_product.py:191-197)."""
    from scipy.linalg.lapack import dgbtrf
    ab, kl, ku = band_to_lapack(band)
    lub, piv, info = dgbtrf(ab, kl, ku)
    if info != 0:
        raise np.linalg.LinAlgError("dgbtrf failed with info=%d" % info)
    return lub, kl, ku, piv


# ---------------------------------------------------------------------------------------------
# polynomial approximation of a banded SPD Toeplitz-type inverse (EXTENSION: smoother of mg.py)
# ---------------------------------------------------------------------------------------------
def symbol_range(band):
    """[min, max] of the symbol t_0 + 2 sum_k t_k cos(k theta) of the middle row of a symmetric
    band; the eigenvalues of the (truncated) Toeplitz matrix lie inside."""
    n, w = band.shape
    p = (w - 1) // 2
    row = band[n // 2]
    th = np.linspace(0.0, np.pi, 4097)
    m = row[p] + 2.0 * sum(row[p + k] * np.cos(k * th) for k in range(1, p + 1))
    return float(m.min()), float(m.max())


def cheb_inverse_poly(lmin, lmax, degree):
    """Monomial coefficients c_0..c_k of q(t) = (1 - T_{k+1}((a-t)/d) / T_{k+1}(a/d)) / t, the
    Chebyshev approximation of 1/t on [lmin, lmax] (a, d = centre, half-width)."""
    from numpy.polynomial import chebyshev as C, polynomial as P
    a, d = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    mono = C.Chebyshev.basis(degree + 1).convert(kind=np.polynomial.Polynomial).coef
    s_poly = np.array([a / d, -1.0 / d])
    out, powr = np.zeros(1), np.ones(1)
    for c in mono:
        out = P.polyadd(out, c * powr)
        powr = P.polymul(powr, s_poly)
    out = out / C.Chebyshev.basis(degree + 1)(a / d)
    num = P.polysub(np.ones(1), out)
    return num[1:]


def band_matmul(A, B):
    """Band of the product of two banded matrices given as (n, 2p+1) bands."""
    n = A.shape[0]
    pa, pb = (A.shape[1] - 1) // 2, (B.shape[1] - 1) // 2
    pc = pa + pb
    Cb = np.zeros((n, 2 * pc + 1))
    for ka in range(-pa, pa + 1):
        for kb in range(-pb, pb + 1):
            i = np.arange(n)
            j = i + ka                      # A[i, j] * B[j, j + kb]
            ok = (j >= 0) & (j < n) & (j + kb >= 0) & (j + kb < n)
            Cb[i[ok], ka + kb + pc] += A[i[ok], ka + pa] * B[j[ok], kb + pb]
    return Cb


def poly_inverse_factors(band, degree=3, widen=0.02):
    """Banded factors F_1, F_2 (half-bandwidths q and (degree-1) q) with F_2 F_1 = q_degree(T) ~ T^-1:
    q(t) = c_k (t - r)(monic polynomial of degree k-1), r a real root (odd degree) -- two narrow band
    passes per axis instead of one wide one.  `band` is trimmed to its true half-bandwidth q first."""
    from numpy.polynomial import polynomial as P
    band = np.asarray(band, dtype=np.float64)
    p = (band.shape[1] - 1) // 2
    q = p
    while q > 0 and not band[:, p - q].any() and not band[:, p + q].any():
        q -= 1
    T = band[:, p - q:p + q + 1]
    n = T.shape[0]
    lo, hi = symbol_range(T)
    c = cheb_inverse_poly(lo * (1.0 - widen), hi * (1.0 + widen), degree)
    roots = P.polyroots(c)
    real = roots[np.abs(roots.imag) < 1e-9 * max(1.0, np.abs(roots).max())].real
    eye = np.zeros((n, 2 * q + 1))
    eye[:, q] = 1.0
    if len(real) == 0 or degree < 2:
        F1 = c[0] * eye.copy() if degree == 0 else None
        raise ValueError("use an odd degree >= 3 (or 2 with a real root)")
    r = real[np.argmax(np.abs(real))]
    rest = P.polydiv(c, np.array([-r, 1.0]))[0]          # q(t) = (t - r) * rest(t)
    F1 = T - r * eye
    # Horner for rest(T), starting from a diagonal band
    F2 = np.full((n, 1), rest[-1])
    for coef in rest[-2::-1]:
        F2 = band_matmul(F2, T)
        w2 = (F2.shape[1] - 1) // 2
        F2[:, w2] += coef
    # make the Toeplitz-interior rows bit-identical (they are equal up to rounding)
    for F in (F1, F2):
        w = (F.shape[1] - 1) // 2
        if n > 4 * w + 1:
            F[2 * w:n - 2 * w] = F[n // 2]
    return F1, F2
