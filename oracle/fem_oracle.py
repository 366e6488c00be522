"""NumPy oracle of poms_b200.fem: dense per-axis quadrature matrices and einsum contractions (small grids).

Same tables as the package (bsplines.quadrature_tables): per axis a, m_a = (elements) x (p+1) points,
    B_a[i, j] = phi_i(x_j)   (n_a x m_a),   D_a = derivatives,   w_a = weights (m_a,)."""
import numpy as np

from poms_b200 import bsplines as bs


def axis_matrices(T, p):
    t = bs.quadrature_tables(T, p)
    E, Q = t["x"].shape
    n = t["n"]
    B = np.zeros((n, E * Q))
    D = np.zeros((n, E * Q))
    for e in range(E):
        for k in range(p + 1):
            B[t["first"][e] + k, e * Q:(e + 1) * Q] = t["v"][e, k]
            D[t["first"][e] + k, e * Q:(e + 1) * Q] = t["d"][e, k]
    return {"x": t["x"].reshape(-1), "w": t["w"].reshape(-1), "B": B, "D": D}


def _contract(mats, arr):
    """out[i, j, k] = sum_{a, b, c} mats[0][i, a] mats[1][j, b] mats[2][k, c] arr[a, b, c] (d = 2, 3)."""
    d = len(mats)
    spec = ",".join("%s%s" % (o, l) for o, l in zip("ijk"[:d], "abc"[:d])) + "," + "abc"[:d] + "->" + "ijk"[:d]
    return np.einsum(spec, *mats, arr, optimize=True)


def load_vector(knots, p, f):
    """b_i = sum_q w_q f(x_q) phi_i(x_q); f takes d broadcastable coordinate arrays."""
    ax = [axis_matrices(T, p) for T in knots]
    d = len(ax)
    xs = np.meshgrid(*[a["x"] for a in ax], indexing="ij", sparse=True)
    F = np.broadcast_to(f(*xs), tuple(len(a["x"]) for a in ax)).astype(float)
    W = [a["B"] * a["w"][None, :] for a in ax]
    return _contract(W, F)


def values(knots, p, x, deriv=None):
    """u_h (deriv None) or d u_h / dx_deriv at every quadrature point, coefficients x of shape npts."""
    ax = [axis_matrices(T, p) for T in knots]
    mats = [(a["D"] if i == deriv else a["B"]).T for i, a in enumerate(ax)]
    d = len(ax)
    spec = ",".join("%s%s" % (l, o) for l, o in zip("abc"[:d], "ijk"[:d])) + "," + "ijk"[:d] + "->" + "abc"[:d]
    return np.einsum(spec, *mats, x, optimize=True)


def error_norms(knots, p, x, u, grad_u=None):
    ax = [axis_matrices(T, p) for T in knots]
    d = len(ax)
    xs = np.meshgrid(*[a["x"] for a in ax], indexing="ij", sparse=True)
    shape = tuple(len(a["x"]) for a in ax)
    w = np.ones(shape)
    for i, a in enumerate(ax):
        w = w * a["w"].reshape([-1 if j == i else 1 for j in range(d)])
    eu = np.broadcast_to(u(*xs), shape) - values(knots, p, x)
    l2 = float(np.sqrt(np.sum(w * eu ** 2)))
    h1 = None
    if grad_u is not None:
        g = grad_u(*xs)
        h1 = float(np.sqrt(sum(np.sum(w * (np.broadcast_to(g[i], shape) - values(knots, p, x, i)) ** 2)
                               for i in range(d))))
    return {"l2": l2, "h1": h1}
