"""Dense NumPy restatement of the particle coupling of poms_b200.fem (evaluate_points, deposit), for small
problems: per-axis design matrices at the points (values and first derivatives) and einsum contractions.
Test infrastructure only, like oracle/fem_oracle.py, whose conventions it follows."""
import numpy as np

from poms_b200 import bsplines as bs


def point_matrices(T, p, x):
    """Dense design matrices at the points x (m,): B[k, i] = phi_i(x_k) and D[k, i] = phi_i'(x_k) (m x n).
    x_k belongs to the span T[s] <= x_k < T[s+1]; x_k = T[n] to the last non-empty span."""
    T = np.asarray(T, dtype=float)
    x = np.asarray(x, dtype=float).reshape(-1)
    n = len(T) - p - 1
    last = max(k for k in range(p, n) if T[k + 1] > T[k])
    spans = np.clip(np.searchsorted(T, x, side="right") - 1, p, last)
    v, dv = bs._all_basis(T, p, spans, x[:, None])
    rows, cols = np.arange(len(x))[:, None], spans[:, None] - p + np.arange(p + 1)[None, :]
    B = np.zeros((len(x), n))
    D = np.zeros((len(x), n))
    B[rows, cols] = v[:, :, 0]
    D[rows, cols] = dv[:, :, 0]
    return B, D


def _at_points(mats, x):
    """out[k] = sum_{i, j, l} mats[0][k, i] mats[1][k, j] mats[2][k, l] x[i, j, l] (d = 2, 3)."""
    d = len(mats)
    spec = ",".join("k" + c for c in "ijl"[:d]) + "," + "ijl"[:d] + "->k"
    return np.einsum(spec, *mats, x, optimize=True)


def evaluate_points(knots, p, x, points):
    """(u_h(points[k]), grad u_h(points[k])) for coefficients x of shape npts and points (m, d)."""
    points = np.asarray(points, dtype=float)
    BD = [point_matrices(T, p, points[:, a]) for a, T in enumerate(knots)]
    d = len(knots)
    u = _at_points([B for B, _ in BD], x)
    g = np.stack([_at_points([BD[b][1] if b == a else BD[b][0] for b in range(d)], x) for a in range(d)], axis=1)
    return u, g


def deposit(knots, p, points, weights):
    """b[i, j, l] = sum_k weights[k] phi_i(points[k, 0]) phi_j(points[k, 1]) (phi_l(points[k, 2]))."""
    points = np.asarray(points, dtype=float)
    mats = [point_matrices(T, p, points[:, a])[0] for a, T in enumerate(knots)]
    d = len(knots)
    spec = "k," + ",".join("k" + c for c in "ijl"[:d]) + "->" + "ijl"[:d]
    return np.einsum(spec, np.asarray(weights, dtype=float), *mats, optimize=True)
