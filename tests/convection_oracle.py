"""NumPy oracle of the constant-velocity convection term and of mg_gmres (small grids).

    advection_1d(p, T)                          dense G[i, j] = int phi_j' phi_i, own Gauss loop
    poisson_operator(p, knots, c, robin, beta)  -Lap u + beta . grad u + c u with the Robin faces of
                                                tests/robin_oracle.py: sum_a (K_a + R_a + beta_a G_a) (x) M_others
                                                + c (x)M_a
    mg_gmres(h, A, b, ...)                      oracle.poms_oracle.gmres on A, right-preconditioned by one
                                                V-cycle of the symmetric oracle hierarchy h

With beta = None the operator is robin_oracle.poisson_operator's, bit for bit."""
import numpy as np

import robin_oracle as ro
from oracle import poms_oracle as po


def advection_1d(p, T):
    """Dense n x n advection matrix on knot vector T with the (p+1)-point Gauss rule per element (exact)."""
    T = np.asarray(T, float)
    n = len(T) - p - 1
    u, w = np.polynomial.legendre.leggauss(p + 1)
    G = np.zeros((n, n))
    for span in range(p, n):
        a, b = T[span], T[span + 1]
        if b <= a:
            continue
        x = 0.5 * (a + b) + 0.5 * (b - a) * u
        wq = 0.5 * (b - a) * w
        v, dv = po._basis_and_ders(T, p, span, x)
        i0 = span - p
        G[i0:i0 + p + 1, i0:i0 + p + 1] += (v * wq) @ dv.T
    return G


def poisson_operator(p, knots_per_axis, c=1.0, robin=None, beta=None):
    """(A, Mb, Kb): Kb[a] = K_a + R_a + beta_a G_a (the reaction term is not in Kb)."""
    if beta is None:
        return ro.poisson_operator(p, knots_per_axis, c, robin)
    _, Mb, Kb = ro.poisson_operator(p, knots_per_axis, c, robin)
    Kb = [k + b * po.dense_to_band(advection_1d(p, T), p) if b != 0.0 else k
          for k, b, T in zip(Kb, beta, knots_per_axis)]
    d = len(Kb)
    terms = [tuple((Kb[b] + c * Mb[b] if a == d - 1 else Kb[b]) if b == a else Mb[b] for b in range(d))
             for a in range(d)]
    return po.KronSumOperator(terms), Mb, Kb


def mg_gmres(h, A, b, tol=1e-10, maxiter=300, restart=30):
    """poms_b200.mg.mg_gmres restated: GMRES on A with psolve = one V-cycle of h from a zero guess."""
    return po.gmres(A, b, tol=tol, maxiter=maxiter, restart=restart, psolve=lambda A_, v: h.vcycle(0, v))
