"""NumPy oracle of the reaction coefficient and the Robin / Neumann boundary terms (small grids).

    poisson_operator(p, knots, c, robin)   -Lap u + c u with alpha int_F u v ds on the faces, as the
                                           Kronecker sum sum_a (K_a + R_a) (x) M_others + c (x)M_a
    MGHierarchy(p, N, ..., c, robin)       oracle.poms_oracle.MGHierarchy on that operator, and with the
                                           'jacobi' smoother of poms_b200.mg (Chebyshev on D^-1 A)
    boundary_load(knots, p, g, axis, side) b_i = int_F g phi_i ds, dense

The defaults (c = 1, no Robin term) are oracle.poms_oracle's operator and hierarchy, bit for bit.  Every
1-D band is assembled by oracle.poms_oracle.assemble_1d; the face terms are R_a = alpha_lo e_0 e_0^T +
alpha_hi e_{n-1} e_{n-1}^T, because on an open knot vector phi_0 (phi_{n-1}) is the only basis function
that is non-zero on the face, with value 1."""
from math import sqrt

import numpy as np
from scipy.linalg import eigh

from oracle import fem_oracle as fo
from oracle import poms_oracle as po


def poisson_operator(p, knots_per_axis, c=1.0, robin=None):
    """(A, Mb, Kb): Kb[a] = K_a + R_a (the reaction term is not in Kb)."""
    MK = [po.assemble_1d(p, T) for T in knots_per_axis]
    Mb = [po.dense_to_band(M, p) for M, K in MK]
    Kb = [po.dense_to_band(K, p) for M, K in MK]
    if robin is not None:
        for a, (lo, hi) in enumerate(robin):
            Kb[a][0, p] += lo
            Kb[a][-1, p] += hi
    d = len(MK)
    terms = []
    for a in range(d):
        terms.append(tuple((Kb[b] + c * Mb[b] if a == d - 1 else Kb[b]) if b == a else Mb[b]
                           for b in range(d)))
    return po.KronSumOperator(terms), Mb, Kb


class MGHierarchy(po.MGHierarchy):
    """The oracle hierarchy with the operator above on every level: the glt / glt_poly lambda_max bound
    reads mu(K_a + R_a + c M_a), and the exact coarse solve divides by c + sum_a l_a with l_a the
    generalised eigenvalues of (K_a + R_a, M_a).  smoother='jacobi' restates poms_b200.mg: lambda_max of
    D^-1 A by 30 power steps from the same seeded start vector, Chebyshev on D^-1 A."""

    def __init__(self, p, N, Nc=8, smoother="glt", nu=1, ratio=4.0, safety=1.1, c=1.0, robin=None):
        self.p, self.smoother, self.nu, self.ratio = p, smoother, nu, ratio
        self.c, self.robin = c, robin
        N = list(N)
        d = len(N)
        self.levels = []
        while True:
            knots = [po.make_open_knots(p, n + p) for n in N]
            A, Mb, Kb = poisson_operator(p, knots, c, robin)
            self.levels.append(dict(N=list(N), knots=knots, A=A, Mb=Mb, Kb=Kb))
            if all(n <= Nc for n in N):
                break
            nxt = [n // 2 if (n > Nc and n % 2 == 0) else n for n in N]
            if nxt == N:
                break
            N = nxt
        for f, cl in zip(self.levels[:-1], self.levels[1:]):
            P1s = []
            for a in range(d):
                nf, nc = f["N"][a] + p, cl["N"][a] + p
                if nf == nc:
                    P1s.append(np.eye(nf))
                    continue
                ts = po.knots_to_insert(f["knots"][a], nf, p, cl["knots"][a], nc, p)
                P1s.append(po.insertion_matrix(ts, nc, p, cl["knots"][a]))
            f["P1s"] = P1s
        cl = self.levels[-1]
        if int(np.prod(cl["A"].npts)) <= self.DENSE_COARSE_MAX:
            self.Ainv_c = np.linalg.inv(cl["A"].tocsr().toarray())
            self._fd = None
        else:
            self.Ainv_c = None
            Qs, D = [], c
            for a, (Mb_, Kb_) in enumerate(zip(cl["Mb"], cl["Kb"])):
                Md, Kd = po.band_to_dense(Mb_), po.band_to_dense(Kb_)
                w, Q = eigh(0.5 * (Kd + Kd.T), 0.5 * (Md + Md.T))
                Qs.append(Q)
                shp = [1] * d
                shp[a] = len(w)
                D = D + w.reshape(shp)
            self._fd = (Qs, D)
        for lv in self.levels[:-1]:
            A = lv["A"]
            if smoother == "jacobi":
                lv["D"] = A.diagonal()
                lv["lmax"] = safety * self._power_lmax_jacobi(lv)
            else:
                q = max(2 * p - 1, 1)
                bands = [po.glt_band(p, n, degree=q) for n in A.npts]
                if smoother == "glt":
                    lv["glt"] = [po.band_factor(b) for b in bands]
                elif smoother == "glt_poly":
                    lv["gband"] = bands
                    lv["qc"] = []
                    for b_ in bands:
                        lo, hi = po._symbol_range(b_)
                        lv["qc"].append(po._cheb_inverse_poly(lo * 0.98, hi * 1.02, 3))
                else:
                    raise NotImplementedError(smoother)
                lv["lmax"] = safety * self.glt_lmax(lv, bands)
            lv["lmin"] = lv["lmax"] / ratio

    def glt_lmax(self, lv, bands):
        """max_a mu(K_a + R_a + c M_a) prod_{b != a} mu(M_b), generalised eigenvalues wrt the GLT bands."""
        d = len(bands)
        muM = [eigh(po.band_to_dense(lv["Mb"][a]), po.band_to_dense(bands[a]), eigvals_only=True)[-1]
               for a in range(d)]
        best = 0.0
        for a in range(d):
            KM = po.band_to_dense(lv["Kb"][a]) + self.c * po.band_to_dense(lv["Mb"][a])
            muK = eigh(KM, po.band_to_dense(bands[a]), eigvals_only=True)[-1]
            best = max(best, muK * float(np.prod([muM[b] for b in range(d) if b != a])))
        return best

    @staticmethod
    def _power_lmax_jacobi(lv, iters=30):
        import torch
        g = torch.Generator(device="cpu").manual_seed(1234)
        v = torch.rand(lv["A"].npts, generator=g, dtype=torch.float64).numpy() + 0.5
        lam = 1.0
        for _ in range(iters):
            w = lv["A"].dot(v) / lv["D"]
            nw = sqrt(float(np.vdot(w, w)))
            lam = nw / sqrt(float(np.vdot(v, v)))
            v = w * (1.0 / nw)
        return lam

    def smooth(self, lv, b, x, zero_guess):
        if self.smoother != "jacobi":
            return super().smooth(lv, b, x, zero_guess)
        A = lv["A"]
        theta = 0.5 * (lv["lmax"] + lv["lmin"])
        delta = 0.5 * (lv["lmax"] - lv["lmin"])
        sigma = theta / delta
        rho = 1.0 / sigma
        d = np.zeros_like(b)
        for k in range(self.nu):
            r = b if (k == 0 and zero_guess) else b - A.dot(x)
            z = r / lv["D"]
            if k == 0:
                c1, c2 = 0.0, 1.0 / theta
            else:
                rho_n = 1.0 / (2.0 * sigma - rho)
                c1, c2 = rho_n * rho, 2.0 * rho_n / delta
                rho = rho_n
            d = c1 * d + c2 * z
            x = x + d
        return x


def boundary_load(knots, p, g, axis, side):
    """b_i = sum_q w_q g(x_q) phi_i(x_q) over the Gauss points of the face axes; phi = 1 on the face for
    the first (side 0) or last (side 1) function along `axis`, 0 for every other one."""
    d = len(knots)
    face = [b for b in range(d) if b != axis]
    ax = [fo.axis_matrices(knots[b], p) for b in face]
    xs = np.meshgrid(*[a["x"] for a in ax], indexing="ij", sparse=True)
    G = np.broadcast_to(g(*xs), tuple(len(a["x"]) for a in ax)).astype(float)
    W = [a["B"] * a["w"][None, :] for a in ax]
    plane = W[0] @ G if d == 2 else W[0] @ G @ W[1].T
    npts = [len(T) - p - 1 for T in knots]
    out = np.zeros(npts)
    idx = [slice(None)] * d
    idx[axis] = 0 if side == 0 else npts[axis] - 1
    out[tuple(idx)] = plane
    return out
