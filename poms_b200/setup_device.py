"""Device-side 1-D setup of the hierarchy (SURVEY.md section 8f-2; csrc/poms_setup.cu).

`device_setup(True)` switches the setup routines of the package from the host NumPy/SciPy
implementations (bsplines.py, the default: they are what the golden-vector parity tests pin) to
hand-written CUDA kernels for the O(n p^2) parts
    assembly of the 1-D mass / stiffness bands   /root/reference/sources/matrix_assembler.py:10-77
    (and of the advection band of the convection term)
    knot-insertion rows of P1 (Oslo recursion)   /root/reference/sources/mg_jac.py:67
    banded LU of the GLT matrices (no pivoting)  /root/reference/sources/kron_product.py:191-197
and to torch.linalg on the device (cuSOLVER: library calls, setup only) for the dense generalised
eigenproblems (coarse eigenbases, /root/reference/sources/mg_jac.py:98-99; smoother bounds).
Only O(n p) results travel back to the host (band rows the launchers pass as kernel parameters).
"""
import contextlib

import numpy as np
import torch

from . import _lib
from . import bsplines as bs

_on = False
_device = None


def enabled():
    return _on


@contextlib.contextmanager
def device_setup(flag=True, device=None):
    global _on, _device
    old = (_on, _device)
    _on, _device = bool(flag), (torch.device(device) if device is not None else torch.device("cuda"))
    try:
        yield
    finally:
        _on, _device = old


def _stream():
    return torch.cuda.current_stream().cuda_stream


def assemble_1d_bands(p, T, toeplitz_interior=True):
    """Device twin of bsplines.assemble_1d_bands: returns host (M, K) band arrays (n, 2p+1)."""
    T = np.asarray(T, dtype=np.float64)
    n = len(T) - p - 1
    dev = _device
    Td = torch.as_tensor(T, device=dev)
    u, w = np.polynomial.legendre.leggauss(p + 1)
    ud, wd = torch.as_tensor(u, device=dev), torch.as_tensor(w, device=dev)
    M = torch.empty((n, 2 * p + 1), dtype=torch.float64, device=dev)
    K = torch.empty_like(M)
    _lib.check(_lib.lib().poms_assemble_1d(Td.data_ptr(), n, p, ud.data_ptr(), wd.data_ptr(), M.data_ptr(),
                                            K.data_ptr(), _stream()), "poms_assemble_1d")
    if toeplitz_interior and n > 4 * p + 1 and bs._is_uniform_open(T, p):
        mid = n // 2                       # same rule as the host routine: bit-identical interior rows
        M[2 * p:n - 2 * p] = M[mid].clone()
        K[2 * p:n - 2 * p] = K[mid].clone()
    return M.cpu().numpy(), K.cpu().numpy()


def assemble_1d_advection(p, T, toeplitz_interior=True):
    """Device twin of bsplines.assemble_1d_advection: returns the host band G (n, 2p+1)."""
    T = np.asarray(T, dtype=np.float64)
    n = len(T) - p - 1
    dev = _device
    Td = torch.as_tensor(T, device=dev)
    u, w = np.polynomial.legendre.leggauss(p + 1)
    ud, wd = torch.as_tensor(u, device=dev), torch.as_tensor(w, device=dev)
    G = torch.empty((n, 2 * p + 1), dtype=torch.float64, device=dev)
    _lib.check(_lib.lib().poms_assemble_1d_advection(Td.data_ptr(), n, p, ud.data_ptr(), wd.data_ptr(),
                                                      G.data_ptr(), _stream()), "poms_assemble_1d_advection")
    if toeplitz_interior and n > 4 * p + 1 and bs._is_uniform_open(T, p):
        G[2 * p:n - 2 * p] = G[n // 2].clone()
    return G.cpu().numpy()


def knot_insertion_rows(Tc, Tf, p):
    """Device twin of bsplines.knot_insertion_rows: (start int32, coef (n_f, p+1), n_c) on the host."""
    Tc = np.asarray(Tc, dtype=np.float64)
    Tf = np.asarray(Tf, dtype=np.float64)
    nc, nf = len(Tc) - p - 1, len(Tf) - p - 1
    dev = _device
    Tcd, Tfd = torch.as_tensor(Tc, device=dev), torch.as_tensor(Tf, device=dev)
    start = torch.empty(nf, dtype=torch.int32, device=dev)
    coef = torch.empty((nf, p + 1), dtype=torch.float64, device=dev)
    _lib.check(_lib.lib().poms_knot_insertion_rows(Tcd.data_ptr(), nc, Tfd.data_ptr(), nf, p, start.data_ptr(),
                                                    coef.data_ptr(), _stream()), "poms_knot_insertion_rows")
    return start.cpu().numpy(), coef.cpu().numpy(), nc


def band_lu(band):
    """Device twin of bsplines.band_lu for bands that need no pivoting: (lu_band, kl, ku, ipiv)."""
    band = np.ascontiguousarray(band, dtype=np.float64)
    n, w = band.shape
    q = (w - 1) // 2
    dev = _device
    bd = torch.as_tensor(band, device=dev)
    ab = torch.empty((3 * q + 1, n), dtype=torch.float64, device=dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().poms_band_lu_nopiv(bd.data_ptr(), n, q, ab.data_ptr(), info.data_ptr(), _stream()),
               "poms_band_lu_nopiv")
    if int(info.item()) != 0:
        raise np.linalg.LinAlgError("band LU without pivoting broke down at column %d" % int(info.item()))
    return ab.cpu().numpy(), q, q, np.arange(n, dtype=np.int32)


def gen_eigh(Kd, Md, device=None):
    """Generalised symmetric eigenproblem K q = l M q on the device (Cholesky reduction +
    torch.linalg.eigh): (eigenvalues ascending, M-orthonormal eigenvectors) as host arrays."""
    dev = device or _device
    K = torch.as_tensor(0.5 * (Kd + Kd.T), device=dev)
    M = torch.as_tensor(0.5 * (Md + Md.T), device=dev)
    Lc = torch.linalg.cholesky(M)
    C = torch.linalg.solve_triangular(Lc, K, upper=False)                      # L^-1 K
    C = torch.linalg.solve_triangular(Lc, C.T.contiguous(), upper=False).T     # L^-1 K L^-T
    w, Z = torch.linalg.eigh(0.5 * (C + C.T))
    Q = torch.linalg.solve_triangular(Lc.T.contiguous(), Z, upper=True)        # L^-T Z
    return w.cpu().numpy(), Q.cpu().numpy()


def gen_eig_max(Kb, Tb, iters=300):
    """Largest generalised eigenvalue of K x = mu T x (banded SPD): dense device eigh for n <= 1500
    (the host rule), power iteration on T^-1 K with dense-free torch band products above."""
    n = Kb.shape[0]
    if n <= 1500:
        w, _ = gen_eigh(bs.band_to_dense(Kb), bs.band_to_dense(Tb))
        return float(w[-1])
    dev = _device
    p = (Kb.shape[1] - 1) // 2
    q = (Tb.shape[1] - 1) // 2
    Kd = torch.as_tensor(np.ascontiguousarray(Kb), device=dev)
    lub, kl, ku, piv = band_lu(Tb)
    from .kron_product import BandLU
    lu = BandLU(lub, kl, ku, piv, dev)
    x = torch.as_tensor(np.cos(np.arange(n) * 0.7) + 1.5, device=dev)
    idx = (torch.arange(n, device=dev)[:, None] + torch.arange(-p, p + 1, device=dev)[None, :]).clamp_(0, n - 1)
    y = torch.empty_like(x)
    lam = 0.0
    L = _lib.lib()
    for _ in range(iters):
        kx = (Kd * x[idx]).sum(dim=1)                   # banded K x (out-of-matrix entries are zero)
        _lib.check(L.poms_band_solve_axis(kx.data_ptr(), y.data_ptr(), lu.ab.data_ptr(), None, n, kl, ku,
                                          1, n, 1, 1, _stream()), "poms_band_solve_axis")
        lam_t = torch.linalg.vector_norm(y) / torch.linalg.vector_norm(x)
        x = y / torch.linalg.vector_norm(y)
        y = torch.empty_like(x)
        lam = lam_t
    return float(lam.item())
