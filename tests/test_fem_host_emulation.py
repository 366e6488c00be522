"""The CUDA source of the finite-element quadrature kernels (poms_b200/csrc/poms_fem3d.cu), compiled for the
HOST over tests/host_emu/cuda_emu.h and run under AddressSanitizer and ThreadSanitizer through the file's own C
entry points (host checks, template dispatch, chunking along axis 1 and the dynamic shared memory of each
launch, exactly sized, included), with the tables poms_b200.fem builds.  Checked against the NumPy oracle
(oracle/fem_oracle.py) on p = 1..5, ragged tiles, graded knots, 2-D and 3-D.  The default run keeps a core set;
POMS_EMU_FULL=1 runs every case under both sanitizers."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import fem_oracle as fo
from poms_b200 import bsplines as bs
from poms_b200.fem import _Axis

EMU = os.path.join(ROOT, "tests", "host_emu")
FULL = os.environ.get("POMS_EMU_FULL") == "1"


@pytest.fixture(scope="module")
def fem_exes(tmp_path_factory):
    """emu_fem under {ASan, TSan}, built like the emu_builds fixture of test_kernel_host_emulation.py."""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("emu_fem")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    procs = {}
    for name, flags in (("asan", ["-fsanitize=address", "-fno-omit-frame-pointer"]), ("tsan", ["-fsanitize=thread"])):
        out = str(d / ("emu_fem_" + name))
        procs[name] = (out, subprocess.Popen(
            [gxx, "-std=c++17", "-O0", "-g"] + flags + ["-I" + EMU, "-I" + os.path.join(ROOT, "include"),
                                                         "-I" + cuda_inc, os.path.join(EMU, "emu_fem.cpp"), "-o", out,
                                                         "-lpthread"],
            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    res = {}
    for name, (out, pr) in procs.items():
        log = pr.communicate()[0]
        assert pr.returncode == 0, log[-3000:]
        probe = subprocess.run([out], capture_output=True, text=True)
        if probe.returncode == 2 and "FATAL" not in probe.stderr:
            res[name] = out
    return res


def _exe(fem_exes, san):
    if san not in fem_exes:
        pytest.skip("emu_fem (%s) cannot start in this environment" % san)
    return fem_exes[san]


def _core(san, core_asan, core_tsan=False):
    if FULL:
        return
    if (san == "asan" and not core_asan) or (san == "tsan" and not core_tsan):
        pytest.skip("not in the core set (POMS_EMU_FULL=1 runs every case under both sanitizers)")


def _call(exe, tmp, hdr, arrays, n_out):
    h = np.zeros(32, dtype=np.int32)
    h[:len(hdr)] = hdr
    fi, fo_ = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        h.tofile(f)
        for a in arrays:
            np.ascontiguousarray(a).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo_], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo_, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:], dtype=np.float64)[:n_out].copy()


def _knots(p, N, graded):
    T = bs.make_open_knots(p, N + p)
    if graded:
        inner = T[p + 1:N + p]
        T[p + 1:N + p] = inner ** 1.5            # graded towards 0, simple knots
    return T


def _case_knots(p, Ns, graded):
    """One knot vector per axis: graded ones on every axis of a 2-D case, on axes 1 and 3 of a 3-D case."""
    return [_knots(p, N, graded and (len(Ns) == 2 or a != 1)) for a, N in enumerate(Ns)]


def _axes(p, knots):
    """Kernel tables of the knot vectors (the oracle integrates on the same ones)."""
    ax = [_Axis(T, p, "cpu") for T in knots]
    if len(knots) == 2:
        ax = [ax[0], _Axis.singleton("cpu"), ax[1]]
    return ax


def _np(t):
    return t.cpu().numpy()


def run_load(exe, tmp, p, knots, chunk, f):
    ax = _axes(p, knots)
    a1, a2, a3 = ax
    n1, n2, n3 = a1.n, a2.n, a3.n
    m2, m3 = a2.E * a2.Q, a3.E * a3.Q
    ld = n3 + 5                                   # a row pitch wider than the pad of a StencilVector
    y = np.full((n1, n2, ld), 0.0)
    x1, x2, x3 = a1.x.reshape(-1), a2.x.reshape(-1), a3.x.reshape(-1)
    for E0 in range(0, a1.E, chunk):
        E1 = min(a1.E, E0 + chunk)
        nq1 = (E1 - E0) * a1.Q
        fld, fpld = m3 + 3, (m2 + 1) * (m3 + 3)    # pitched chunk values
        F = np.zeros((nq1, fpld))
        vals = np.broadcast_to(f(x1[E0 * a1.Q:E1 * a1.Q, None, None], x2[None, :, None], x3[None, None, :]),
                               (nq1, m2, m3))
        Fv = F[:, :m2 * fld].reshape(nq1, m2, fld)
        Fv[:, :, :m3] = vals
        store_from = 0 if E0 == 0 else int(a1.first[E0 - 1]) + a1.K
        hdr = [0, n1, n2, n3, m2, m3, p, E0, E1, a1.K, a1.Q, store_from, a2.K * a2.Q, a3.E, nq1, a1.E, fld, fpld, ld]
        arrays = [a1.first, _np(a1.b_elem), a2.row_q0, _np(a2.row_coef), a3.row_e0, _np(a3.row_coef), F, y]
        y = _call(exe, tmp, hdr, arrays, n1 * n2 * ld).reshape(n1, n2, ld)
    assert not y[:, :, n3:].any()                 # the pad columns stay zero
    return y[:, :, :n3].reshape([n1] + ([n2] if len(knots) == 3 else []) + [n3])


def run_err(exe, tmp, p, knots, chunk, x, u, grad):
    ax = _axes(p, knots)
    a1, a2, a3 = ax
    n1, n2, n3 = a1.n, a2.n, a3.n
    m1, m2, m3 = a1.E * a1.Q, a2.E * a2.Q, a3.E * a3.Q
    ld = n3 + 1
    xp = np.zeros((n1, n2, ld))
    xp[:, :, :n3] = x.reshape(n1, n2, n3)
    c = [a.x.reshape(-1) for a in ax]
    out = np.zeros(2)
    for E0 in range(0, a1.E, chunk):
        E1 = min(a1.E, E0 + chunk)
        j0, j1 = E0 * a1.Q, E1 * a1.Q
        nq1 = j1 - j0
        X = (c[0][j0:j1, None, None], c[1][None, :, None], c[2][None, None, :])
        refs = [u(*X)] + (list(grad(*X)) if grad else [])
        if len(knots) == 2 and grad:
            refs = [refs[0], refs[1], None, refs[2]]
        refs += [None] * (4 - len(refs))
        has, rld, rpld, arrs = [], [], [], []
        for r in refs:
            has.append(int(r is not None))
            rld.append(m3 + 2)
            rpld.append(m2 * (m3 + 2) + 1)
            if r is not None:
                buf = np.zeros((nq1, m2 * (m3 + 2) + 1))
                buf[:, :m2 * (m3 + 2)].reshape(nq1, m2, m3 + 2)[:, :, :m3] = np.broadcast_to(r, (nq1, m2, m3))
                arrs.append(buf)
        hdr = [1, n1, n2, n3, m2, m3, p, j0, nq1, a1.K, a2.K, m1, int(grad is not None), ld] + has + rld + rpld
        arrays = [xp]
        for a in ax:
            arrays += [a.pt_s, _np(a.pt_v), _np(a.pt_d), _np(a.pt_w)]
        out = _call(exe, tmp, hdr, arrays + arrs + [out], 2)
    return np.sqrt(out)


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _f3(x, y, z):
    return np.cos(2.0 * x) * (1.0 + y * y) + z * np.sin(3.0 * y) + 0.5


CASES = [(3, (9, 13, 70), False, 3), (1, (5, 40, 7), True, 1), (2, (6, 9, 35), False, 2), (4, (5, 6, 34), True, 2),
         (5, (4, 5, 33), False, 1), (3, (7, 70), True, 3), (5, (5, 40), False, 100)]


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,Ns,graded,chunk", CASES)
def test_fem_kernels_emulated(fem_exes, tmp_path, san, p, Ns, graded, chunk):
    _core(san, (p, Ns) == (3, (9, 13, 70)), (p, Ns) == (2, (6, 9, 35)))
    exe = _exe(fem_exes, san)
    knots = _case_knots(p, Ns, graded)
    f = _f3 if len(Ns) == 3 else (lambda x, y: np.cos(2.0 * x) * (1.0 + y * y) + 0.5)
    b = run_load(exe, tmp_path, p, knots, chunk, lambda x, y, z: f(x, y, z) if len(Ns) == 3 else f(x[:, :, 0], z[0])[:, None, :])
    bo = fo.load_vector(knots, p, f)
    assert rel(b.reshape(bo.shape), bo) < 1e-13
    rng = np.random.default_rng(3)
    npts = tuple(len(T) - p - 1 for T in knots)
    x = rng.standard_normal(npts)
    if len(Ns) == 3:
        u = lambda X, Y, Z: np.sin(X) * np.cos(Y) + Z
        g = lambda X, Y, Z: (np.cos(X) * np.cos(Y), -np.sin(X) * np.sin(Y), 1.0 + 0 * Z)
        uo, go = u, g
    else:
        u = lambda X, Y, Z: np.sin(X) * np.cos(Z)
        g = lambda X, Y, Z: (np.cos(X) * np.cos(Z), -np.sin(X) * np.sin(Z))
        uo = lambda X, Z: np.sin(X) * np.cos(Z)
        go = lambda X, Z: (np.cos(X) * np.cos(Z), -np.sin(X) * np.sin(Z))
    l2, h1 = run_err(exe, tmp_path, p, knots, chunk, x, u, g)
    ref = fo.error_norms(knots, p, x, uo, go)
    assert abs(l2 - ref["l2"]) < 1e-13 * ref["l2"] and abs(h1 - ref["h1"]) < 1e-13 * ref["h1"], (l2, h1, ref)
