"""The CUDA source of the particle-coupling kernels (poms_b200/csrc/poms_points.cu), compiled for the HOST over
tests/host_emu/cuda_emu.h and run under AddressSanitizer and ThreadSanitizer through the file's own C entry
points (host checks, template dispatch, the moments / assembly chunks along axis 1 and the dynamic shared
memory of each launch, exactly sized), checked against the NumPy oracle (tests/points_oracle.py): p = 1..5, 2-D
and 3-D, uniform, graded and C0 knots, a crowded cell beside empty ones, points on every breakpoint and on
both ends, several chunks.  The default run keeps a core set; POMS_EMU_FULL=1 runs every case under both
sanitizers."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
import points_oracle as po
from poms_b200 import bsplines as bs

EMU = os.path.join(ROOT, "tests", "host_emu")
FULL = os.environ.get("POMS_EMU_FULL") == "1"


@pytest.fixture(scope="module")
def points_exes(tmp_path_factory):
    """emu_points under {ASan, TSan}, built like the fixture of test_fem_host_emulation.py."""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("emu_points")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    procs = {}
    for name, flags in (("asan", ["-fsanitize=address", "-fno-omit-frame-pointer"]), ("tsan", ["-fsanitize=thread"])):
        out = str(d / ("emu_points_" + name))
        procs[name] = (out, subprocess.Popen(
            [gxx, "-std=c++17", "-O1", "-g"] + flags + ["-I" + EMU, "-I" + os.path.join(ROOT, "include"),
                                                         "-I" + cuda_inc, os.path.join(EMU, "emu_points.cpp"),
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


def _exe(exes, san):
    if san not in exes:
        pytest.skip("emu_points (%s) cannot start in this environment" % san)
    return exes[san]


def _call(exe, tmp, hdr, arrays, n_out):
    h = np.zeros(32, dtype=np.int32)
    h[:len(hdr)] = hdr
    fi, fo_ = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        h.tofile(f)
        for a in arrays:
            np.ascontiguousarray(a, dtype=np.float64).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo_], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo_, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:], dtype=np.float64)[:n_out].copy()


def _knots(p, N, kind):
    if kind == "c0":                    # one interior breakpoint of multiplicity p
        br = np.arange(1, N) / N
        inner = np.sort(np.concatenate([br, np.full(p - 1, br[len(br) // 2])]))
        return np.concatenate([np.zeros(p + 1), inner, np.ones(p + 1)])
    T = bs.make_open_knots(p, N + p)
    if kind == "graded":
        T[p + 1:N + p] = T[p + 1:N + p] ** 1.5
    return T


def _points(rng, knots, p, m_rand, crowd=0):
    """Random points, every breakpoint on every axis (others random), the corners, and `crowd` points in
    one cell."""
    d = len(knots)
    P = [rng.uniform(0.0, 1.0, (m_rand, d))]
    for a, T in enumerate(knots):
        br = np.unique(T)
        q = rng.uniform(0.0, 1.0, (len(br), d))
        q[:, a] = br
        P.append(q)
    P.append(np.array(np.meshgrid(*[[0.0, 1.0]] * d, indexing="ij")).reshape(d, -1).T)
    if crowd:
        lo = [np.unique(T)[1] for T in knots]
        hi = [np.unique(T)[2] for T in knots]
        P.append(rng.uniform(lo, hi, (crowd, d)))
    return np.concatenate(P)


def _dims(knots, p):
    n = [len(T) - p - 1 for T in knots]
    return (n[0], n[1], n[2]) if len(n) == 3 else (n[0], 1, n[1])


def run_eval(exe, tmp, p, knots, x, pts, grad):
    n1, n2, n3 = _dims(knots, p)
    d, m = len(knots), len(pts)
    ld = n3 + 3
    xp = np.zeros((n1, n2, ld))
    xp[:, :, :n3] = x.reshape(n1, n2, n3)
    out = _call(exe, tmp, [0, n1, n2, n3, p, d, m, int(grad), ld], list(knots) + [xp, pts],
                m * (1 + (d if grad else 0)))
    return out[:m], (out[m:].reshape(m, d) if grad else None)


def run_deposit(exe, tmp, p, knots, pts, w, chunk):
    n1, n2, n3 = _dims(knots, p)
    d, m = len(knots), len(pts)
    ld = n3 + 1
    y = np.zeros((n1, n2, ld))
    y[:, :, :n3] = np.nan                         # every owned entry must be overwritten
    out = _call(exe, tmp, [1, n1, n2, n3, p, d, m, chunk, ld], list(knots) + [pts, w, y], n1 * n2 * ld)
    out = out.reshape(n1, n2, ld)
    assert not out[:, :, n3:].any()               # the pad column stays zero
    return out[:, :, :n3].reshape([n1] + ([n2] if d == 3 else []) + [n3])


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# (p, elements per axis, knot family, cell planes per chunk, points in the crowded cell)
CASES = [(3, (4, 3, 5), "uniform", 2, 600), (1, (5, 4, 3), "graded", 1, 0), (2, (4, 5, 3), "c0", 3, 0),
         (4, (3, 4, 4), "graded", 100, 300), (5, (3, 3, 4), "c0", 1, 0), (2, (7, 6), "c0", 2, 0),
         (5, (5, 6), "graded", 3, 0), (4, (6, 5), "uniform", 1, 2000), (1, (6, 9), "c0", 4, 0)]


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,Ns,kind,chunk,crowd", CASES)
def test_points_kernels_emulated(points_exes, tmp_path, san, p, Ns, kind, chunk, crowd):
    core = {"asan": [(3, (4, 3, 5)), (2, (4, 5, 3)), (2, (7, 6))], "tsan": [(4, (6, 5))]}
    if not FULL and (p, Ns) not in core[san]:
        pytest.skip("not in the core set (POMS_EMU_FULL=1 runs every case under both sanitizers)")
    exe = _exe(points_exes, san)
    knots = [_knots(p, N, kind) for N in Ns]
    rng = np.random.default_rng(p + 10 * len(Ns))
    pts = _points(rng, knots, p, 150, crowd)
    npts = tuple(len(T) - p - 1 for T in knots)
    x = rng.standard_normal(npts)
    u, g = run_eval(exe, tmp_path, p, knots, x, pts, True)
    uo, go = po.evaluate_points(knots, p, x, pts)
    assert rel(u, uo) < 1e-13 and rel(g, go) < 1e-12
    u0, _ = run_eval(exe, tmp_path, p, knots, x, pts, False)
    assert np.array_equal(u0, u)
    w = rng.standard_normal(len(pts))
    b = run_deposit(exe, tmp_path, p, knots, pts, w, chunk)
    assert rel(b, po.deposit(knots, p, pts, w)) < 1e-13


@pytest.mark.parametrize("san", ["asan"])
def test_points_edge_sizes_emulated(points_exes, tmp_path, san):
    """m = 0 (zeros, no launch) and m = 1; a chunk of one plane on a 2-D space."""
    exe = _exe(points_exes, san)
    p = 2
    knots = [_knots(p, 4, "uniform"), _knots(p, 3, "graded")]
    for pts in (np.zeros((0, 2)), np.array([[1.0, 0.0]])):
        w = np.full(len(pts), 1.5)
        b = run_deposit(exe, tmp_path, p, knots, pts, w, 1)
        assert rel(b, po.deposit(knots, p, pts, w)) < 1e-13 if len(pts) else not b.any()
