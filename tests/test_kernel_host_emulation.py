"""The CUDA source of the one-pass transfer kernels (poms_b200/csrc/poms_transfer3d_v2.cu and the round-1
kernels of poms_transfer3d.cuh), compiled for the HOST over tests/host_emu/cuda_emu.h (one OS thread per CUDA thread, pthread barrier =
__syncthreads, function-local statics = shared memory) and run under AddressSanitizer and
ThreadSanitizer through the file's own C entry points (host checks, chunking and template dispatch
included).  What this catches without a GPU: out-of-bounds global / shared accesses (every array is an
exactly sized heap block), missing or misplaced barriers (data races between the emulated threads),
and wrong results, on every row width p = 1..5, ragged tiles and the row tables of a slab plan
(starts relative to a rank's plane block, also negative).  TEST INFRASTRUCTURE: libpoms_b200.so never
contains this build (POMS_HOST_EMU is not defined by build.py), and timing it means nothing."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import poms_oracle as po
from poms_b200 import bsplines as bs

EMU = os.path.join(ROOT, "tests", "host_emu")
# Default run (the driver's CPU suite): a CORE set -- one or two cases per kernel family under the address
# sanitizer, the thread sanitizer on the two newest families (TMA mat-vec, one-pass transfers).
# POMS_EMU_FULL=1 runs every case under both sanitizers (profiles/r02_host_emulation_kernels.txt is such a
# run; it takes 3 to 10 minutes depending on the machine: 256 OS threads per emulated block).
FULL = os.environ.get("POMS_EMU_FULL") == "1"
TSAN_PROGS = ("emu_matvec3d_tma", "emu_matvec2d_tma", "emu_transfer")


def _core(san, core_asan, core_tsan=False):
    """Skip unless the case belongs to the core set (or the full run was requested)."""
    if FULL:
        return
    if (san == "asan" and not core_asan) or (san == "tsan" and not core_tsan):
        pytest.skip("not in the core set (POMS_EMU_FULL=1 runs every case under both sanitizers)")


@pytest.fixture(scope="module")
def emu_builds(tmp_path_factory):
    """The twelve executables ({TMA 3-D mat-vec, TMA 2-D mat-vec, transfer, band solve, generic 3-D mat-vec, 2-D mat-vec +
    vector algebra} x {ASan, TSan}), compiled in parallel; -O0: the runs are short and the harnesses have up to 150 template instantiations."""
    import sys
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    sys.path.insert(0, EMU)
    import make_emu_source
    d = tmp_path_factory.mktemp("emu")
    src, nlaunch = make_emu_source.band_solve_section()
    assert nlaunch == 5
    (d / "band_solve_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.generic_mv3_section()
    assert nlaunch == 5
    (d / "mv3_generic_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.tu0_middle_section()
    assert nlaunch == 18
    (d / "tu0_middle_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.tma_mv3_section((2, 3, 4))
    (d / "mv3_tma_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.tma_mv2_section()
    (d / "mv2_tma_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.axis_gather_section()
    assert nlaunch == 3
    (d / "axis_gather_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.dmma_section()
    assert nlaunch == 2
    (d / "dmma_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.setup_section()
    assert nlaunch == 3
    (d / "setup_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.stencil3d_section()
    assert nlaunch == 2
    (d / "stencil3d_emu.cuh").write_text(src)
    src, nlaunch = make_emu_source.halo_section()
    assert nlaunch == 1
    (d / "halo_emu.cuh").write_text(src)
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    procs = {}
    for prog in ("emu_matvec3d_tma", "emu_matvec2d_tma", "emu_transfer", "emu_bandsolve", "emu_matvec3d", "emu_tu0",
                 "emu_axis_gather", "emu_dmma", "emu_setup", "emu_stencil3d", "emu_halo"):
        if "_tma" in prog and not os.path.exists(os.path.join(cuda_inc, "cuda.h")):
            continue
        for name, flags in (("asan", ["-fsanitize=address", "-fno-omit-frame-pointer"]),
                            ("tsan", ["-fsanitize=thread"])):
            if name == "tsan" and ((not FULL and prog not in TSAN_PROGS) or prog in ("emu_axis_gather", "emu_halo")):
                continue                      # (the gather kernels have no barrier and no shared memory)
            out = str(d / (prog + "_" + name))
            procs[prog, name] = (out, subprocess.Popen(
                [gxx, "-std=c++17", "-O0", "-g"] + flags + ["-I" + EMU, "-I" + str(d), "-I" + os.path.join(ROOT, "include"),
                                                             "-I" + cuda_inc,
                                                             os.path.join(EMU, prog + ".cpp"), "-o", out, "-lpthread"],
                stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    res = {}
    for key, (out, pr) in procs.items():
        log = pr.communicate()[0]
        assert pr.returncode == 0, log[-3000:]
        # a sanitizer runtime that cannot start in this environment (e.g. ThreadSanitizer's "unexpected
        # memory mapping" under some ASLR settings) is an environment problem, not a kernel bug: skip
        probe = subprocess.run([out], capture_output=True, text=True)
        if probe.returncode == 2 and "FATAL" not in probe.stderr:
            res[key] = out
    return res


class _Exes:
    """exes[san] -> path of the executable, or skip when it was not built / cannot start here."""

    def __init__(self, builds, prog):
        self.builds, self.prog = builds, prog

    def __getitem__(self, san):
        exe = self.builds.get((self.prog, san))
        if exe is None:
            pytest.skip("%s (%s) is not available in this environment" % (self.prog, san))
        return exe


@pytest.fixture(scope="module")
def exes(emu_builds):
    return _Exes(emu_builds, "emu_transfer")


@pytest.fixture(scope="module")
def bs_exes(emu_builds):
    return _Exes(emu_builds, "emu_bandsolve")


@pytest.fixture(scope="module")
def mv_exes(emu_builds):
    return _Exes(emu_builds, "emu_matvec3d")


@pytest.fixture(scope="module")
def tma_exes(emu_builds):
    if ("emu_matvec3d_tma", "asan") not in emu_builds:
        pytest.skip("no <cuda.h> (the emulation uses the real CUtensorMap type)")
    return _Exes(emu_builds, "emu_matvec3d_tma")


@pytest.fixture(scope="module")
def tma2_exes(emu_builds):
    if ("emu_matvec2d_tma", "asan") not in emu_builds:
        pytest.skip("no <cuda.h> (the emulation uses the real CUtensorMap type)")
    return _Exes(emu_builds, "emu_matvec2d_tma")


@pytest.fixture(scope="module")
def tu0_exes(emu_builds):
    return _Exes(emu_builds, "emu_tu0")


def _pitch(n):
    return n + (n & 1)


def _run(exe, tmp, op, rows, src, dst, nf, nc):
    """op 0: dst(coarse) = R src(fine);  op 1: dst(fine) += P src(coarse)  (round-2 kernels; 2, 3: the
    round-1 kernels).  rows: [(start, coef)] * 3."""
    opx, op = op, op & 1
    ldf, ldc = _pitch(nf[2]), _pitch(nc[2])

    def pitched(a, ld):
        t = np.zeros(a.shape[:2] + (ld,))
        t[:, :, :a.shape[2]] = a
        return t

    hdr = np.array([opx, *nf, *nc, *[r[1].shape[1] for r in rows], 1, ldf, ldc, *[len(r[0]) for r in rows]],
                   dtype=np.int32)
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        for s, c in rows:
            np.ascontiguousarray(s, dtype=np.int32).tofile(f)
            np.ascontiguousarray(c, dtype=np.float64).tofile(f)
        pitched(src, ldf if op == 0 else ldc).tofile(f)
        pitched(dst, ldc if op == 0 else ldf).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    shp, ld = (nc, ldc) if op == 0 else (nf, ldf)
    out = np.frombuffer(raw[4:], dtype=np.float64).reshape(shp[0], shp[1], ld)
    assert not out[:, :, shp[2]:].any()            # the pad column stays zero
    return out[:, :, :shp[2]]


def _tables(p, N):
    Nc = [n // 2 for n in N]
    nf, nc = [n + p for n in N], [n + p for n in Nc]
    P, R, P1s = [], [], []
    for a in range(3):
        Tf, Tc = bs.make_open_knots(p, nf[a]), bs.make_open_knots(p, nc[a])
        st, cf, _ = bs.knot_insertion_rows(Tc, Tf, p)
        stt, cft = bs.rows_transpose(st, cf, nc[a])
        P.append((st, cf))
        R.append((stt, cft))
        ts = po.knots_to_insert(Tf, nf[a], p, Tc, nc[a], p)
        P1s.append(po.insertion_matrix(ts, nc[a], p, Tc))
    return nf, nc, P, R, P1s


def rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


CASES = [(3, (20, 36, 140)), (1, (8, 8, 16)), (2, (36, 18, 130)), (5, (12, 44, 72)), (4, (16, 20, 70)),
         (3, (130, 16, 16))]


GEN = {"round2": 0, "round1": 2}


@pytest.mark.parametrize("gen", ["round2", "round1"])
@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,N", CASES)
def test_transfer_kernels_emulated(exes, tmp_path, san, p, N, gen):
    _core(san, p == 3 and N == (20, 36, 140), p == 3 and N == (20, 36, 140) and gen == "round2")
    op0 = GEN[gen]
    nf, nc, P, R, P1s = _tables(p, N)
    rng = np.random.default_rng(1)
    rf, ec, xf = rng.standard_normal(nf), rng.standard_normal(nc), rng.standard_normal(nf)
    assert rel(_run(exes[san], tmp_path, op0, R, rf, np.zeros(nc), nf, nc), po.restrict(P1s, rf)) < 1e-14
    assert rel(_run(exes[san], tmp_path, op0 + 1, P, ec, xf, nf, nc), xf + po.prolong(P1s, ec)) < 1e-14


@pytest.mark.parametrize("gen", ["round2", "round1"])
@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,N,size", [(3, (48, 20, 70), 2), (2, (40, 36, 24), 3)])
def test_transfer_kernels_emulated_on_slab_plan_rows(exes, tmp_path, san, p, N, size, gen):
    """Rows of dist.slab_transfer_plan: starts relative to a rank's plane block; the prolongation rows
    of the inner ranks start BEFORE the block (leading zero coefficients).  The round-1 prolongation
    kernel read those planes out of bounds until this test ran it under AddressSanitizer."""
    from poms_b200.dist import slab_transfer_plan
    _core(san, size == 2)
    op0 = GEN[gen]
    nf, nc, P, R, P1s = _tables(p, N)
    rng = np.random.default_rng(5)
    rf, ec, xf = rng.standard_normal(nf), rng.standard_normal(nc), rng.standard_normal(nf)
    rc_ref, xf_ref = po.restrict(P1s, rf), xf + po.prolong(P1s, ec)
    plan = slab_transfer_plan(P[0][0], P[0][1], nc[0], size, True)
    assert min(pl[0].min() for pl in plan["P0"]) < 0        # the case the kernels clamp
    for q in range(size):
        (fs, fe), (cs, ce) = plan["tf"][q], plan["tc"][q]
        lo, hi = plan["need_f"][q]
        s0, c0, _ = plan["R0"][q]
        out = _run(exes[san], tmp_path, op0, [(s0, c0), R[1], R[2]], rf[lo:hi + 1],
                   np.zeros((ce - cs + 1, nc[1], nc[2])), (hi - lo + 1, nf[1], nf[2]), (ce - cs + 1, nc[1], nc[2]))
        assert rel(out, rc_ref[cs:ce + 1]) < 1e-14
        lo, hi = plan["need_c"][q]
        s0, c0, _ = plan["P0"][q]
        out = _run(exes[san], tmp_path, op0 + 1, [(s0, c0), P[1], P[2]], ec[lo:hi + 1], xf[fs:fe + 1],
                   (fe - fs + 1, nf[1], nf[2]), (hi - lo + 1, nc[1], nc[2]))
        assert rel(out, xf_ref[fs:fe + 1]) < 1e-14


# ------------------------------------------------------------------------------------------------
# banded line solves (section K4 of poms_kernels.cu): general dgbtrs with pivots, the no-pivot
# streaming kernels for a strided and for the contiguous axis (cp.async tiles, __syncwarp), the
# fused epilogue and the chunked substitution -- source rewritten for g++ by host_emu/make_emu_source.py
# ------------------------------------------------------------------------------------------------
def _band(rng, n, kl, ku, dominant):
    from scipy.linalg.lapack import dgbtrf
    A = np.zeros((n, n))
    for k in range(-kl, ku + 1):
        A += np.diag(rng.standard_normal(n - abs(k)), k)
    if dominant:
        A += np.diag(np.abs(A).sum(1) + 1.0)
    ab = np.zeros((2 * kl + ku + 1, n))
    for j in range(n):
        for i in range(max(0, j - ku), min(n, j + kl + 1)):
            ab[kl + ku + i - j, j] = A[i, j]
    lub, piv, info = dgbtrf(ab, kl, ku)
    assert info == 0
    return A, lub, piv


def _run_bs(exe, tmp, variant, lub, piv, kl, ku, y, chunk=0, warm=0, scale=1.0, add=None):
    n_outer, n, n_inner = y.shape
    hdr = np.array([variant, n, kl, ku, n_outer, n * n_inner, n_inner, n_inner, 0 if piv is None else 1, y.size,
                    chunk, warm, warm, 0 if add is None else 1, 0, 0], dtype=np.int32)
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        np.array([scale]).tofile(f)
        np.ascontiguousarray(lub, dtype=np.float64).tofile(f)
        if piv is not None:
            np.ascontiguousarray(piv, dtype=np.int32).tofile(f)
        np.ascontiguousarray(y).tofile(f)
        if add is not None:
            np.ascontiguousarray(add).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:], dtype=np.float64).reshape(y.shape)


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("n,kl,ku,dominant", [(37, 1, 1, True), (70, 3, 3, True), (33, 2, 3, False),
                                              (45, 3, 1, False), (40, 5, 5, True), (9, 1, 1, True)])
def test_band_solve_kernels_emulated(bs_exes, tmp_path, san, n, kl, ku, dominant):
    _core(san, (n, kl) in ((70, 3), (33, 2)))
    rng = np.random.default_rng(n)
    A, lub, piv = _band(rng, n, kl, ku, dominant)
    nopiv = np.array_equal(piv, np.arange(n))
    assert nopiv == dominant
    # (n_outer, n, n_inner): strided axis (one thread per line), contiguous axis (warp tiles), ragged
    for shape in [(3, n, 70), (1, n, 5), (130, n, 1), (7, n, 1)]:
        y = rng.standard_normal(shape)
        ref = np.stack([np.linalg.solve(A, y[o]) for o in range(shape[0])])
        x = _run_bs(bs_exes[san], tmp_path, 0, lub, None if nopiv else piv, kl, ku, y)
        assert rel(x, ref) < 1e-13
        if shape[2] == 1 and nopiv:
            add = rng.standard_normal(shape)
            x = _run_bs(bs_exes[san], tmp_path, 1, lub, None, kl, ku, y, scale=0.37, add=add)
            assert rel(x, add + 0.37 * ref) < 1e-13


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("n,kl,ku", [(150, 2, 2), (97, 3, 3)])
def test_band_chunk_kernels_emulated(bs_exes, tmp_path, san, n, kl, ku):
    """Chunked substitution against its host model (kron_product.BandLU._emulate_chunked: the same
    recurrences chunk by chunk, whatever the warm-up length)."""
    torch = pytest.importorskip("torch")
    from poms_b200.kron_product import BandLU
    _core(san, n == 97)
    rng = np.random.default_rng(n)
    A, lub, piv = _band(rng, n, kl, ku, True)
    lu = BandLU(lub, kl, ku, piv, torch.device("cpu"))
    for shape, chunk, warm in [((2, n, 3), 16, 12), ((1, n, 1), 24, 9), ((3, n, 70), 32, 20)]:
        y = rng.standard_normal(shape)
        x = _run_bs(bs_exes[san], tmp_path, 2, lub, None, kl, ku, y, chunk=chunk, warm=warm)
        ref = np.empty(shape)
        for o in range(shape[0]):
            for c in range(shape[2]):
                ref[o, :, c] = lu._emulate_chunked(y[o, :, c], chunk, warm)
        assert rel(x, ref) < 1e-14


# ------------------------------------------------------------------------------------------------
# generic 3-D Kronecker mat-vec (kron_matvec3d_kernel, translation unit 6: the fallback for tiny or
# misaligned grids -- every coarse level of a hierarchy runs it) with its five epilogues and the
# deterministic grid reduction of the fused dot (warp shuffles, ticket counter, last-CTA sum)
# ------------------------------------------------------------------------------------------------
def _consts():
    import re
    txt = open(os.path.join(ROOT, "include", "poms_b200.h")).read()
    get = lambda name: int(re.search(r"#define\s+%s\s+(\d+)" % name, txt).group(1))
    return ({k: get("POMS_EPI_" + k.upper()) for k in ("store", "resid", "jacobi", "dinv", "axpy")},
            {k: get("POMS_FORM_" + k.upper()) for k in ("single", "sum")})


def _run_mv(exe, tmp, p, form, epi, bands, x, b, omega, chunk, has_dot=True):
    n1, n2, n3 = x.shape
    ld = n3 + (n3 & 1)

    def pitched(a):
        t = np.zeros((n1, n2, ld))
        t[:, :, :n3] = a
        return t

    hdr = np.zeros(16, dtype=np.int32)
    hdr[:10] = [p, form, epi, n1, n2, n3, ld, chunk, 0 if b is None else 1, 1 if has_dot else 0]
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        np.array([omega]).tofile(f)
        for m_, k_ in bands:
            np.ascontiguousarray(m_, dtype=np.float64).tofile(f)
            np.ascontiguousarray(k_, dtype=np.float64).tofile(f)
        pitched(x).tofile(f)
        if b is not None:
            pitched(b).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    y = np.frombuffer(raw[12:], dtype=np.float64).reshape(n1, n2, ld)
    assert not y[:, :, n3:].any()
    return np.frombuffer(raw[4:12], dtype=np.float64)[0], y[:, :, :n3]


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,N,chunk", [(1, (5, 6, 7), 3), (2, (9, 20, 70), 4), (3, (12, 17, 66), 5),
                                       (4, (10, 18, 30), 20), (5, (8, 9, 10), 4)])
def test_generic_matvec3d_emulated(mv_exes, tmp_path, san, p, N, chunk):
    _core(san, p == 3)
    EPI, FORM = _consts()
    rng = np.random.default_rng(p)

    def randband(n):
        B = rng.standard_normal((n, 2 * p + 1))
        i, k = np.indices(B.shape)
        B[(i + k - p < 0) | (i + k - p >= n)] = 0.0
        B[:, p] += 4.0
        return B

    ms, ks = [randband(n) for n in N], [randband(n) for n in N]
    x, b = rng.standard_normal(N), rng.standard_normal(N)
    ab, d = po.apply_band, (lambda B: B[:, p])

    def A_sum(v):
        return (ab(ks[0], ab(ms[1], ab(ms[2], v, 2), 1), 0) + ab(ms[0], ab(ks[1], ab(ms[2], v, 2), 1), 0)
                + ab(ms[0], ab(ms[1], ab(ks[2], v, 2), 1), 0))

    D_sum = (np.einsum("i,j,k->ijk", d(ks[0]), d(ms[1]), d(ms[2])) + np.einsum("i,j,k->ijk", d(ms[0]), d(ks[1]), d(ms[2]))
             + np.einsum("i,j,k->ijk", d(ms[0]), d(ms[1]), d(ks[2])))
    cases = [("sum", A_sum, D_sum),
             ("single", lambda v: ab(ms[0], ab(ms[1], ab(ms[2], v, 2), 1), 0),
              np.einsum("i,j,k->ijk", d(ms[0]), d(ms[1]), d(ms[2])))]
    bands = list(zip(ms, ks))
    om = 0.7
    run = lambda form, epi, bb, omega, **kw: _run_mv(mv_exes[san], tmp_path, p, FORM[form], EPI[epi], bands, x, bb,
                                                     omega, chunk, **kw)
    for form, A, D in (cases if FULL else cases[:1]):
        yo = A(x)
        dr = om * (b - yo) / D
        dot, y = run(form, "store", None, 1.0)
        assert rel(y, yo) < 1e-14 and abs(dot - np.vdot(x, yo)) < 1e-13 * np.vdot(np.abs(x), np.abs(yo))
        dot, y = run(form, "resid", b, 1.0)
        assert rel(y, b - yo) < 1e-14 and abs(dot - np.vdot(b - yo, b - yo)) < 1e-13 * dot
        dot, y = run(form, "jacobi", b, om)
        assert rel(y, x + dr) < 1e-14 and abs(dot - np.vdot(dr, dr)) < 1e-13 * dot
        if san == "asan" and FULL:            # (the remaining epilogues share every barrier with the ones above)
            assert rel(run(form, "dinv", b, om, has_dot=False)[1], dr) < 1e-14
            dot, y = run(form, "axpy", b, om)
            assert rel(y, b + om * yo) < 1e-14 and abs(dot - np.vdot(om * yo, om * yo)) < 1e-13 * dot
            assert rel(run(form, "axpy", None, om)[1], om * yo) < 1e-14


# ------------------------------------------------------------------------------------------------
# round-1 2-D Kronecker mat-vec through poms_kron_matvec_2d (tiny / misaligned grids: C1; the TMA fast
# path is stubbed out), poms_jacobi_first_2d, and the vector algebra of the CG drivers
# ------------------------------------------------------------------------------------------------
def _call_tu0(exe, tmp, hdr_vals, scal, arrays, out_sizes):
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:len(hdr_vals)] = hdr_vals
    sc = np.zeros(4)
    sc[:len(scal)] = scal
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        sc.tofile(f)
        for a in arrays:
            np.ascontiguousarray(a, dtype=np.float64).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    outs, off = [], 12
    for n in out_sizes:
        outs.append(np.frombuffer(raw[off:off + 8 * n], dtype=np.float64))
        off += 8 * n
    return np.frombuffer(raw[4:12], dtype=np.float64)[0], outs


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,N", [(1, (16, 16)), (2, (10, 13)), (3, (64, 64)), (5, (40, 300)), (4, (9, 9)),
                                 (3, (7, 515)), (2, (120, 5))])
def test_matvec2d_round1_emulated(tu0_exes, tmp_path, san, p, N):
    _core(san, N == (64, 64))
    EPI, FORM = _consts()
    rng = np.random.default_rng(p + N[1])

    def randband(n):
        B = rng.standard_normal((n, 2 * p + 1))
        i, k = np.indices(B.shape)
        B[(i + k - p < 0) | (i + k - p >= n)] = 0.0
        B[:, p] += 4.0
        return B

    ms, ks = [randband(n) for n in N], [randband(n) for n in N]
    x, b = rng.standard_normal(N), rng.standard_normal(N)
    n1, n2 = N
    ld = n2 + (n2 & 1)
    pit = lambda a: np.pad(a, ((0, 0), (0, ld - n2)))

    def mv2(form, epi, bb, omega, has_dot=True, op=0):
        arrays = [ms[0], ks[0], ms[1], ks[1], pit(x)] + ([pit(bb)] if bb is not None else [])
        dot, (y,) = _call_tu0(tu0_exes[san], tmp_path, [op, n1, n2, ld, p, FORM[form], EPI[epi], 0 if bb is None else 1,
                                                         1 if has_dot else 0, 0], [omega], arrays, [n1 * ld])
        y = y.reshape(n1, ld)
        assert not y[:, n2:].any()
        return dot, y[:, :n2]

    ab, d = po.apply_band, (lambda B: B[:, p])
    om = 0.7
    for form, A, D in (("sum", lambda v: ab(ks[0], ab(ms[1], v, 1), 0) + ab(ms[0], ab(ks[1], v, 1), 0),
                        np.outer(d(ks[0]), d(ms[1])) + np.outer(d(ms[0]), d(ks[1]))),
                       ("single", lambda v: ab(ms[0], ab(ms[1], v, 1), 0), np.outer(d(ms[0]), d(ms[1])))):
        yo = A(x)
        dr = om * (b - yo) / D
        dot, y = mv2(form, "store", None, 1.0)
        assert rel(y, yo) < 1e-14 and abs(dot - np.vdot(x, yo)) < 1e-13 * np.vdot(np.abs(x), np.abs(yo))
        dot, y = mv2(form, "resid", b, 1.0)
        assert rel(y, b - yo) < 1e-14 and abs(dot - np.vdot(b - yo, b - yo)) < 1e-13 * dot
        dot, y = mv2(form, "jacobi", b, om)
        assert rel(y, x + dr) < 1e-14 and abs(dot - np.vdot(dr, dr)) < 1e-13 * dot
        if san == "asan":
            assert rel(mv2(form, "dinv", b, om, has_dot=False)[1], dr) < 1e-14
            assert rel(mv2(form, "axpy", b, om)[1], b + om * yo) < 1e-14
            dot, y = mv2(form, "store", b, om, op=5)               # poms_jacobi_first_2d
            assert rel(y, om * b / D) < 1e-14 and abs(dot - np.vdot(y, y)) < 1e-13 * dot


@pytest.mark.parametrize("san", ["asan", "tsan"])
def test_remaining_vector_kernels_emulated(tu0_exes, tmp_path, san):
    """poms_axpy_dev, poms_diag_scale (with and without the fused sum) and the 3-D form of poms_jacobi_first (several
    planes per block column: gridDim.z < n1), sum and single forms."""
    _core(san, False)
    exe = tu0_exes[san]
    _, FORM = _consts()
    rng = np.random.default_rng(8)
    for n in (1, 777, 5001):
        x, y, d = rng.standard_normal(n), rng.standard_normal(n), 1.0 + rng.random(n)
        z = np.zeros(n)
        _, (o,) = _call_tu0(exe, tmp_path, [8, 0, 0, 0, 0, 0, 0, 0, 0, n], [-1.0, 3.0, 7.0], [y, x, z, z], [n])
        assert rel(o, y - 3.0 / 7.0 * x) < 1e-15
        dot, (o,) = _call_tu0(exe, tmp_path, [9, 0, 0, 0, 0, 0, 0, 0, 1, n], [0.8], [z, x, d, z], [n])
        assert rel(o, 0.8 * x / d) < 1e-15 and abs(dot - np.sum((0.8 * x / d) ** 2)) <= 1e-13 * dot
        _, (o,) = _call_tu0(exe, tmp_path, [9, 0, 0, 0, 0, 0, 0, 0, 0, n], [0.8], [z, x, d, z], [n])
        assert rel(o, 0.8 * x / d) < 1e-15
    for p, N in [(2, (70, 5, 9)), (3, (9, 8, 300))]:
        n1, n2, n3 = N
        ld = n3 + (n3 & 1)
        bands = [rng.standard_normal((n, 2 * p + 1)) + 5.0 * (np.arange(2 * p + 1) == p) for n in N for _ in (0, 1)]
        m1, k1, m2, k2, m3, k3 = bands
        b = np.zeros((n1, n2, ld))
        b[..., :n3] = rng.standard_normal(N)
        M = [m[:, p] for m in (m1, m2, m3)]
        K = [k[:, p] for k in (k1, k2, k3)]
        o3 = lambda a, bb, c: a[:, None, None] * bb[None, :, None] * c[None, None, :]
        diag = {"single": o3(*M), "sum": o3(K[0], M[1], M[2]) + o3(M[0], K[1], M[2]) + o3(M[0], M[1], K[2])}
        for form in ("sum", "single"):
            dot, (o,) = _call_tu0(exe, tmp_path, [10, n1, n2, ld, p, FORM[form], 0, 1, 1, 0, n3], [0.7],
                                  bands + [b], [n1 * n2 * ld])
            o = o.reshape(n1, n2, ld)
            ref = 0.7 * b[..., :n3] / diag[form]
            assert rel(o[..., :n3], ref) < 1e-14 and abs(dot - np.sum(ref ** 2)) <= 1e-13 * dot and not o[..., n3:].any()


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("N,pads,glo,ghi", [((9, 13), (1, 1), 0, 0), ((12, 301), (3, 2), 0, 0), ((7, 40), (2, 3), 2, 1)])
def test_full_stencil2d_emulated(tu0_exes, tmp_path, san, N, pads, glo, ghi):
    """poms_stencil_matvec_2d = spl's StencilMatrix.dot (SURVEY 8a-3): unequal pads, a last extent that is odd and wider
    than one block, ghost rows on both sides (the slab form), the four epilogues with their fused reduction."""
    _core(san, N == (12, 301))
    EPI, _ = _consts()
    rng = np.random.default_rng(N[1])
    n1, n2 = N
    p1, p2 = pads
    ld = n2 + (n2 & 1)
    S = rng.standard_normal(N + (2 * p1 + 1, 2 * p2 + 1))
    S[..., p1, p2] += 20.0
    xg = np.zeros((glo + n1 + ghi, ld))
    xg[:, :n2] = rng.standard_normal((glo + n1 + ghi, n2))
    b = np.zeros((n1, ld))
    b[:, :n2] = rng.standard_normal(N)
    xpad = np.zeros((n1 + 2 * p1, n2 + 2 * p2))
    xpad[p1 - glo:p1 + n1 + ghi, p2:p2 + n2] = xg[:, :n2]
    Ax = np.zeros(N)
    for k1 in range(2 * p1 + 1):
        for k2 in range(2 * p2 + 1):
            Ax += S[..., k1, k2] * xpad[k1:k1 + n1, k2:k2 + n2]
    x, bb, dg, om = xg[glo:glo + n1, :n2], b[:, :n2], S[..., p1, p2], 0.6
    dr = om * (bb - Ax) / dg
    want = {"store": (Ax, np.sum(x * Ax)), "resid": (bb - Ax, np.sum((bb - Ax) ** 2)),
            "jacobi": (x + dr, np.sum(dr ** 2)), "dinv": (dr, np.sum(dr ** 2))}
    for name, (y_ref, dot_ref) in want.items():
        dot, (y,) = _call_tu0(tu0_exes[san], tmp_path, [7, n1, n2, ld, p1, p2, EPI[name], 1, 1, 0, glo, ghi], [om],
                              [S, xg, b], [n1 * ld])
        y = y.reshape(n1, ld)
        assert rel(y[:, :n2], y_ref) < 1e-14 and abs(dot - dot_ref) <= 1e-13 * abs(dot_ref)
        assert not y[:, n2:].any()
    _, (y,) = _call_tu0(tu0_exes[san], tmp_path, [7, n1, n2, ld, p1, p2, EPI["store"], 0, 0, 0, glo, ghi], [om],
                        [S, xg], [n1 * ld])
    assert rel(y.reshape(n1, ld)[:, :n2], Ax) < 1e-14


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("n", [1, 31, 1000, 100003])
def test_cg_vector_algebra_emulated(tu0_exes, tmp_path, san, n):
    """poms_cg_update, poms_p_update, poms_dot, poms_axpby, poms_cheb_update
    (/root/reference/sources/solvers.py:104-124) with the deterministic grid reduction."""
    _core(san, n == 1000)
    rng = np.random.default_rng(n)
    a = [rng.standard_normal(n) for _ in range(4)]
    num, den = 1.7, -0.9
    al = num / den
    exe = tu0_exes[san]
    dot, (x, r) = _call_tu0(exe, tmp_path, [1, 0, 0, 0, 0, 0, 0, 0, 1, n], [0, num, den, 0], a, [n, n])
    rr = a[1] - al * a[3]
    assert rel(x, a[0] + al * a[2]) < 1e-15 and rel(r, rr) < 1e-15 and abs(dot - np.vdot(rr, rr)) < 1e-13 * dot
    dot, (pp,) = _call_tu0(exe, tmp_path, [2, 0, 0, 0, 0, 0, 0, 0, 0, n], [0, num, den, 0], a, [n])
    assert rel(pp, a[1] + al * a[0]) < 1e-15
    dot, _ = _call_tu0(exe, tmp_path, [3, 0, 0, 0, 0, 0, 0, 0, 1, n], [], a, [])
    assert abs(dot - np.vdot(a[0], a[1])) < 1e-13 * np.vdot(np.abs(a[0]), np.abs(a[1]))
    dot, (z,) = _call_tu0(exe, tmp_path, [4, 0, 0, 0, 0, 0, 0, 0, 0, n], [0.3, -1.1], a, [n])
    assert rel(z, 0.3 * a[1] - 1.1 * a[2]) < 1e-15
    dot, (x, dd) = _call_tu0(exe, tmp_path, [6, 0, 0, 0, 0, 0, 0, 0, 0, n], [0.25, 0, 0, 1.5], a, [n, n])
    dn = 0.25 * a[1] + 1.5 * a[2]
    assert rel(dd, dn) < 1e-15 and rel(x, a[0] + dn) < 1e-15


# ------------------------------------------------------------------------------------------------
# THE HOT PATH: TMA-staged 3-D Kronecker mat-vec (kron_matvec3d_v3_kernel, and the round-1
# kron_matvec3d_tma_kernel kept as variant 0) through poms_kron_matvec_3d_dotv.  host_emu/emu_tma.h
# stands in for the tensor map, cp.async.bulk.tensor (immediate copy, zero fill outside the tensor) and
# the mbarrier (arrival / byte counts and phase under a mutex); tensor-map creation, Toeplitz tables,
# variant selection and chunking are the product's own host code.
# ------------------------------------------------------------------------------------------------
def _toeplitz_tables(ms, ks, p):
    """stencil.KronSumMatrix._toeplitz: interior rows bit-identical to the middle row, per axis."""
    W = 2 * p + 1
    coef, rng = np.zeros((3, 2, W)), np.zeros(6, dtype=np.int32)
    for a in range(3):
        m, k = ms[a], ks[a]
        n = m.shape[0]
        mid = n // 2
        same = np.all(m == m[mid], axis=1) & np.all(k == k[mid], axis=1)
        lo, hi = mid, mid + 1
        while lo > 0 and same[lo - 1]:
            lo -= 1
        while hi < n and same[hi]:
            hi += 1
        coef[a, 0], coef[a, 1] = m[mid], k[mid]
        rng[2 * a], rng[2 * a + 1] = lo, hi
    return coef, rng


def _run_tma(exe, tmp, p, form, epi, ms, ks, x, b, omega, variant, toep, has_dot=True, glo=0, ghi=0):
    """x holds glo + n1 + ghi planes (ghost planes of a slab sub-problem); the result has n1 planes."""
    n1, n2, n3 = x.shape
    n1 -= glo + ghi
    ld = n3 + (n3 & 1)
    pit = lambda a: np.pad(a, ((0, 0), (0, 0), (0, ld - n3)))
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:15] = [p, form, epi, n1, n2, n3, ld, variant, 0 if b is None else 1, 1 if has_dot else 0,
                0 if toep is None else 1, 0, 0, glo, ghi]
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        np.array([omega]).tofile(f)
        for a in range(3):
            np.ascontiguousarray(ms[a]).tofile(f)
            np.ascontiguousarray(ks[a]).tofile(f)
        if toep is not None:
            np.ascontiguousarray(toep[0]).tofile(f)
            np.ascontiguousarray(toep[1], dtype=np.int32).tofile(f)
        pit(x).tofile(f)
        if b is not None:
            pit(b).tofile(f)
    env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, env=env, timeout=1200)
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    dot, ntma = np.frombuffer(raw[8:24], dtype=np.float64)
    assert ntma > 0, "the TMA path was not taken"
    y = np.frombuffer(raw[24:], dtype=np.float64).reshape(n1, n2, ld)
    assert not y[:, :, n3:].any()
    return dot, y[:, :, :n3]


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,N,variant", [(3, (20, 20, 70), 1), (3, (20, 20, 70), 0), (3, (30, 50, 200), 1),
                                         (3, (12, 40, 140), 0), (2, (14, 30, 100), 1), (4, (12, 28, 90), 1)])
def test_tma_matvec3d_emulated(tma_exes, tmp_path, san, p, N, variant):
    """Operator of the bench (p = 3, Kronecker sum of the assembled mass / stiffness bands: Toeplitz
    interior rows from the constant bank, boundary rows from memory, ragged tiles; (30, 50, 200) also
    has interior tiles on the check-free fast path) and single Kronecker products of degree 2 and 4 (the
    shapes of the two smoother factors), every epilogue the V-cycle uses."""
    if san == "tsan" and N == (30, 50, 200):
        pytest.skip("largest case under the address sanitizer only")
    _core(san, variant == 1 and N in ((20, 20, 70), (14, 30, 100), (12, 28, 90)), N == (20, 20, 70) and variant == 1)
    EPI, FORM = _consts()
    nf = [n + p for n in N]
    MK = [bs.assemble_1d_bands(p, bs.make_open_knots(p, n)) for n in nf]
    ms, ks = [m for m, k in MK], [k for m, k in MK]
    ks[2] = ks[2] + ms[2]
    toep = _toeplitz_tables(ms, ks, p)
    assert all(toep[1][2 * a + 1] - toep[1][2 * a] >= nf[a] - 4 * p for a in range(3))
    rng = np.random.default_rng(p)
    x, b = rng.standard_normal(nf), rng.standard_normal(nf)
    ab, d = po.apply_band, (lambda B: B[:, p])
    A_sum = lambda v: (ab(ks[0], ab(ms[1], ab(ms[2], v, 2), 1), 0) + ab(ms[0], ab(ks[1], ab(ms[2], v, 2), 1), 0)
                       + ab(ms[0], ab(ms[1], ab(ks[2], v, 2), 1), 0))
    D_sum = (np.einsum("i,j,k->ijk", d(ks[0]), d(ms[1]), d(ms[2])) + np.einsum("i,j,k->ijk", d(ms[0]), d(ks[1]), d(ms[2]))
             + np.einsum("i,j,k->ijk", d(ms[0]), d(ms[1]), d(ks[2])))
    cases = [("single", lambda v: ab(ms[0], ab(ms[1], ab(ms[2], v, 2), 1), 0),
              np.einsum("i,j,k->ijk", d(ms[0]), d(ms[1]), d(ms[2])))]
    if p == 3:
        cases.insert(0, ("sum", A_sum, D_sum))
        if not FULL:
            cases = cases[:1]                 # core set: the bench operator; single products at p = 2, 4
    om = 0.7
    run = lambda form, epi, bb, omega, **kw: _run_tma(tma_exes[san], tmp_path, p, FORM[form], EPI[epi], ms, ks, x, bb,
                                                      omega, variant, toep, **kw)
    for form, A, D in cases:
        yo = A(x)
        dr = om * (b - yo) / D
        tol = 1e-14
        dot, y = run(form, "store", None, 1.0)
        assert rel(y, yo) < tol and abs(dot - np.vdot(x, yo)) < 1e-13 * np.vdot(np.abs(x), np.abs(yo))
        dot, y = run(form, "resid", b, 1.0)
        assert rel(y, b - yo) < tol and abs(dot - np.vdot(b - yo, b - yo)) < 1e-13 * dot
        if san == "tsan" or max(N) >= 200:
            continue                          # (the other epilogues share every barrier with these two)
        assert rel(run(form, "axpy", b, om)[1], b + om * yo) < tol
        if not FULL:
            continue
        assert rel(run(form, "axpy", None, om)[1], om * yo) < tol
        dot, y = run(form, "jacobi", b, om)
        assert rel(y, x + dr) < tol and abs(dot - np.vdot(dr, dr)) < 1e-13 * dot


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("case", ["graded23", "graded1", "synthetic"])
def test_tma_matvec3d_emulated_nonuniform(tma_exes, tmp_path, san, case):
    """The operator on inputs the uniform cases never produce (tests/test_gpu_nonuniform.py runs them on
    the GPU).  graded23: power-graded axes 2 and 3 leave one asymmetric Toeplitz row, so the host code
    sends a variant-1 request to the round-1 kernel (variant 0), whose whole-tile fix-up then runs on
    every other column and row.  graded1: a graded axis 1 keeps variant 1 but leaves it no steady plane
    range.  synthetic: uniform bands with Toeplitz ranges that start and end off the 2p margins and off
    the tile edges (the column-pair and plane-range arithmetic of both variants)."""
    import test_gpu_nonuniform as nu
    _core(san, True, case == "graded23")
    EPI, FORM = _consts()
    # graded23: N = 70 keeps the asymmetry of the graded rows (9e-3) within two decades of the threshold
    p, N = 3, {"graded23": (12, 70, 70), "graded1": (20, 20, 70), "synthetic": (20, 36, 140)}[case]
    kinds = {"graded23": ("u", "pow", "pow"), "graded1": ("pow", "u", "u"), "synthetic": ("u", "u", "u")}[case]
    knots = [nu.family_knots(k, p, n) for k, n in zip(kinds, N)]
    MK = [bs.assemble_1d_bands(p, T) for T in knots]
    ms, ks = [m for m, k in MK], [k for m, k in MK]
    ks[2] = ks[2] + ms[2]
    nf = [m.shape[0] for m in ms]
    coef, rg = _toeplitz_tables(ms, ks, p)
    for a in range(3):
        assert nu.range_ok(kinds[a], p, nf[a], *rg[2 * a:2 * a + 2])
    sym = all(np.all(np.abs(r - r[::-1]) <= 1e-13 * np.abs(r).max()) for a in (1, 2) for r in coef[a])
    assert sym == (case != "graded23")
    if case == "synthetic":
        # hi1 - lo1 >= 2p: planes whose window ends at row hi1 exist; lo3 even: at odd p the column pair
        # (lo3 - 1, lo3) straddles the range start
        rg = np.array([7, 16, 9, 30, 42, 101], dtype=np.int32)
        for a in range(3):
            ms[a], ks[a] = nu.perturb_outside([ms[a], ks[a]], rg[2 * a], rg[2 * a + 1], seed=a)
    rng = np.random.default_rng(5)
    x, b = rng.standard_normal(nf), rng.standard_normal(nf)
    ab = po.apply_band
    yo = (ab(ks[0], ab(ms[1], ab(ms[2], x, 2), 1), 0) + ab(ms[0], ab(ks[1], ab(ms[2], x, 2), 1), 0)
          + ab(ms[0], ab(ms[1], ab(ks[2], x, 2), 1), 0))
    ys = {}
    for variant in (1, 0):
        run = lambda epi, bb, om: _run_tma(tma_exes[san], tmp_path, p, FORM["sum"], EPI[epi], ms, ks, x, bb, om,
                                           variant, (coef, rg))
        dot, ys[variant] = run("store", None, 1.0)
        assert rel(ys[variant], yo) < 1e-14
        assert abs(dot - np.vdot(x, yo)) < 1e-13 * np.vdot(np.abs(x), np.abs(yo))
        assert rel(run("resid", b, 1.0)[1], b - yo) < 1e-14
        if san == "tsan":
            break
    if case == "graded23" and san == "asan":
        assert np.array_equal(ys[1], ys[0]), "a variant-1 request must run variant 0 on asymmetric rows"


# ------------------------------------------------------------------------------------------------
# the 2-D fast path (BASELINE configs C2 and C4): warp-autonomous TMA mat-vec (kron_matvec2d_tma_kernel,
# translation unit 7: private 4-stage ring of 2-D boxes per warp, no CTA barrier in the march) through
# poms_kron_matvec_2d_ex with the product's own tensor-map / Toeplitz / chunking host code
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p,N", [(3, (40, 150)), (5, (30, 300)), (2, (64, 64)), (3, (12, 515)), (1, (20, 70)),
                                 (4, (50, 129))])
def test_tma_matvec2d_emulated(tma2_exes, tmp_path, san, p, N):
    _core(san, p in (3, 5) and N[0] >= 30, (p, N) == (3, (40, 150)))
    EPI, FORM = _consts()
    nf = [n + p for n in N]
    MK = [bs.assemble_1d_bands(p, bs.make_open_knots(p, n)) for n in nf]
    ms, ks = [m for m, k in MK], [k for m, k in MK]
    ks[1] = ks[1] + ms[1]
    W = 2 * p + 1
    coef, rg = np.zeros((2, 2, W)), np.zeros(4, dtype=np.int32)
    for a in range(2):                       # stencil.KronSumMatrix._toeplitz
        m, k = ms[a], ks[a]
        mid = m.shape[0] // 2
        same = np.all(m == m[mid], axis=1) & np.all(k == k[mid], axis=1)
        lo, hi = mid, mid + 1
        while lo > 0 and same[lo - 1]:
            lo -= 1
        while hi < m.shape[0] and same[hi]:
            hi += 1
        coef[a, 0], coef[a, 1], rg[2 * a], rg[2 * a + 1] = m[mid], k[mid], lo, hi
    rng = np.random.default_rng(p)
    x, b = rng.standard_normal(nf), rng.standard_normal(nf)
    n1, n2 = nf
    ld = n2 + (n2 & 1)
    pit = lambda a: np.pad(a, ((0, 0), (0, ld - n2)))

    def run(form, epi, bb, omega, toep=True, has_dot=True):
        hdr = np.zeros(16, dtype=np.int32)
        hdr[:10] = [p, FORM[form], EPI[epi], n1, n2, ld, 1, 0 if bb is None else 1, 1 if has_dot else 0, 1 if toep else 0]
        fi, fo = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
        with open(fi, "wb") as f:
            hdr.tofile(f)
            np.array([omega]).tofile(f)
            for a in range(2):
                np.ascontiguousarray(ms[a]).tofile(f)
                np.ascontiguousarray(ks[a]).tofile(f)
            if toep:
                coef.tofile(f)
                rg.tofile(f)
            pit(x).tofile(f)
            if bb is not None:
                pit(bb).tofile(f)
        env = dict(os.environ, TSAN_OPTIONS="exitcode=66", ASAN_OPTIONS="detect_leaks=0")
        r = subprocess.run([tma2_exes[san], fi, fo], capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
        raw = open(fo, "rb").read()
        assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
        dot, ntma = np.frombuffer(raw[8:24], dtype=np.float64)
        assert ntma > 0, "the TMA path was not taken"
        y = np.frombuffer(raw[24:], dtype=np.float64).reshape(n1, ld)
        assert not y[:, n2:].any()
        return dot, y[:, :n2]

    ab, d = po.apply_band, (lambda B: B[:, p])
    om = 0.7
    for form, A, D in (("sum", lambda v: ab(ks[0], ab(ms[1], v, 1), 0) + ab(ms[0], ab(ks[1], v, 1), 0),
                        np.outer(d(ks[0]), d(ms[1])) + np.outer(d(ms[0]), d(ks[1]))),
                       ("single", lambda v: ab(ms[0], ab(ms[1], v, 1), 0), np.outer(d(ms[0]), d(ms[1])))):
        yo = A(x)
        dr = om * (b - yo) / D
        tol = 3e-14                           # (the sum form uses the mean of the two halves of a symmetric row)
        dot, y = run(form, "store", None, 1.0)
        assert rel(y, yo) < tol and abs(dot - np.vdot(x, yo)) < 1e-13 * np.vdot(np.abs(x), np.abs(yo))
        dot, y = run(form, "resid", b, 1.0)
        assert rel(y, b - yo) < tol and abs(dot - np.vdot(b - yo, b - yo)) < 1e-12 * dot
        if san == "tsan" and not FULL:
            continue
        dot, y = run(form, "jacobi", b, om)
        assert rel(y, x + dr) < tol and abs(dot - np.vdot(dr, dr)) < 1e-12 * dot
        assert rel(run(form, "dinv", b, om, has_dot=False)[1], dr) < tol
        assert rel(run(form, "axpy", b, om)[1], b + om * yo) < tol
        assert rel(run(form, "store", None, 1.0, toep=False)[1], yo) < tol      # no Toeplitz hints


# ------------------------------------------------------------------------------------------------
# poms_axis_gather (section K5): the per-axis sparse row gather behind the 2-D transfers, the fallback of
# the 3-D ones and the slab-plan rows (negative starts); address sanitizer only: no barrier, no shared memory
# ------------------------------------------------------------------------------------------------
def _gather(exe, tmp, start, coef, n_in, src, axis, acc=None):
    shape = list(src.shape)
    nd, n_out, W = len(shape), len(start), coef.shape[1]
    out_shape = list(shape)
    out_shape[axis] = n_out
    ld = shape[-1]
    if axis == nd - 1:
        ld_out = n_out + (n_out & 1)
        out_shape[-1] = ld_out
        geo = [int(np.prod(shape[:-1])), ld, 1, ld_out, 1, 1]
    elif axis == 0:
        rest = int(np.prod(shape[1:]))
        geo = [1, 0, rest, 0, rest, rest]
    else:
        geo = [shape[0], shape[1] * ld, ld, n_out * ld, ld, ld]
    out0 = np.zeros(out_shape) if acc is None else acc.copy()
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:5] = [W, n_in, n_out, 0 if acc is None else 1, n_out]
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        np.array(geo, dtype=np.int64).tofile(f)
        np.array([src.size, out0.size], dtype=np.int64).tofile(f)
        np.ascontiguousarray(start, dtype=np.int32).tofile(f)
        np.ascontiguousarray(coef).tofile(f)
        np.ascontiguousarray(src).tofile(f)
        np.ascontiguousarray(out0).tofile(f)
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:], dtype=np.float64).reshape(out_shape)


def _gather_ref(start, coef, n_in, src, axis):
    n_out, W = coef.shape
    A = np.zeros((n_out, n_in))
    for i in range(n_out):
        for w in range(W):
            if 0 <= start[i] + w < n_in:
                A[i, start[i] + w] += coef[i, w]
    return np.moveaxis(np.tensordot(A, src, axes=(1, axis)), 0, axis)


@pytest.mark.parametrize("p,n", [(3, 16), (2, 40), (5, 130)])
def test_axis_gather_emulated(emu_builds, tmp_path, p, n):
    from poms_b200.dist import slab_transfer_plan
    _core("asan", p == 3)
    exe = _Exes(emu_builds, "emu_axis_gather")["asan"]
    nf, nc = n + p, n // 2 + p
    st, cf, _ = bs.knot_insertion_rows(bs.make_open_knots(p, nc), bs.make_open_knots(p, nf), p)
    rng = np.random.default_rng(n)
    for rest in [(7,), (3, 130), (66,)]:
        for axis in range(len(rest) + 1):
            shp = list(rest)
            shp.insert(axis, nc)
            last = shp[-1]
            src = np.zeros(shp[:-1] + [last + (last & 1)])
            src[..., :last] = rng.standard_normal(shp)
            lastax = axis == len(shp) - 1
            cut = (lambda a: a[..., :nf]) if lastax else (lambda a: a)
            r = _gather_ref(st, cf, nc, src[..., :last] if lastax else src, axis)
            y = _gather(exe, tmp_path, st, cf, nc, src, axis)
            assert rel(cut(y), cut(r)) < 1e-14
            acc = rng.standard_normal(y.shape)
            if lastax:
                acc[..., nf:] = 0
            assert rel(cut(_gather(exe, tmp_path, st, cf, nc, src, axis, acc=acc) - acc), cut(r)) < 1e-13
    plan = slab_transfer_plan(st, cf, nc, 3, True)
    assert min(pl[0].min() for pl in plan["P0"]) < 0
    for q in range(3):
        s0, c0, n_in = plan["P0"][q]
        src = rng.standard_normal((n_in, 5, 66))
        assert rel(_gather(exe, tmp_path, s0, c0, n_in, src, 0), _gather_ref(s0, c0, n_in, src, 0)) < 1e-14


# ------------------------------------------------------------------------------------------------
# poms_axis_dense_dmma: the dense eigenbasis contraction of the coarse solve on the fp64 tensor cores.  The
# kernel source runs unchanged; only the one-instruction wrapper around mma.sync.m8n8k4.f64 is replaced by
# cuda_emu.h's lane-by-lane model of the PTX fragment layout (so a wrong fragment index in the kernel shows).
# ------------------------------------------------------------------------------------------------
def _dmma(exe, tmp, Q, src, axis):
    shape = list(src.shape)
    n_out, n_in = Q.shape
    assert shape[axis] == n_in and len(shape) == 3
    out_shape = list(shape)
    out_shape[axis] = n_out
    if axis == 2:
        geo = [shape[0] * shape[1], n_in, 1, n_out, 1, 1]
    elif axis == 0:
        rest = shape[1] * shape[2]
        geo = [1, 0, rest, 0, rest, rest]
    else:
        geo = [shape[0], n_in * shape[2], shape[2], n_out * shape[2], shape[2], shape[2]]
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:2] = [n_in, n_out]
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        np.array(geo, dtype=np.int64).tofile(f)
        np.array([src.size, int(np.prod(out_shape))], dtype=np.int64).tofile(f)
        np.ascontiguousarray(Q).tofile(f)
        np.ascontiguousarray(src).tofile(f)
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:], dtype=np.float64).reshape(out_shape)


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("shape,n_out", [((19, 70, 9), None), ((35, 33, 67), None), ((8, 5, 130), 11)])
def test_dense_dmma_contraction_emulated(emu_builds, tmp_path, san, shape, n_out):
    """Square (the eigenbasis Q and Q^T of the coarse solve) and rectangular Q along each of the three axes, extents
    that are not multiples of the 64 x 64 x 32 tile: exact against numpy to rounding, no out-of-bounds access,
    no race between the staging loops and the fragment loads."""
    _core(san, shape[0] == 19)
    exe = _Exes(emu_builds, "emu_dmma")[san]
    rng = np.random.default_rng(shape[1])
    src = rng.standard_normal(shape)
    for axis in range(3):
        m = n_out or shape[axis]
        Q = rng.standard_normal((m, shape[axis]))
        ref = np.moveaxis(np.tensordot(Q, src, axes=(1, axis)), 0, axis)
        assert rel(_dmma(exe, tmp_path, Q, src, axis), ref) < 1e-14


# ------------------------------------------------------------------------------------------------
# Device-side 1-D set-up (poms_setup.cu, SURVEY 8f-2): assembly by quadrature, knot-insertion rows by the Oslo
# recursion, banded LU without pivoting -- the same comparisons as tests/test_gpu_setup.py, on exactly sized buffers
# ------------------------------------------------------------------------------------------------
def _setup(exe, tmp, hdr_vals, arrays):
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:len(hdr_vals)] = hdr_vals
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        for a in arrays:
            a = np.ascontiguousarray(a, dtype=np.float64)
            np.array([a.size], dtype=np.int64).tofile(f)
            a.tofile(f)
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return raw[4:]


def _graded_knots(p, N, uniform):
    T = bs.make_open_knots(p, N + p)
    if not uniform:
        inner = np.linspace(0.0, 1.0, N + 1)[1:-1] ** 1.7
        T = np.concatenate([np.zeros(p + 1), inner, np.ones(p + 1)])
    return T


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_setup_kernels_emulated(emu_builds, tmp_path, san, p):
    _core(san, p == 3)
    exe = _Exes(emu_builds, "emu_setup")[san]
    # assembly: uniform and graded open knot vectors, n not a multiple of the block
    for N, uniform in [(8, True), (37, True), (23, False), (150, True)]:
        T = _graded_knots(p, N, uniform)
        n = N + p
        Mh, Kh = bs.assemble_1d_bands(p, T, toeplitz_interior=False)
        u, w = np.polynomial.legendre.leggauss(p + 1)
        raw = _setup(exe, tmp_path, [0, n, p], [T, u, w])
        MK = np.frombuffer(raw, dtype=np.float64).reshape(2, n, 2 * p + 1)
        assert np.abs(MK[0] - Mh).max() <= 1e-13 * np.abs(Mh).max()
        assert np.abs(MK[1] - Kh).max() <= 1e-13 * np.abs(Kh).max()
    # knot-insertion rows: dyadic and wider refinements, and a graded coarse vector refined by midpoints
    cases = [(bs.make_open_knots(p, Nc + p), bs.make_open_knots(p, Nc * ratio + p))
             for Nc, ratio in [(4, 2), (5, 4), (16, 8), (70, 2)]]
    Tg = _graded_knots(p, 11, False)
    br = np.unique(Tg)
    cases.append((Tg, np.concatenate([np.zeros(p), np.sort(np.concatenate([br, 0.5 * (br[1:] + br[:-1])])), np.ones(p)])))
    for Tc, Tf in cases:
        sh, ch, nc = bs.knot_insertion_rows(Tc, Tf, p)
        nf = len(Tf) - p - 1
        raw = _setup(exe, tmp_path, [1, 0, p, nc, nf], [Tc, Tf])
        sd = np.frombuffer(raw[:4 * nf], dtype=np.int32)
        cd = np.frombuffer(raw[4 * nf:], dtype=np.float64).reshape(nf, p + 1)
        assert np.array_equal(sd, sh)
        assert np.abs(cd - ch).max() <= 1e-15
        assert np.abs(cd.sum(axis=1) - 1.0).max() < 1e-14
    # banded LU without pivoting against LAPACK's dgbtrf (no interchanges on these bands)
    for n in (3 * p + 2, 67, 140):
        band = bs.glt_band(p, n, degree=max(2 * p - 1, 1))
        c = (band.shape[1] - 1) // 2
        q = c
        while q > 0 and not band[:, c - q].any():
            q -= 1
        band = band[:, c - q:c + q + 1]
        lh, kl, ku, piv = bs.band_lu(band)
        assert np.array_equal(piv, np.arange(n)) and kl == ku == q
        raw = _setup(exe, tmp_path, [2, n, p, 0, 0, q], [band])
        assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
        ab = np.frombuffer(raw[4:], dtype=np.float64).reshape(3 * q + 1, n)
        assert np.abs(ab - lh).max() <= 1e-13 * np.abs(lh).max()
    # a zero pivot is reported through info, not divided by
    band = np.zeros((9, 3))
    band[:, 1] = 1.0
    band[4, 1] = 0.0
    raw = _setup(exe, tmp_path, [2, 9, 1, 0, 0, 1], [band])
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 5


# ------------------------------------------------------------------------------------------------
# poms_stencil_matvec_3d (full, non-separable 3-D stencil = spl's StencilMatrix.dot in 3-D; one warp per point,
# shared offset table in dynamic shared memory, deterministic grid reduction) and poms_color_add
# ------------------------------------------------------------------------------------------------
def _stencil3d(exe, tmp, op, N, pads, ld, epi=0, has_dot=0, glo=0, ghi=0, omega=1.0, off=0, colour=0, arrays=(), has_b=0):
    hdr = np.zeros(16, dtype=np.int32)
    hdr[:15] = [op, N[0], N[1], N[2], pads[0], pads[1], pads[2], epi, has_dot, glo, ghi, ld, off, colour, has_b]
    fi, fo = str(tmp / "in.bin"), str(tmp / "out.bin")
    with open(fi, "wb") as f:
        hdr.tofile(f)
        np.array([omega]).tofile(f)
        for a in arrays:
            np.ascontiguousarray(a, dtype=np.float64).tofile(f)
    r = subprocess.run([exe, fi, fo], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0 and not r.stderr.strip(), (r.returncode, r.stderr[-4000:])
    raw = open(fo, "rb").read()
    assert np.frombuffer(raw[:4], dtype=np.int32)[0] == 0
    return np.frombuffer(raw[4:12], dtype=np.float64)[0], np.frombuffer(raw[12:], dtype=np.float64).reshape(N[0], N[1], ld)


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("N,pads,glo,ghi", [((6, 7, 9), (1, 1, 1), 0, 0), ((5, 6, 11), (2, 1, 3), 0, 0),
                                            ((4, 9, 10), (2, 2, 2), 2, 1)])
def test_full_stencil3d_emulated(emu_builds, tmp_path, san, N, pads, glo, ghi):
    """Interior (check-free) and boundary points, unequal pads per axis, odd last extent (pad column), ghost planes
    below and above (the slab form), every epilogue with its fused reduction."""
    _core(san, pads == (2, 1, 3))
    exe = _Exes(emu_builds, "emu_stencil3d")[san]
    rng = np.random.default_rng(N[2])
    n1, n2, n3 = N
    p1, p2, p3 = pads
    ld = n3 + (n3 & 1)
    W = (2 * p1 + 1, 2 * p2 + 1, 2 * p3 + 1)
    S = rng.standard_normal(N + W)
    S[..., p1, p2, p3] += 30.0                                   # a usable diagonal for the Jacobi epilogues
    xg = np.zeros((glo + n1 + ghi, n2, ld))
    xg[..., :n3] = rng.standard_normal((glo + n1 + ghi, n2, n3))
    b = np.zeros((n1, n2, ld))
    b[..., :n3] = rng.standard_normal(N)
    xpad = np.zeros((n1 + 2 * p1, n2 + 2 * p2, n3 + 2 * p3))
    xpad[p1 - glo:p1 + n1 + ghi, p2:p2 + n2, p3:p3 + n3] = xg[..., :n3]
    Ax = np.zeros(N)
    for k1 in range(W[0]):
        for k2 in range(W[1]):
            for k3 in range(W[2]):
                Ax += S[..., k1, k2, k3] * xpad[k1:k1 + n1, k2:k2 + n2, k3:k3 + n3]
    x = xg[glo:glo + n1, :, :n3]
    dg = S[..., p1, p2, p3]
    om = 0.7
    want = {0: (Ax, np.sum(x * Ax)), 1: (b[..., :n3] - Ax, np.sum((b[..., :n3] - Ax) ** 2)),
            2: (x + om * (b[..., :n3] - Ax) / dg, np.sum((om * (b[..., :n3] - Ax) / dg) ** 2)),
            3: (om * (b[..., :n3] - Ax) / dg, np.sum((om * (b[..., :n3] - Ax) / dg) ** 2)),
            4: (b[..., :n3] + om * Ax, np.sum((om * Ax) ** 2))}
    for epi, (y_ref, dot_ref) in want.items():
        dot, y = _stencil3d(exe, tmp_path, 0, N, pads, ld, epi=epi, has_dot=1, glo=glo, ghi=ghi, omega=om,
                            arrays=[xg, b, S], has_b=1)
        assert rel(y[..., :n3], y_ref) < 1e-14 and abs(dot - dot_ref) <= 1e-13 * abs(dot_ref)
        assert not y[..., n3:].any()                             # the pad column is never written
    _, y = _stencil3d(exe, tmp_path, 0, N, pads, ld, epi=0, has_dot=0, glo=glo, ghi=ghi, arrays=[xg, S])
    assert rel(y[..., :n3], Ax) < 1e-14
    # two-colour half sweeps: both colours, both offsets
    d = np.zeros((n1, n2, ld))
    d[..., :n3] = rng.standard_normal(N)
    i1, i2, i3 = np.meshgrid(np.arange(n1), np.arange(n2), np.arange(n3), indexing="ij")
    for off in (0, 1):
        for colour in (0, 1):
            _, xn = _stencil3d(exe, tmp_path, 1, N, pads, ld, off=off, colour=colour, arrays=[b, d])
            mask = ((i1 + i2 + i3 + off) & 1) == colour
            assert np.array_equal(xn[..., :n3], np.where(mask, b[..., :n3] + d[..., :n3], b[..., :n3]))


# ------------------------------------------------------------------------------------------------
# Peer-store halo exchange (halo_push_kernel behind poms_halo_exchange_p2p): one PROCESS per rank, the ranks' "IPC"
# memory is one file mapped shared by all of them, so the ENTER / DATA flag protocol runs between concurrent address
# spaces that drift apart by random sleeps.  Address sanitizer only (ThreadSanitizer does not see other processes).
# ------------------------------------------------------------------------------------------------
def _halo_run(exe, tmp, size, n, exchanges, seed):
    per = 8 + 2 * n + 8                        # flags | canary | ghost_lo | canary | canary | ghost_hi | canary
    buf = np.zeros((size, per))
    buf[:, 8:10] = buf[:, 10 + n:14 + n] = buf[:, 14 + 2 * n:16 + 2 * n] = -7.25e300
    path = str(tmp / "halo.bin")
    buf.tofile(path)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    procs = [subprocess.Popen([exe, path, str(r), str(size), str(n), str(exchanges), str(seed)],
                              stderr=subprocess.PIPE, text=True, env=env) for r in range(size)]
    res = []
    try:
        for pr in procs:
            res.append((pr.wait(timeout=300), pr.stderr.read()[-2000:]))
    finally:
        for pr in procs:
            if pr.poll() is None:
                pr.kill()                      # (exactly the processes started above)
    return res


@pytest.mark.parametrize("size,n,exchanges", [(2, 64, 4), (3, 5000, 8), (4, 40000, 5), (3, 0, 3)])
def test_halo_exchange_p2p_emulated(emu_builds, tmp_path, size, n, exchanges):
    """Every rank's ghost planes hold its neighbours' planes of THE SAME exchange after each call (no rank runs ahead
    into planes that are still being read, no data missing), sequence numbers advance, the block ticket is reset, the
    canaries around the ghost planes survive; edge ranks have one neighbour; 1 to 10 blocks; an empty exchange."""
    _core("asan", size == 3 and n == 5000)
    exe = _Exes(emu_builds, "emu_halo")["asan"]
    for rc, err in _halo_run(exe, tmp_path, size, n, exchanges, seed=n + size):
        assert rc == 0 and not err.strip(), (rc, err)


@pytest.mark.parametrize("san", ["asan", "tsan"])
@pytest.mark.parametrize("variant", [1, 0])
def test_tma_matvec3d_emulated_on_slab_subproblems(tma_exes, tmp_path, san, variant):
    """The multi-GPU form of the hot kernel: axis 1 cut into three slabs, every rank's sub-problem with
    its ghost planes (glo / ghi = p; the tensor maps cover owned + ghost planes, the axis-1 band rows and
    the Toeplitz range are the slab's: stencil.KronSumMatrix._launch), against the global operator."""
    _core(san, variant == 1)
    EPI, FORM = _consts()
    p, N = 3, (60, 20, 70)
    nf = [n + p for n in N]
    MK = [bs.assemble_1d_bands(p, bs.make_open_knots(p, n)) for n in nf]
    ms, ks = [m for m, k in MK], [k for m, k in MK]
    ks[2] = ks[2] + ms[2]
    coef, rg = _toeplitz_tables(ms, ks, p)
    rng = np.random.default_rng(0)
    xg, bg = rng.standard_normal(nf), rng.standard_normal(nf)
    ab = po.apply_band
    yo = (ab(ks[0], ab(ms[1], ab(ms[2], xg, 2), 1), 0) + ab(ms[0], ab(ks[1], ab(ms[2], xg, 2), 1), 0)
          + ab(ms[0], ab(ms[1], ab(ks[2], xg, 2), 1), 0))
    for s, e in ((0, 20), (21, 41), (42, 62)):
        n1 = e - s + 1
        glo, ghi = (p if s > 0 else 0), (p if e < nf[0] - 1 else 0)
        r = rg.copy()
        r[0] = max(0, int(rg[0]) - s)
        r[1] = max(int(r[0]), min(n1, int(rg[1]) - s))
        ms_l, ks_l = [ms[0][s:e + 1], ms[1], ms[2]], [ks[0][s:e + 1], ks[1], ks[2]]
        run = lambda epi, bb, om: _run_tma(tma_exes[san], tmp_path, p, FORM["sum"], EPI[epi], ms_l, ks_l,
                                           xg[s - glo:e + ghi + 1], bb, om, variant, (coef, r), glo=glo, ghi=ghi)
        dot, y = run("store", None, 1.0)
        assert rel(y, yo[s:e + 1]) < 1e-14
        assert abs(dot - np.vdot(xg[s:e + 1], yo[s:e + 1])) < 1e-13 * np.vdot(np.abs(xg[s:e + 1]), np.abs(yo[s:e + 1]))
        assert rel(run("resid", bg[s:e + 1], 1.0)[1], (bg - yo)[s:e + 1]) < 1e-14
        assert rel(run("axpy", bg[s:e + 1], 0.7)[1], (bg + 0.7 * yo)[s:e + 1]) < 1e-14
