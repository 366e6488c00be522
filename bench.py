#!/usr/bin/env python
"""bench.py -- the POMS hot path on B200: MG-preconditioned CG to 1e-10 relative residual.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c5|c2|c3|c4|c1] [--impl reference]
                    [--dump-outputs DIR]

A "step" is ONE complete MG-PCG solve (b = 1 on every DOF, x0 = 0) of the synthetic
-Lap(u)+u problem of the chosen BASELINE config; `value` = DOF / (seconds per solve), inputs
resident in HBM.  `e2e` is the same solve through the public API with HOST buffers: pinned
host b -> device, solve, x -> pinned host, all inside the timed region.
Default config: c5 (3-D, degree 3, 512^3 elements per GPU), the configuration the BASELINE
metric is quoted on; it fits one GPU.  Under torchrun (N > 1) the grid is slab-partitioned along
axis 1, 512 element planes per GPU (weak scaling).

--impl reference times the reference's CPU algorithm (oracle port: the reference itself is
pure Python over an absent third-party package and cannot travel) on the host cores, on a
bounded sample of the same workload.

--dump-outputs DIR writes what the last timed solve returned (see dump_outputs) so that two builds
can be compared output for output; the inputs are the same on every run with the same arguments.
The bench writes nothing into the source tree, which may be read-only.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

CONFIGS = {
    # name: (ndim, p, elements per axis, description)
    "c1": (2, 3, 64, "2-D Poisson p=3 64x64"),
    "c2": (2, 3, 2048, "2-D Poisson p=3 2048x2048"),
    "c3": (3, 3, 128, "3-D Poisson p=3 128^3"),
    "c4": (2, 5, 8192, "2-D Poisson p=5 8192x8192"),
    "c5": (3, 3, 512, "3-D Poisson p=3 512^3"),
}
METRIC = "DOF/s to 1e-10 rel. residual (MG-PCG); Kron matvec GB/s vs HBM peak"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


_cpu_port = {}


def pin_cpu_threads():
    """The CPU port parallelises with numba prange; BLAS/OpenMP pools underneath it oversubscribe the
    cores (round 1: 2.7x run-to-run spread, the torchrun arm -- which exports OMP_NUM_THREADS=1 -- being
    the fast one).  Pin: numba = all host cores, every BLAS/OpenMP pool = 1 thread.  Must run before
    numba / numpy are imported."""
    n = os.cpu_count() or 1
    os.environ["NUMBA_NUM_THREADS"] = str(n)
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    return n


def numba_cache_outside_tree():
    """The CPU port compiles with numba cache=True, which writes next to its source (or fails at
    import when no cache location is writable): point numba at a temporary directory instead, unless
    the caller chose one.  Must run before numba is imported."""
    if "NUMBA_CACHE_DIR" not in os.environ:
        d = tempfile.mkdtemp(prefix="poms_b200_numba_")
        atexit.register(shutil.rmtree, d, True)
        os.environ["NUMBA_CACHE_DIR"] = d


def cpu_port_solve(ndim, p, N, tol=1e-10, smoother="glt", Nc=8, ratio=4.0):
    """One MG-PCG solve with the CPU port of the same algorithm: oracle/poms_oracle_mt.py (numba,
    all host threads), or the single-threaded NumPy oracle if numba is unavailable.  b = A x0 like
    the GPU arm.  Returns (dof, seconds, info, cores, label)."""
    import numpy as np
    if "mod" not in _cpu_port:
        try:
            import numba
            from oracle import poms_oracle_mt as mt
            mt.warmup()                      # JIT compilation is not timed
            _cpu_port.update(mod=mt, cls=mt.MGHierarchyMT, cores=int(numba.get_num_threads()),
                             label="numba-threaded port (oracle/poms_oracle_mt.py)")
        except Exception as exc:             # pragma: no cover
            from oracle import poms_oracle as po
            _cpu_port.update(mod=po, cls=po.MGHierarchy, cores=1,
                             label="NumPy/SciPy oracle, single thread (numba unavailable: %s)" % exc)
    # same hierarchy rule as the GPU arm: uniform coarsening down to Nc elements per axis
    h = _cpu_port["cls"](p, [N] * ndim, smoother=smoother, nu=1, Nc=Nc, coarsen="uniform", ratio=ratio)
    A = h.levels[0]["A"]
    x0 = np.zeros(A.npts)
    for a in range(ndim):
        shp = [1] * ndim
        shp[a] = -1
        x0 = x0 + np.arange(A.npts[a], dtype=float).reshape(shp)
    b = A.dot(x0 + 1.0)
    t0 = time.perf_counter()
    x, info = h.mg_pcg(b, tol=tol, maxiter=200)
    dt = time.perf_counter() - t0
    return int(np.prod(b.shape)), dt, info, _cpu_port["cores"], _cpu_port["label"]


def resolve_smoother(name, p):
    """'auto': the polynomial GLT smoother (three fused Kronecker band passes) where its second
    factor fits the kernels' half-bandwidth limit (2 <= p <= 3); exact GLT line solves otherwise.
    Both arms (GPU and CPU port) use the same choice."""
    if name == "auto":
        return "glt_poly" if 2 <= p <= 3 else "glt"
    return name


def cpu_sample_size(ndim):
    # bounded sample: ~10-30 s of CPU work
    return 128 if ndim == 3 else 1024


DUMP_SAMPLE = 1 << 22       # entries of x written by --dump-outputs: 32 MB of float64


def dump_indices(npts):
    """Flat row-major indices into the global grid of the x entries --dump-outputs writes: every
    point when there are at most DUMP_SAMPLE, else a sorted sample drawn with a fixed seed (C5:
    515^3 points, 1.1 GB in full)."""
    import numpy as np
    n = int(np.prod(npts))
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLE))


def dump_outputs(path, x, info, world, rank):
    """Write what mg_pcg returned to the caller as path/<name>.npy, all float64: x.npy (x at
    dump_indices(V.npts), gathered over the slabs), residual_history.npy, and the scalars niter,
    restarts, success, res_norm, res_norm0.  Collective when world > 1; rank 0 writes."""
    import numpy as np
    import torch
    V = x.space
    dev = x.data.device
    sub = np.unravel_index(dump_indices(V.npts), V.npts)
    own = (sub[0] >= V.starts[0]) & (sub[0] <= V.ends[0])
    loc = tuple(torch.as_tensor(s[own] - (V.starts[0] if a == 0 else 0), device=dev)
                for a, s in enumerate(sub))
    xs = torch.zeros(len(own), dtype=torch.float64, device=dev)
    xs[torch.as_tensor(np.flatnonzero(own), device=dev)] = x.data[loc]
    if world > 1:
        torch.distributed.all_reduce(xs)        # every sampled point is owned by exactly one slab
    if rank != 0:
        return
    out = {"x": xs.cpu().numpy(), "residual_history": np.asarray(info["history"], dtype=np.float64)}
    for k in ("niter", "restarts", "success", "res_norm", "res_norm0"):
        out[k] = np.float64(info[k])
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)


_JSON_OUT = None


def _claim_stdout():
    """Keep the real stdout for the ONE JSON line and send everything else a library may print
    there (NCCL's version banner, numba / torch notices) to stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


REFERENCE_TIME_BUDGET_S = 240.0
# Tier-A baseline (SURVEY section 8d): the UNMODIFIED reference timed in the dev container, one core
# (it cannot travel: /root/reference does not exist on the GPU box) -- oracle/time_reference_c1.py
TIER_A_NOTE = ("unmodified reference on C1 (2-D p=3 64x64, 4489 DOF), 1 core, dev container: see "
               "profiles/r02_reference_tierA_c1.txt (oracle/time_reference_c1.py)")


def run_reference(args, rank):
    """--impl reference: the reference's CPU algorithm on the host cores (oracle port).  Every step is
    one full solve of the bounded sample; the run stops after REFERENCE_TIME_BUDGET_S seconds of
    solves (reported: `steps` = solves actually timed, `steps_requested`, `time_budget_s`)."""
    if rank != 0:
        return
    pin_cpu_threads()
    ndim, p, N, desc = CONFIGS[args.config]
    Ns = min(N, cpu_sample_size(ndim))
    vals = []
    t_all = time.perf_counter()
    for i in range(args.warmup + args.steps):
        dof, dt, info, cores, label = cpu_port_solve(ndim, p, Ns, ratio=args.ratio,
                                                     smoother=resolve_smoother(args.smoother, p))
        if i >= args.warmup:
            vals.append(dof / dt)
        if time.perf_counter() - t_all > REFERENCE_TIME_BUDGET_S and i >= min(args.warmup, 1):
            if not vals:
                vals.append(dof / dt)
            break
    v = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "DOF/s", "n_gpus": args.gpus,
        "steps": len(vals), "steps_requested": args.steps, "time_budget_s": REFERENCE_TIME_BUDGET_S,
        "warmup": args.warmup, "ms_per_step": 1e3 * dof / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "%s (CPU sample: %d^%d elements, same MG-PCG algorithm, b = A x0)"
                               % (desc, Ns, ndim), "p": p, "ndim": ndim, "elements_per_axis": Ns,
                   "iterations": info["niter"]},
        "cpu_baseline": {"value": v, "unit": "DOF/s", "cores": cores, "kind": "port",
                         "threads": {k: os.environ.get(k) for k in
                                     ("NUMBA_NUM_THREADS", "OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS")},
                         "sample": "%d^%d elements, %s, %s smoother, full MG-PCG solve to 1e-10"
                                   % (Ns, ndim, label, resolve_smoother(args.smoother, p)),
                         "literal_reference_c1": TIER_A_NOTE},
        "e2e": {"value": v, "unit": "DOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c5", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--smoother", default="auto", choices=["auto", "glt", "glt_poly", "jacobi"])
    ap.add_argument("--nu", type=int, default=1)
    ap.add_argument("--ratio", type=float, default=6.0,
                    help="smoothing interval [lmax/ratio, lmax] of the Richardson / Chebyshev smoother "
                         "(step 1/theta, theta = (lmax + lmin)/2).  Measured on C5: ratio 2.5 / 3 / 4 / 6 / 10 "
                         "-> 22 / 21 / 21 / 20 / 20 iterations, 258 / 247 / 246 / 236 / 237 ms "
                         "(profiles/r02_bench_c5_ratio*.json); both arms use the same value")
    ap.add_argument("--nc", type=int, default=0, help="coarsest grid (elements per axis); 0 = auto")
    ap.add_argument("--rhs", default="auto", choices=["auto", "ones", "manufactured"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-timing", action="store_true")
    ap.add_argument("--scaling", default="auto", choices=["auto", "weak", "strong"],
                    help="N > 1: weak = N element planes per GPU along axis 1 (c5: BASELINE's weak-scaling "
                         "sweep), strong = the named grid split into slabs (c4: BASELINE config 4, "
                         "sources/scalability.py:7-19); auto = strong for c4, weak otherwise")
    ap.add_argument("--setup", default="host", choices=["host", "device"],
                    help="where the 1-D setup of the hierarchy runs (device: csrc/poms_setup.cu)")
    ap.add_argument("--no-exact-glt", action="store_true",
                    help="skip the extra solves with the reference's exact GLT smoother (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the solution and solver info of the last timed "
                         "step to DIR/<name>.npy (float64; x sampled at fixed points, at most 34 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    numba_cache_outside_tree()
    pin_cpu_threads()
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from poms_b200 import _lib, profiling
    from poms_b200.mg import Hierarchy, mg_pcg
    from poms_b200.stencil import StencilVector, EPI_RESID

    if args.steps < 1 or args.warmup < 0:
        raise SystemExit("steps >= 1, warmup >= 0")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    slab = None
    if world > 1:
        from poms_b200.dist import Slab
        # NCCL writes its version banner to stdout when NCCL_DEBUG is set; stdout carries the JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
        slab = Slab(dist.group.WORLD, dev)
    ndim, p, N, desc = CONFIGS[args.config]
    args.smoother = resolve_smoother(args.smoother, p)
    Ns = [N] * ndim
    scaling = args.scaling if args.scaling != "auto" else ("strong" if args.config == "c4" else "weak")
    if world > 1 and scaling == "weak":
        Ns[0] = N * world          # weak scaling: N element planes per GPU along axis 1
    # weak scaling: the domain grows with the grid, [0, G] x [0,1]^(d-1), so the elements stay cubes
    # (keeping [0,1]^d would make the global problem anisotropic and change the iteration count)
    lengths = [float(world) if scaling == "weak" else 1.0] + [1.0] * (ndim - 1)
    # coarsest level: solved exactly by fast diagonalisation, so it need not be tiny; stopping at 32
    # elements per axis in 3-D saves two levels of launch-latency-bound kernels per V-cycle
    # Coarsest grid (solved exactly by fast diagonalisation; its dense 1-D eigenbasis contractions run on
    # the fp64 tensor cores, poms_axis_dense_dmma).  One GPU, 3-D: a quarter of the fine resolution per
    # axis, at most 128 elements (C5: 131^3 unknowns, 3 levels; measured 246 ms vs 259 ms with 64 and
    # 262 ms with 32 elements, profiles/r02_bench_c5_nc*.json).  With slabs the coarsest level is gathered
    # and solved redundantly on every GPU, so it stays at 32 elements per axis per GPU (5 levels at
    # every N > 1; its slab-axis eigenbasis is (32 G + p)^2).  --nc forces one value for every N.
    if args.nc > 0:
        Nc = args.nc
    elif ndim == 3:
        Nc = max(32, min(128, N // 4)) if world == 1 else 32
    else:
        Nc = 8
    t_setup = time.perf_counter()
    h = Hierarchy(p, Ns, device=dev, smoother=args.smoother, nu=args.nu, slab=slab,
                  lengths=lengths, Nc=Nc, coarsen="uniform", setup=args.setup, ratio=args.ratio)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup
    t_setup_other = None
    if world == 1:
        # the other setup mode, timed for the record (its hierarchy is dropped: work vectors are lazy)
        other = "device" if args.setup == "host" else "host"
        try:
            if other == "device":           # first use compiles nothing but loads kernels / cuSOLVER: warm
                Hierarchy(p, [16] * ndim, device=dev, smoother=args.smoother, Nc=8, setup="device")
            t0 = time.perf_counter()
            Hierarchy(p, Ns, device=dev, smoother=args.smoother, nu=args.nu, lengths=lengths, Nc=Nc,
                      coarsen="uniform", setup=other)
            torch.cuda.synchronize()
            t_setup_other = (other, round(time.perf_counter() - t0, 3))
        except Exception as exc:             # informational
            t_setup_other = (other, "failed: %r" % (exc,))
    V = h.levels[0].V
    dof_global = int(np.prod(V.npts))
    b = StencilVector(V)
    rhs = args.rhs
    if rhs == "auto":
        # b = 1 (mg_jac.py:59-61) is a coefficient vector, not a load vector: at 2048^2 (2-D) or
        # 4096x512x512 (3-D, 8 GPUs) |A||x| / |b| ~ 1e6, so the TRUE relative residual floors at
        # 1e-10 .. 5e-10 in fp64 whatever the solver does (measured).  The bench therefore uses the
        # reference's other right-hand side, b = A x0 with x0[i] = i1 + i2 (+ i3) + 1
        # (sources/tests/test_pcg.py:52-58); --rhs ones selects the script's b = 1.
        rhs = "manufactured"
    if rhs == "ones":
        b.data.fill_(1.0)
    else:
        x0 = StencilVector(V)
        idx = [torch.arange(V.starts[a] if a == 0 else 0,
                            (V.ends[a] + 1) if a == 0 else V.npts[a], dtype=torch.float64,
                            device=dev) for a in range(ndim)]
        ramp = idx[0].reshape([-1] + [1] * (ndim - 1)) + 1.0
        for a in range(1, ndim):
            ramp = ramp + idx[a].reshape([1] * a + [-1] + [1] * (ndim - 1 - a))
        x0.data.copy_(ramp)
        b = h.levels[0].A.dot(x0)
    L = _lib.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def solve():
        return mg_pcg(h, b, tol=1e-10, maxiter=200)

    for _ in range(args.warmup):
        x, info = solve()
    # ---- timed region: K solves, device-resident inputs, NO per-kernel instrumentation ---------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    profiling.enable(False)
    barrier()
    l0 = L.poms_launch_count()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        x, info = solve()
    e1.record()
    barrier()
    launches = L.poms_launch_count() - l0
    ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # now: x is the hierarchy's persistent solution vector, which the passes below overwrite
        dump_outputs(args.dump_outputs, x, info, world, rank)
    # ---- separate instrumented pass (CUDA events around every kernel family) for the roofline and
    # the per-kernel breakdown: its event records perturb the latency-bound coarse levels, so it
    # is kept out of the headline timing above
    kern, kern_fine, prof_steps, ms_prof = {}, {}, 0, 0.0
    if not args.no_kernel_timing:
        prof_steps = min(args.steps, 3)
        profiling.enable(True)
        barrier()
        e0.record()
        for _ in range(prof_steps):
            solve()
        e1.record()
        barrier()
        ms_prof = e0.elapsed_time(e1) / prof_steps
        kern = profiling.summary()
        try:
            kern_fine = profiling.summary_largest()
        except Exception:                        # informational only
            kern_fine = {}
        profiling.enable(False)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # true residual of the returned solution (work is not skipped / cached)
    r = StencilVector(V)
    h.levels[0].A.apply(x, r, EPI_RESID, b=b)
    true_rel = (r.dot(r) / b.dot(b)) ** 0.5

    # ---- e2e: host buffers, H2D + solve + D2H inside the timed region -------------------------
    nloc = V.local_size
    b_host = b.data.cpu().pin_memory()
    x_host = torch.empty(V.local_shape, dtype=torch.float64).pin_memory()

    def solve_host():
        bb = StencilVector(V)
        bb.data.copy_(b_host, non_blocking=True)
        xx, inf = mg_pcg(h, bb, tol=1e-10, maxiter=200)
        x_host.copy_(xx.data, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return inf

    solve_host()
    barrier()
    e0.record()
    for _ in range(args.steps):
        solve_host()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e2e = float(t.item())

    # ---- the reference's own smoother beside the headline: glt_poly (polynomial approximation of the
    # GLT solve, an EXTENSION) is the default for p <= 3; the exact GLT Kronecker solve
    # (sources/solvers.py:260,288: kron_solve_par(M2, M1, r)) is timed on the same problem
    exact_glt = None
    if args.smoother == "glt_poly" and world == 1 and not args.no_exact_glt:
        try:
            hg = Hierarchy(p, Ns, device=dev, smoother="glt", nu=args.nu, slab=slab, lengths=lengths,
                           Nc=Nc, coarsen="uniform", ratio=args.ratio)
            xg, infog = mg_pcg(hg, b, tol=1e-10, maxiter=200)
            barrier()
            ng = min(args.steps, 3)
            e0.record()
            for _ in range(ng):
                xg, infog = mg_pcg(hg, b, tol=1e-10, maxiter=200)
            e1.record()
            barrier()
            exact_glt = {"smoother": "glt (exact banded Kronecker solves, the reference's post-smoother)",
                         "ms_per_step": e0.elapsed_time(e1) / ng, "iterations": infog["niter"],
                         "value": dof_global / (e0.elapsed_time(e1) / ng * 1e-3), "unit": "DOF/s"}
            del hg, xg
        except Exception as exc:                 # informational: never loses the headline
            exact_glt = {"failed": repr(exc)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    steps = max(prof_steps, 1)
    ms_headline, ms = ms, (ms_prof if prof_steps else ms)      # shares refer to the instrumented pass
    for d in kern.values():
        d["ms_per_step"] = d["ms"] / steps
        d["share"] = d["ms"] / (ms * steps) if ms > 0 else 0.0
    mv_name = "kron_matvec_%dd" % ndim
    dominant = max(kern, key=lambda k: kern[k]["ms"]) if kern else mv_name
    roof = None
    if kern:
        k = kern[dominant]
        avg_ms = k["ms"] / k["launches"]
        achieved = k["bytes"] / k["launches"] / (avg_ms * 1e-3) / 1e9
        # DRAM traffic per launch: the per-variant ncu table (profiles/traffic.json: dram bytes read +
        # written of one fine-level launch of every variant the solve uses) weighted by the variants'
        # launch counts in one PCG iteration; null when no capture of this kernel family exists
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f).get(dominant)
            if tj:
                traffic = tj["traffic_over_algorithmic"] * k["bytes"] / k["launches"]
                traffic_src = tj.get("source")
        roof = {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src, "launches": k["launches"],
                "avg_launch_ms": avg_ms, "share_of_step": k["share"],
                "algorithmic_bytes_per_launch": k["bytes"] / k["launches"]}
        kf = kern_fine.get(dominant)
        if kf and kf.get("launches") and kf.get("ms", 0.0) > 0:
            # the same kernel family restricted to its largest (fine-level) launches: the aggregate
            # above also averages over the latency-bound coarse-level launches of the V-cycle
            roof["fine_level"] = {"achieved": kf["gbs"], "frac": kf["gbs"] / peak,
                                  "launches": kf["launches"],
                                  "avg_launch_ms": kf["ms"] / kf["launches"],
                                  "share_of_step": kf["ms"] / (ms * steps) if ms > 0 else 0.0}
    ms = ms_headline
    # which transfer kernel every level pair takes (mg.Transfer._want_fused): "v2" = one-pass kernels of
    # poms_transfer3d_v2.cu, "v1" = round-1 one-pass kernels, None = per-axis gathers
    try:
        transfer_note = [{"fine_points_per_gpu": int(np.prod(l.V.local_shape)),
                          "restrict": l.transfer._want_fused(l.V.local_shape, "restrict"),
                          "prolong": l.transfer._want_fused(l.V.local_shape, "prolong")}
                         for l in h.levels[:-1]]
    except Exception as exc:                     # informational only
        transfer_note = "n/a: %r" % (exc,)
    line = {
        "metric": METRIC, "value": dof_global / (ms * 1e-3), "unit": "DOF/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc + ((" per GPU, slab-partitioned along axis 1" if scaling == "weak"
                                        else " split into %d slabs along axis 1" % world) if world > 1
                                       else ""),
                   "ndim": ndim, "p": p, "elements": Ns, "dof": dof_global, "domain": lengths,
                   "solver": "pcg + V(%d,%d) %s-Chebyshev multigrid (smoothing interval lmax/%g .. lmax), "
                             "tol 1e-10 relative" % (args.nu, args.nu, args.smoother, args.ratio),
                   "smoother_note": ("glt_poly = degree-3 polynomial approximation of the reference's GLT "
                                     "Kronecker solve, an EXTENSION (DESIGN.md section 3); `exact_glt` "
                                     "carries the same solve with the reference's exact GLT smoother")
                                    if args.smoother == "glt_poly" else "reference smoother family",
                   "setup_seconds": round(t_setup, 3), "setup_mode": args.setup,
                   "setup_seconds_other_mode": t_setup_other,
                   "setup_note": "Hierarchy construction (1-D operators, transfers, smoother bounds, "
                                 "coarse eigenbases), outside the timed region",
                   "rhs": "b = 1 (mg_jac.py:59-61)" if rhs == "ones" else
                          "b = A x0, x0[i] = sum(i_a) + 1 (tests/test_pcg.py:52-58)",
                   "coarsest_elements": Nc,
                   "iterations": info["niter"], "restarts": info.get("restarts", 0),
                   "levels": len(h.levels),
                   "transfer_kernels": transfer_note,
                   "rel_residual_reported": info["res_norm"] / info["res_norm0"],
                   "rel_residual_true": true_rel,
                   "l2_note": "vectors are %.0f MB each, larger than the 126 MB L2"
                              % (8 * dof_global / world / 1e6)},
        "gpu_launches": int(launches),
        "e2e": {"value": dof_global / (ms_e2e * 1e-3), "unit": "DOF/s",
                "ms_per_step": ms_e2e, "h2d_bytes_per_step": 8 * nloc * world,
                "d2h_bytes_per_step": 8 * nloc * world},
        "clocks": clocks,
        "exact_glt": exact_glt,
        "roofline": roof,
        "kernels": {k: {"launches": v["launches"], "ms_per_step": round(v["ms_per_step"], 4),
                        "share": round(v["share"], 4), "gbs": round(v["gbs"], 1)}
                    for k, v in sorted(kern.items(), key=lambda kv: -kv[1]["ms"])},
    }
    if mv_name in kern:
        k = kern[mv_name]
        line["kron_matvec"] = {"achieved_gbs": k["gbs"], "frac_of_peak": k["gbs"] / peak,
                               "launches": k["launches"]}
    if not args.no_cpu_baseline and world == 1:      # reported on rank 0 at N = 1 only
        Ns_cpu = min(N, cpu_sample_size(ndim))
        # the CPU port has the two GLT smoothers only
        smo = "glt" if args.smoother == "jacobi" else args.smoother
        try:
            # the CPU port inverts its coarsest operator densely: its coarsest grid stays small
            # (same rule as --impl reference: 8 elements per axis)
            dofc, dtc, infoc, cores, label = cpu_port_solve(ndim, p, Ns_cpu, smoother=smo, Nc=8,
                                                            ratio=args.ratio)
            line["cpu_baseline"] = {
                "value": dofc / dtc, "unit": "DOF/s", "cores": cores, "kind": "port",
                "host_cores_available": os.cpu_count(),
                "threads": {k: os.environ.get(k) for k in
                            ("NUMBA_NUM_THREADS", "OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS")},
                "literal_reference_c1": TIER_A_NOTE,
                "sample": "%d^%d elements (%d DOF), one full MG-PCG solve to 1e-10, %s, %s smoother, "
                          "%d iterations, %.1f s" % (Ns_cpu, ndim, dofc, label, smo, infoc["niter"], dtc)}
        except Exception as exc:             # the GPU numbers above must still be reported
            line["cpu_baseline"] = {"value": None, "unit": "DOF/s", "cores": 0, "kind": "port",
                                    "sample": "failed: %r" % (exc,)}
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
