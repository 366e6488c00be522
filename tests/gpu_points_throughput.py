"""Throughput of the particle coupling of poms_b200.fem on one GPU: 3-D, p = 3, m = 10^8 points uniform in
[0,1]^3, on a 128^3-element space (about 48 points per cell) and a 512^3-element space (fewer than one).

Per space, CUDA-event means over `--reps` (default 20) calls after 3 warm-up calls:
  * evaluate_points without and with grad, for the points in random order and sorted by cell;
  * deposit as a whole, and split into its stages: the locate kernel, the stable torch.sort of the cell keys,
    and the chunk loop (torch.searchsorted of the chunk's cell offsets + poms_points_moments +
    poms_points_assemble), the last restated here with the library's entry points as fem.deposit runs it.
Each time is set against the algorithmic bytes: evaluate 24 B of coordinates + 8 B of u (+ 24 B of gradient)
per point + one read of the coefficients; deposit 24 + 8 B per point + one write of the coefficients.  The
sort and the moments move more (the sorted keys and the permutation, the moments: 8 (p+1)^3 B per cell
written and read back); the bandwidth column uses the algorithmic bytes only.  The card name and power limit
are read in the same run and written with the numbers.  profiles/r03_points_p3.txt is the output of
    python tests/gpu_points_throughput.py"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from poms_b200 import _lib, fem  # noqa: E402
from poms_b200 import bsplines as bs  # noqa: E402
from poms_b200.stencil import StencilVector, StencilVectorSpace, _stream  # noqa: E402


def timed(fn, reps):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_points_p3.txt"))
    ap.add_argument("--m", type=int, default=10 ** 8)
    ap.add_argument("--N", default="128,512")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else torch.cuda.get_device_name(0)
    p, d, m = 3, 3, args.m
    L = _lib.lib()
    lines = ["# poms_b200.fem particle coupling, 3-D p=%d, m=%d uniform random points; card: %s" % (p, m, card),
             "# ms: CUDA-event mean over %d calls after 3 warm-up calls; GBps: algorithmic bytes / time" % args.reps]
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    P = torch.rand((m, d), dtype=torch.float64, device=dev, generator=g)
    w = torch.rand(m, dtype=torch.float64, device=dev, generator=g)
    for N in [int(v) for v in args.N.split(",")]:
        knots = [bs.make_open_knots(p, N + p)] * d
        V = StencilVectorSpace([N + p] * d, [p] * d, [False] * d, device=dev)
        x = StencilVector(V, zero=False)
        x.data.copy_(torch.rand(V.npts, dtype=torch.float64, device=dev, generator=g))
        ndof = (N + p) ** d
        # cell keys and the cell-sorted copy of the points
        pts, _, Tdev, T = fem._points(knots, p, d, dev, P)
        n1, n2, n3, ld, pld = fem._geom(V)
        key = torch.empty(m, dtype=torch.int64, device=dev)
        locate = lambda: _lib.check(L.poms_points_locate(pts.data_ptr(), d, m, n1, n2, n3, p, T[0], T[1], T[2],
                                                         key.data_ptr(), _stream()), "poms_points_locate")
        locate()
        skey, perm = torch.sort(key, stable=True)
        Ps = P[perm]
        row = {"N": N, "dofs": ndof, "m": m, "points_per_cell": m / N ** d}
        by_ev = 32.0 * m + 8.0 * ndof
        by_evg = 56.0 * m + 8.0 * ndof
        by_dep = 32.0 * m + 8.0 * ndof
        for name, Q in (("random", P), ("sorted", Ps)):
            t = timed(lambda: fem.evaluate_points(x, knots, p, Q), args.reps)
            row["eval_%s_ms" % name], row["eval_%s_GBps" % name] = t, by_ev / t / 1e6
            t = timed(lambda: fem.evaluate_points(x, knots, p, Q, grad=True), args.reps)
            row["eval_grad_%s_ms" % name], row["eval_grad_%s_GBps" % name] = t, by_evg / t / 1e6
        out = StencilVector(V, zero=False)
        t = timed(lambda: fem.deposit(V, knots, p, P, w, out=out), args.reps)
        row["deposit_ms"], row["deposit_GBps"] = t, by_dep / t / 1e6
        row["deposit_locate_ms"] = timed(locate, args.reps)
        row["deposit_sort_ms"] = timed(lambda: torch.sort(key, stable=True), args.reps)
        C1 = C2 = C3 = N
        nt = (p + 1) ** d
        ch = min(C1, max(1, fem.CHUNK_BYTES // (8 * C2 * C3 * nt)))
        mom = torch.empty(ch * C2 * C3 * nt, dtype=torch.float64, device=dev)

        def stages():
            for c0 in range(0, C1, ch):
                c1 = min(C1, c0 + ch)
                cells = torch.arange(c0 * C2 * C3, c1 * C2 * C3 + 1, dtype=torch.int64, device=dev)
                offs = torch.searchsorted(skey, cells)
                _lib.check(L.poms_points_moments(pts.data_ptr(), w.data_ptr(), d, perm.data_ptr(), offs.data_ptr(),
                                                 c0, c1, n1, n2, n3, p, T[0], T[1], T[2], mom.data_ptr(),
                                                 _stream()), "poms_points_moments")
                _lib.check(L.poms_points_assemble(mom.data_ptr(), c0, c1, n1, n2, n3, p, out.flat.data_ptr(), ld,
                                                  pld, 0 if c0 == 0 else c0 + p, _stream()), "poms_points_assemble")
        row["deposit_chunks"] = -(-C1 // ch)
        row["deposit_moments_assemble_ms"] = timed(stages, args.reps)
        ref = fem.deposit(V, knots, p, P, w)
        row["stages_match_deposit"] = bool(torch.equal(ref.flat, out.flat))
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)
        del x, out, ref, mom, key, skey, perm, Ps, pts
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
