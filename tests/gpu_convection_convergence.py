"""mg_gmres on one GPU: 3-D, p = 3, -Lap u + beta . grad u + u = f with alpha = |beta_a| / 2 on the inflow faces
(du/dn = 0 elsewhere), a seeded random right-hand side, tol 1e-10, restart 30, glt smoother, at N = 64 .. 512
elements per axis for a few velocities.  Per case: GMRES iterations, solve time (host clock around the solve,
ending in a device synchronise; one warm-up solve first), time per iteration, and its split into the mat-vec of
h.op, the V-cycle (with the copy out of the workspace) and the rest (the CGS2 orthogonalisation, the basis
updates and the host reads of the Arnoldi coefficients).  The split comes from CUDA events recorded around every
mat-vec and V-cycle call inside the timed solve; gmres reads its Arnoldi coefficients on the host every step, so
the calls do not overlap.  The card name and power limit are read in the same run and written with the numbers.
profiles/r03_convection_p3.txt is the output of
    python tests/gpu_convection_convergence.py                (= --N 64,128,256,512, the default --out)"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from poms_b200 import mg  # noqa: E402
from poms_b200.mg import Hierarchy, mg_gmres  # noqa: E402
from poms_b200.stencil import StencilVector  # noqa: E402

BETAS = [(1.0, 0.0, 0.0), (10.0, -5.0, 3.0), (50.0, 20.0, 0.0)]


class TimedOp:
    """h.op with CUDA events around every apply."""

    def __init__(self, A):
        self.A, self.shape, self.ev = A, A.shape, []

    def apply(self, *a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = self.A.apply(*a, **k)
        e1.record()
        self.ev.append((e0, e1))
        return out


def _ms(ev):
    return sum(a.elapsed_time(b) for a, b in ev)


def run(N, beta, p=3):
    robin = [((0.5 * b, 0.0) if b > 0 else (0.0, -0.5 * b)) for b in beta]
    h = Hierarchy(p, [N] * 3, device="cuda", c=1.0, robin=robin, beta=beta)
    V = h.levels[0].V
    b = StencilVector(V)
    g = torch.Generator(device="cuda").manual_seed(7)
    b.data.copy_(torch.rand(b.data.shape, generator=g, dtype=torch.float64, device="cuda") - 0.5)
    mg_gmres(h, b, tol=1e-10)                       # warm-up: modules, tensor maps, allocations
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    x, info = mg_gmres(h, b, tol=1e-10)
    torch.cuda.synchronize()
    t_solve = time.perf_counter() - t0
    # split, in a second solve with events (same operations)
    op, orig_op, orig_vc = TimedOp(h.op), h.op, mg.vcycle
    vc_ev = []

    def vcycle(h_, l, v, final_dot=None):
        if l != 0:
            return orig_vc(h_, l, v, final_dot)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = orig_vc(h_, l, v, final_dot)
        e1.record()
        vc_ev.append((e0, e1))
        return out
    h.op, mg.vcycle = op, vcycle
    try:
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        _, info2 = mg_gmres(h, b, tol=1e-10)
        torch.cuda.synchronize()
        t_inst = time.perf_counter() - t1
    finally:
        h.op, mg.vcycle = orig_op, orig_vc
    assert info2["niter"] == info["niter"]
    t_mv, t_vc = _ms(op.ev) / 1e3, _ms(vc_ev) / 1e3
    return dict(N=N, beta=beta, dofs=int(np.prod(V.npts)), niter=info["niter"], success=info["success"],
                rel_res=info["res_norm"] / info["res_norm0"], t_solve=t_solve, t_inst=t_inst, n_mv=len(op.ev),
                n_vc=len(vc_ev), t_mv=t_mv, t_vc=t_vc, t_rest=t_inst - t_mv - t_vc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", default="64,128,256,512")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else torch.cuda.get_device_name(0)
    out = args.out or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                   "r03_convection_p3.txt")
    lines = ["# mg_gmres, 3-D p=3, c=1, alpha=|beta_a|/2 on inflow faces, random rhs, tol 1e-10, restart 30, glt "
             "smoother; card: %s (name, power limit, max SM clock)" % card,
             "# solve = host clock around one solve after a warm-up solve; the split (mat-vec of h.op, V-cycle incl. "
             "its copy, rest = orthogonalisation + basis updates + host reads) is from CUDA events in a second, "
             "instrumented solve whose total is t_inst",
             "%5s %-18s %11s %6s %9s %10s %12s %9s %9s %9s %9s" % ("N", "beta", "DOFs", "iters", "rel.res", "solve s",
                                                                  "ms/iter", "t_inst s", "matvec", "vcycle", "rest")]
    for N in [int(v) for v in args.N.split(",")]:
        for beta in BETAS:
            r = run(N, beta)
            per = 1e3 * r["t_solve"] / max(r["niter"], 1)
            lines.append("%5d %-18s %11d %6d %9.1e %10.3f %12.2f %9.3f %8.0f%% %8.0f%% %8.0f%%" % (
                r["N"], str(beta), r["dofs"], r["niter"], r["rel_res"], r["t_solve"], per, r["t_inst"],
                100 * r["t_mv"] / r["t_inst"], 100 * r["t_vc"] / r["t_inst"], 100 * r["t_rest"] / r["t_inst"]))
            print(lines[-1], "(mat-vecs %d, V-cycles %d, success %s)" % (r["n_mv"], r["n_vc"], r["success"]),
                  flush=True)
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
