"""Manufactured-solution study of poms_b200.fem on one GPU: 3-D, p = 3, u = prod cos(pi x_a) on [0,1]^3,
f = (1 + 3 pi^2) u, b = load_vector(f), mg_pcg to 1e-12, error_norms(u, grad u), at N = 64 .. 512 elements
per axis.  Per N: errors, observed orders, iterations, and CUDA-event times of the torch evaluation of the
callables, of the poms_quad_to_coef_3d kernel, of the solve and of the poms_quad_error_3d kernel (the callable
and kernel intervals of every chunk are separated by events recorded inside the callable wrapper), with each
kernel's algorithmic bytes (8 (p+1)^3 B per element per array of values, plus the coefficient vector),
bandwidth and share of the measured 6416.7 GB/s peak.  The card name and power limit are read in the same run
and written with the numbers.  A kernel interval runs from the end of one callable to the start of the next, so
it includes the host's launch overhead of that chunk: where it is a few milliseconds or less (N = 64, 128: one
chunk each) the bandwidths measure that overhead, not the kernel; from N = 256 on the intervals are
kernel-dominated.  profiles/r03_fem_convergence_p3.txt is the output of
    python tests/gpu_fem_convergence.py                       (= --p 3 --N 64,128,256,512, the default --out)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from poms_b200 import fem  # noqa: E402
from poms_b200.mg import Hierarchy, mg_pcg  # noqa: E402

PEAK = 6416.7e9


class Timed:
    """Wraps a callable: events before / after each call; the interval from the end of one call to the start
    of the next (or to `close`) is the kernel that consumed the values."""

    def __init__(self, fn):
        self.fn, self.ev = fn, []

    def __call__(self, *X):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = self.fn(*X)
        b.record()
        self.ev.append((a, b))
        return out

    def close(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        torch.cuda.synchronize()
        t_f = sum(a.elapsed_time(b) for a, b in self.ev)
        ends = [a for a, _ in self.ev[1:]] + [e]
        t_k = sum(b.elapsed_time(n) for (_, b), n in zip(self.ev, ends))
        return t_f, t_k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="default: profiles/r03_fem_convergence_p<p>.txt")
    ap.add_argument("--N", default="64,128,256,512")
    ap.add_argument("--p", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else torch.cuda.get_device_name(0)
    p, d, kp = args.p, 3, np.pi
    u = lambda X, Y, Z: torch.cos(kp * X) * torch.cos(kp * Y) * torch.cos(kp * Z)
    f = lambda X, Y, Z: (1.0 + d * kp * kp) * u(X, Y, Z)
    gu = lambda X, Y, Z: (-kp * torch.sin(kp * X) * torch.cos(kp * Y) * torch.cos(kp * Z),
                          -kp * torch.cos(kp * X) * torch.sin(kp * Y) * torch.cos(kp * Z),
                          -kp * torch.cos(kp * X) * torch.cos(kp * Y) * torch.sin(kp * Z))
    out = args.out or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                   "r03_fem_convergence_p%d.txt" % p)
    lines = ["# poms_b200.fem manufactured solution, 3-D p=%d, u = prod cos(pi x_a); card: %s" % (p, card),
             "# t_quad_to_coef_ms / t_quad_error_ms: CUDA-event intervals between the callables, host launch "
             "overhead included (dominant at N <= 128, one chunk each; kernel-dominated from N = 256)"]
    rows = []
    for N in [int(v) for v in args.N.split(",")]:
        h = Hierarchy(p, [N] * d, device=dev)
        lv = h.levels[0]
        b = lv.ws("b")
        for rep in range(2):                       # first pass warms up every shape
            tf = Timed(f)
            fem.load_vector(lv.V, lv.knots, p, tf, out=b)
            t_fl, t_q2c = tf.close()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            x, info = mg_pcg(h, b, tol=1e-12, maxiter=200)
            e1.record()
            torch.cuda.synchronize()
            t_solve = e0.elapsed_time(e1)
            tu = Timed(lambda X, Y, Z: u(X, Y, Z))
            tg = Timed(gu)
            err = fem.error_norms(x, lv.knots, p, tu, tg)
            t_ue, _ = tu.close()
            t_ge, _ = tg.close()
            # kernel interval: from the end of grad_u to the next u call (or the end)
            ends = [a for a, _ in tu.ev[1:]] + [None]
            t_err = 0.0
            last = torch.cuda.Event(enable_timing=True)
            last.record()
            torch.cuda.synchronize()
            for (_, b_), n in zip(tg.ev, ends):
                t_err += b_.elapsed_time(n if n is not None else last)
        E = N ** d
        ndof = (N + p) ** d
        by_q2c = 8.0 * (p + 1) ** d * E + 8.0 * ndof
        by_err = 8.0 * (p + 1) ** d * E * (1 + d) + 8.0 * ndof
        row = {"N": N, "dofs": ndof, "l2": err["l2"], "h1": err["h1"], "iters": info["niter"],
               "t_f_torch_ms": t_fl, "t_quad_to_coef_ms": t_q2c, "t_solve_ms": t_solve,
               "t_u_grad_torch_ms": t_ue + t_ge, "t_quad_error_ms": t_err,
               "q2c_GBps": by_q2c / t_q2c / 1e6, "err_GBps": by_err / t_err / 1e6}
        row["q2c_peak_share"] = row["q2c_GBps"] * 1e9 / PEAK
        row["err_peak_share"] = row["err_GBps"] * 1e9 / PEAK
        if rows:
            r0 = rows[-1]
            row["order_l2"] = float(np.log(r0["l2"] / row["l2"]) / np.log(N / r0["N"]))
            row["order_h1"] = float(np.log(r0["h1"] / row["h1"]) / np.log(N / r0["N"]))
        rows.append(row)
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)
        del h, lv, b, x
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("wrote", out)


if __name__ == "__main__":
    main()
