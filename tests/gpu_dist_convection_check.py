"""Multi-GPU check of the convection term and mg_gmres (run under torchrun on the GPU box):
    timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29536 tests/gpu_dist_convection_check.py
The velocity component along axis 1 couples planes of neighbouring slabs in the non-symmetric mat-vec, and its
inflow / outflow faces are operator rows of rank 0 and of the last rank.  The slab-partitioned mg_gmres solve must
give the iteration count and the solution of the single-device solve of the same problem (which every rank also
runs, on its own GPU)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from poms_b200.dist import Slab
from poms_b200.mg import Hierarchy, mg_gmres
from poms_b200.stencil import StencilVector

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
slab = Slab(dist.group.WORLD, dev)
ok = True


def check(name, cond, info=""):
    global ok
    flag = torch.tensor([1 if cond else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("%-72s %s %s" % (name, "ok" if flag.item() else "FAIL", info))
    ok = ok and bool(flag.item())


CASES = [
    # (p, N, smoother, c, robin, beta): inflow face of axis 1 on rank 0 (beta_1 > 0) or on the last rank (< 0)
    (3, (32 * world, 16, 24), "glt", 1.0, [(5.0, 0.0), (0.0, 2.5), (1.5, 0.0)], (10.0, -5.0, 3.0)),
    (2, (32 * world, 24, 16), "glt_poly", 0.0, [(0.0, 10.0), (0.5, 0.0), (0.0, 0.0)], (-20.0, 0.0, 0.0)),
    (3, (64 * world, 32), "glt", 1.0, [(25.0, 0.0), (10.0, 0.0)], (50.0, 20.0)),
    (2, (64 * world, 40), "jacobi", 0.0, [(0.5, 1.0), (0.0, 2.0)], (1.0, -4.0)),
]
for p, N, smoother, c, robin, beta in CASES:
    d = len(N)
    rhs = np.random.default_rng(11).standard_normal([n + p for n in N])
    kw = dict(device=dev, smoother=smoother, c=c, robin=robin, beta=beta)
    h1 = Hierarchy(p, list(N), **kw)
    b1 = StencilVector.from_array(h1.levels[0].V, rhs)
    x1, i1 = mg_gmres(h1, b1, tol=1e-10, maxiter=600)
    ref = x1.data.cpu().numpy().copy()
    h = Hierarchy(p, list(N), slab=slab, min_planes=8, **kw)
    V = h.levels[0].V
    s, e = V.starts[0], V.ends[0]
    x, info = mg_gmres(h, StencilVector.from_array(V, rhs), tol=1e-10, maxiter=600)
    err = np.abs(x.data.cpu().numpy() - ref[s:e + 1]).max() / np.abs(ref).max()
    check("mg_gmres %dD p=%d %s c=%g beta=%s dist=%s" % (d, p, smoother, c, beta,
                                                        [int(l.distributed) for l in h.levels]),
          info["niter"] == i1["niter"] and info["success"] and i1["success"] and err < 1e-10,
          "iters %d vs %d, err %.1e" % (info["niter"], i1["niter"], err))
if rank == 0:
    print("ALL OK" if ok else "SOME FAILED")
dist.destroy_process_group()
sys.exit(0 if ok else 1)
