"""Slab-partitioned mg_gmres with a convection term: runs tests/gpu_dist_convection_check.py under torchrun on every
GPU of the box (2, 4 or 8; skipped below 2).  The velocity along axis 1 couples the slabs in the non-symmetric
mat-vec; the script compares iteration counts and solutions with the single-device solve."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT


@pytest.mark.gpu
def test_slab_partitioned_convection_matches_single_device():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs (found %d)" % n)
    n = 8 if n >= 8 else 4 if n >= 4 else 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29536",
           os.path.join(ROOT, "tests", "gpu_dist_convection_check.py")]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    print(r.stdout[-6000:])
    assert r.returncode == 0, r.stdout[-3000:]
    assert "ALL OK" in r.stdout
