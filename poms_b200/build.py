"""Build libpoms_b200.so in-tree with nvcc for sm_100a (no torch headers: pure C ABI).

The one source file is compiled as several translation units (-DPOMS_TU=k, see the top of
csrc/poms_kernels.cu) in parallel, then linked; objects go to build/ (git-ignored)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SRC = os.path.join(CSRC, "poms_kernels.cu")
EXTRA_SRC = [os.path.join(CSRC, "poms_extra.cu"), os.path.join(CSRC, "poms_setup.cu"),
             os.path.join(CSRC, "poms_transfer3d_v2.cu"),
             os.path.join(CSRC, "poms_fem3d.cu")]              # self-contained units (own kernels + C ABI)
OUT = os.path.join(HERE, "libpoms_b200.so")
OBJDIR = os.path.join(ROOT, "build", "obj")
TUS = [0, 1, 2, 3, 4, 5, 6, 7]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-diag-suppress", "177,550",
]


def _deps():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(ROOT, "include", "poms_b200.h")]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in _deps() if os.path.exists(d))


def _compile(job):
    src, obj, defs, verbose = job
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + defs + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    print("[poms_b200.build]", " ".join(cmd[-6:]), file=sys.stderr)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.returncode, r.stdout


def build(force=False, verbose=False, only=None):
    """only: list of TU ids to recompile (kernel development); the others reuse their objects."""
    if not force and only is None and not needs_build():
        return OUT
    os.makedirs(OBJDIR, exist_ok=True)
    jobs, objs = [], []
    # heaviest units first
    for k in sorted(TUS, key=lambda k: -k):
        obj = os.path.join(OBJDIR, "poms_tu%d.o" % k)
        objs.append(obj)
        if only is None or k in only or not os.path.exists(obj):
            jobs.append((SRC, obj, ["-DPOMS_TU=%d" % k], verbose))
    for i, src in enumerate(EXTRA_SRC):
        if not os.path.exists(src):
            continue
        obj = os.path.join(OBJDIR, "poms_extra%d.o" % i)
        objs.append(obj)
        if only is None or ("x%d" % i) in only or not os.path.exists(obj):
            jobs.append((src, obj, [], verbose))
    nproc = max(1, min(len(jobs), os.cpu_count() or 1))
    with ThreadPoolExecutor(nproc) as ex:
        for rc, out in ex.map(_compile, jobs):
            if out.strip() and (rc != 0 or verbose):
                print(out, file=sys.stderr)
            if rc != 0:
                raise subprocess.CalledProcessError(rc, "nvcc")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs + ["-o", OUT]
    print("[poms_b200.build] link", OUT, file=sys.stderr)
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    only = None
    for a in sys.argv[1:]:
        if a.startswith("--only="):
            only = [int(t) if t.isdigit() else t for t in a[7:].split(",")]
    build(force="--force" in sys.argv, verbose="-v" in sys.argv, only=only)
