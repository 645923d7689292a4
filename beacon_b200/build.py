"""Build libbeacon_b200.so (hand-written sm_100a CUDA + the C-ABI) in-tree with nvcc.

    python -m beacon_b200.build [--force]

nvcc cross-compiles without a GPU.  The resulting .so is git-ignored but travels to the GPU box
with the repo snapshot.
"""
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libbeacon_b200.so")
SOURCES = ["capi.cu", "shkadov.cu", "burgers.cu", "sloshing.cu", "ode.cu", "mac2d.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "mac_reg_kernel.cuh"), os.path.join(HERE, "..", "include", "beacon_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr",
]


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libbeacon_b200.so cannot be built")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, tag=None, defines=()):
    """tag / defines: A/B variants for tuning (tools/ab.sh): objects in lib/obj_<tag>/, library lib/libbeacon_b200_<tag>.so,
    extra -D flags; the product build has neither."""
    objdir = os.path.join(LIBDIR, "obj" + (f"_{tag}" if tag else ""))
    LIB = os.path.join(LIBDIR, "libbeacon_b200" + (f"_{tag}" if tag else "") + ".so")
    os.makedirs(objdir, exist_ok=True)
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + HEADERS):
            jobs.append([nvcc()] + NVCC_FLAGS + list(defines) + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            for cmd, res in zip(jobs, ex.map(lambda c: subprocess.run(c, capture_output=True, text=True), jobs)):
                if verbose and res.stderr:
                    print(res.stderr, file=sys.stderr)
                if res.returncode != 0:
                    raise RuntimeError("nvcc failed: %s\n%s" % (" ".join(cmd), res.stderr))
    if jobs or force or _stale(LIB, objs):
        cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed: %s\n%s" % (" ".join(cmd), res.stderr))
    census = os.path.join(LIBDIR, "sass_census.json")
    tool = os.path.join(HERE, "..", "tools", "sass_census.py")
    if not tag and (jobs or force or _stale(census, objs + [tool])):
        # static SASS census of the hot loops (fp64 / shared-memory instructions per sub-step and per Jacobi sweep):
        # bench.py turns it into the in-run roofline fraction
        res = subprocess.run([sys.executable, tool, census], capture_output=True, text=True)
        if res.returncode != 0:
            print("sass census failed (bench.py will report the S-model only):\n" + res.stderr[-2000:], file=sys.stderr)
    return LIB


if __name__ == "__main__":
    tag = next((a.split("=", 1)[1] for a in sys.argv if a.startswith("--tag=")), None)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, tag=tag, defines=[a for a in sys.argv if a.startswith("-D")]))
