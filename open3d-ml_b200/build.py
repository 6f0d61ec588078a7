"""Builds libo3dml_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python open3d-ml_b200/build.py [--force]

The library has no torch dependency: it is a plain C ABI (include/o3dml_b200.h)
over CUDA kernels, statically linked against cudart.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(OUT_DIR, "libo3dml_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
DEBUG = (["-DO3DML_DEBUG_NAN"] if os.environ.get("O3DML_DEBUG_NAN") else []) + \
        (["-DO3DML_DEBUG_TIMING"] if os.environ.get("O3DML_DEBUG_TIMING") else [])
FLAGS = DEBUG + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr",
         "-ccbin", "/usr/bin/g++"]


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _newest_dep():
    inc = os.path.join(os.path.dirname(HERE), "include")
    t = max(os.path.getmtime(os.path.join(inc, f)) for f in os.listdir(inc))
    for f in os.listdir(CSRC):
        t = max(t, os.path.getmtime(os.path.join(CSRC, f)))
    return t


def build(force=False, verbose=False):
    """Compiles what is stale and links the library.  Safe to call from several processes at once (one rank per GPU
    under torch.distributed.run): an exclusive lock on lib/.build.lock serialises them and the late comers find the
    library fresh."""
    os.makedirs(OUT_DIR, exist_ok=True)
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_dep():
        return LIB
    import fcntl
    with open(os.path.join(OUT_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_dep():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
    objs = []

    def cc(src):
        obj = os.path.join(OUT_DIR, src[:-3] + ".o")
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(cc, sources()))
    tmp = LIB + ".tmp.%d" % os.getpid()      # linked aside and renamed: a concurrent freshness check never sees a partial file
    cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs + [
        "-cudart", "static", "-ccbin", "/usr/bin/g++",
                                                  "-Xlinker", "--no-undefined"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
