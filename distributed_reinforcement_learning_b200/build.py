"""In-tree build of the C-ABI library ``csrc/libdrl_b200.so`` with nvcc for sm_100a.

``python -m distributed_reinforcement_learning_b200.build`` (or ``__graft_entry__.build()``)
cross-compiles without a GPU.  The .so is git-ignored but travels with gpurun snapshots.
"""
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(CSRC, "libdrl_b200.so")
SOURCES = ["learner.cu", "layers.cu", "apex.cu", "r2d2.cu", "elementwise.cu", "vtrace.cu", "optimizer.cu", "ring.cu", "per.cu", "debug.cu",
           "peer.cu", "replay.cu"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _deps():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))) + \
        [os.path.join(HERE, "..", "include", "drl_b200.h")]


def _stamp():
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for p in _deps():
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile all CUDA sources for sm_100a and link the shared library.  Returns its path."""
    os.makedirs(OBJ, exist_ok=True)
    stamp_file = os.path.join(OBJ, "stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file):
        with open(stamp_file) as f:
            if f.read().strip() == stamp:
                return LIB
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        p = subprocess.run(cmd, capture_output=True, text=True)
        log = p.stdout + p.stderr
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + log)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, log))
        return obj, log

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        results = list(ex.map(compile_one, SOURCES))
    objs = [o for o, _ in results]
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lpthread"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("link failed:\n" + p.stdout + p.stderr)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
