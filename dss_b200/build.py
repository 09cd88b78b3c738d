"""Build libdss_b200.so (hand-written sm_100a CUDA behind the C ABI of include/dss_b200.h).

    python -m dss_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so is built in-tree (dss_b200/lib/) so it travels to the GPU
box with the repo snapshot.  No torch headers are involved: the ABI is plain C.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libdss_b200.so")
SOURCES = ["ctx.cu", "binning.cu", "raster_fwd.cu", "backward.cu", "occ_backward.cu", "knn.cu", "render.cu", "loss.cu"]
HEADERS = ["common.cuh", "kernels.cuh", os.path.join("..", "..", "include", "dss_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not (force or _stale()):
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(LIBDIR, s.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(" ".join(cmd))
            print(out)
        if p.returncode:
            raise RuntimeError("nvcc failed for " + cmd[-3])
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
