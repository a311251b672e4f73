"""In-tree build of libsparsifyme_b200.so (nvcc, sm_100a only).

The library is the product: hand-written CUDA behind the C ABI of include/spfy_b200.h.
It is built IN-TREE (sparsify.me_b200/lib/) so that the .so travels with the repo
snapshot to the GPU box; nothing is JIT-compiled at import time.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libsparsifyme_b200.so")
SOURCES = ["api.cu", "prune.cu", "transpose24.cu", "spmma_sm100.cu", "gemm_sm100.cu", "spmm.cu", "multigpu.cu", "optim24.cu"]
NVCC_FLAGS = [
    "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libsparsifyme_b200.so cannot be built")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, dev=False):
    """Compile every .cu under csrc/ for sm_100a and link the shared library.
    dev=True builds lib_dev/libsparsifyme_b200.so (objects in build_dev/) next to the release library: the same
    code with the SPFY_* environment switches compiled in; select it with SPFY_LIB=<path> (tuning runs only)."""
    global OBJ, LIBDIR, LIB
    if dev:
        OBJ, LIBDIR = os.path.join(HERE, "build_dev"), os.path.join(HERE, "lib_dev")
        LIB = os.path.join(LIBDIR, "libsparsifyme_b200.so")
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "spfy_b200.h"))
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = ([nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) +
                   (["-DSPFY_DEV_SWITCHES"] if dev else []) + ["-c", s, "-o", o])
            subprocess.run(cmd, check=True)
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                    "-cudart", "static", "-ldl"]
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    # --dev: compile the SPFY_* environment switches in (tuning / timing experiments only, see common.cuh)
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv, dev="--dev" in sys.argv))
