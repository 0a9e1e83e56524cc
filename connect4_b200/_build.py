"""Build libc4b200.so (the C-ABI CUDA library, include/c4b200.h) in-tree for sm_100a with nvcc."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libc4b200.so")
SOURCES = ["c4_board.cu", "c4_search.cu", "c4_net.cu", "c4_layers.cu", "c4_fused.cu", "c4_split.cu"]
HEADERS = ["c4_common.cuh", "c4_tree.cuh", "c4_tc.cuh", "c4_fz.cuh", "c4_layers.cuh", os.path.join("..", "..", "include", "c4b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library. Returns its path."""
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(LIBDIR, s.replace(".cu", ".o"))
        extra = os.environ.get("C4_NVCC_EXTRA", "").split()       # e.g. -DC4_TC_PROFILE for per-role cycle accounting
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(out.decode())
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
