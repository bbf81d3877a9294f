"""Builds libcuba_b200.so (sm_100a only) in-tree with nvcc.  Used by __graft_entry__.build()."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcuba_b200.so")
SOURCES = ["cuba_engine.cu", "cuba_structure.cpp", "cuba_api.cpp"]
HEADERS = ["cuba_kernels.cuh", "cuba_jh4.cuh", "cuba_schur3.cuh", "cuba_pcg2.cuh", "cuba_pcg3.cuh", "cuba_pcg4.cuh", "cuba_pcg5.cuh", "cuba_pcg5t.cuh", "cuba_coarse_dense.cuh", "cuba_peer_reduce.cuh", "cuba_structure_gpu.cuh", "cuba_math.cuh", "cuba_structure.h",
           "../../include/cuba_b200.h", "../../include/cuda_bundle_adjustment.h", "../../include/cuda_bundle_adjustment_types.h"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = (["-DCUBA_JH4_DEBUG"] if os.environ.get("CUBA_JH4_DEBUG") else []) + ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function", "-shared"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-I", os.path.join(HERE, "..", "include"), "-o", LIB] + srcs + ["-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force=True, verbose="-v" in sys.argv))
