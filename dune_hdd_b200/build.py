"""Builds dune_hdd_b200/libhdd_b200.so in-tree with nvcc for sm_100a (no JIT cache, the .so travels with the repo)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libhdd_b200.so")
SOURCES = ["mesh.cu", "swipdg.cu", "products.cu", "kernels_assembly.cu", "kernels_cg.cu", "kernels_estimators.cu",
           "kernels_products.cu", "multigrid.cu", "expr.cpp",
           "grids.cpp", "partition.cpp"]
HEADERS = ["common.hpp", "expr.hpp", "quadrature.hpp", "device.cuh", "reduce.cuh", "kernels.hpp", "handles.hpp",
           "partition.hpp",
           os.path.join("..", "..", "include", "hdd_b200.h"), os.path.join("..", "..", "include", "hdd_b200_testing.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
         "-Xcompiler", "-fPIC,-Wall,-Wno-unknown-pragmas", "-x", "cu"]


def _stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return SO
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src + ".o")
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([NVCC, "-shared", "-o", SO] + objs + ["-lcudart", "-ldl"])
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
