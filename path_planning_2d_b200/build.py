"""Build the sm_100a shared library (libpp2d.so) in-tree with nvcc.

The product is the C-ABI library declared in include/pp2d.h; this script is
what `__graft_entry__.build()` calls.  nvcc cross-compiles for sm_100a without
a GPU, so it also runs in the CPU-only build container.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpp2d.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SOURCES = ["mdp.cu", "pomdp.cu", "pbvi.cu", "sim.cu", "rollout.cu"]
FLAGS = [
    "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fopenmp", "-shared",
    "-I", os.path.join(ROOT, "include"),
]


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC)
                   if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(ROOT, "include", "pp2d.h"))
    if (not force and os.path.exists(LIB)
            and os.path.getmtime(LIB) >= _newest(deps)):
        return LIB
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
        ["-o", LIB] + srcs + ["-ldl", "-lgomp"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libpp2d.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
