"""Build libtuna_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "tuna_b200.cu")
DEPS = [SRC, os.path.join(HERE, "csrc", "devbuf.hpp"), os.path.join(HERE, "csrc", "eri_core.cuh"), os.path.join(HERE, "csrc", "pairtable.hpp"),
        os.path.join(HERE, "csrc", "shell_jk.cuh"), os.path.join(HERE, "csrc", "shell_host.hpp"), os.path.join(HERE, "csrc", "shell4.cuh"), os.path.join(HERE, "csrc", "shell4_host.hpp"), os.path.join(HERE, "csrc", "mo_transform.cuh"), os.path.join(HERE, "csrc", "oneel_core.cuh"), os.path.join(os.path.dirname(HERE), "include", "tuna_b200.h")]
OUT = os.environ.get("TUNA_B200_LIB") or os.path.join(HERE, "libtuna_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC,-fopenmp,-O2", "-shared", "-lgomp"]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if force or needs_build():
        extra = os.environ.get("TUNA_B200_NVCC_EXTRA", "").split()
        cmd = [NVCC] + FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT, SRC]
        subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
