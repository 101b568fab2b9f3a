"""Build libgantts_b200.so in-tree with nvcc for sm_100a (no GPU needed: cross-compiles)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "lib.cu")
OUT = os.path.join(HERE, "libgantts_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-I", os.path.join(os.path.dirname(HERE), "include")]


def sources():
    """The files the library is compiled from (not the .ptxas.log that build() writes next to them after linking)."""
    d = os.path.join(HERE, "csrc")
    inc = os.path.join(os.path.dirname(HERE), "include")
    return [os.path.join(p, f) for p in (d, inc) for f in os.listdir(p) if f.endswith((".cu", ".cuh", ".h"))]


def up_to_date():
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(s) <= t for s in sources())


def build(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    cmd = [NVCC] + FLAGS + ["-o", OUT, SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libgantts_b200.so (see stderr)")
    with open(os.path.join(HERE, "csrc", ".ptxas.log"), "w") as f:
        f.write(res.stdout + res.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
