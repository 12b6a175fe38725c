"""Build libloma_nerf_b200.so in-tree with nvcc for sm_100a (B200).

    python -m loma_nerf_b200.build [--force] [--verbose]

The library is the product: hand-written CUDA kernels + the C ABI of include/loma_nerf_b200.h.
nvcc cross-compiles without a GPU; the built .so is git-ignored but travels with the tree.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libloma_nerf_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CFLAGS = (["-DLNB_TC_CLK"] if os.environ.get("LNB_TC_CLK") else []) + (["-DLNB_WIDE_CLK"] if os.environ.get("LNB_WIDE_CLK") else []) + ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=hidden",
          "--expt-relaxed-constexpr", "-I", INCLUDE]


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest():
    h = hashlib.sha256()
    files = sources() + [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".h", ".cuh", ".inc"))]
    files += [os.path.join(INCLUDE, f) for f in sorted(os.listdir(INCLUDE))]
    for p in files:
        h.update(p.encode())
        with open(p, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(ARCH + CFLAGS).encode())
    return h.hexdigest()


def build_library(force=False, verbose=False):
    """Compile every csrc/*.cu for sm_100a and link the shared library. Returns its path."""
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB

    def compile_one(src):
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
        cmd = [NVCC] + ARCH + CFLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(sources()))) as ex:
        objs = list(ex.map(compile_one, sources()))
    cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart_static", "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(stamp, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
