"""Build libsuperbblas_b200.so (CUDA kernels + host planner + C ABI) for sm_100a, in tree.

    python -m superbblas_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so lands in superbblas_b200/lib/ (git-ignored; it travels
to the GPU box with the working tree).
"""
import concurrent.futures
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "lib")
LIB = os.path.join(OUT, "libsuperbblas_b200.so")
SOURCES = ["geometry.cpp", "plan.cpp", "driver.cpp", "contract_plan.cpp", "dense_plan.cpp", "bsr_plan.cpp", "runtime.cpp", "capi.cpp",
           "kernels_copy.cu", "kernels_contract.cu", "kernels_contract_tc.cu", "kernels_dense.cu",
           "kernels_bsr.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++"]


def source_hash():
    """sha1 of everything the library is built from; compiled into the .so (sbb_source_hash) so that a
    stale binary is detected when it is loaded, whatever the file times or a stamp file say."""
    h = hashlib.sha1()
    for f in sorted(os.listdir(SRC)) + ["../../include/superbblas_b200.h"]:
        with open(os.path.join(SRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def embedded_hash(path=None):
    """The source hash compiled into an existing library (None if it cannot be read)."""
    import ctypes
    try:
        lib = ctypes.CDLL(path or LIB)
        lib.sbb_source_hash.restype = ctypes.c_char_p
        return lib.sbb_source_hash().decode()
    except (OSError, AttributeError):
        return None


def _compile(src):
    obj = os.path.join(OUT, src + ".o")
    cmd = [NVCC] + FLAGS + ["-c", os.path.join(SRC, src), "-o", obj]
    if src == "capi.cpp":
        cmd.append('-DSBB_SOURCE_HASH="%s"' % source_hash())
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    return obj


def build(force=False, verbose=True):
    os.makedirs(OUT, exist_ok=True)
    if not force and os.path.exists(LIB) and embedded_hash() == source_hash():
        return LIB
    if verbose:
        print("[superbblas_b200] compiling for sm_100a ...", file=sys.stderr)
    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(_compile, SOURCES))
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-ccbin", "/usr/bin/g++", "-lpthread", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
