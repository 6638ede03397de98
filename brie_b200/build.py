"""In-tree build of libbrie_b200.so for sm_100a (`python -m brie_b200.build`).

Each translation unit under csrc/ is compiled to build/<name>.o (in parallel, only when
stale) and the objects are linked into brie_b200/libbrie_b200.so.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
UNITS = ["brie_abi.cu", "brie_ingest.cu", "brie_comm.cu"]
HEADERS = [os.path.join(_CSRC, h) for h in ("brie_kernels.cuh", "brie_margin.cuh", "brie_wald.cuh", "brie_philox.h", "brie_host.h")] + \
    [os.path.join(os.path.dirname(_HERE), "include", "brie_b200.h")]
OBJ_DIR = os.path.join(_HERE, "build")
OUT = os.path.join(_HERE, "libbrie_b200.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(p) > t for p in deps)


def up_to_date():
    srcs = [os.path.join(_CSRC, u) for u in UNITS]
    return not _stale(OUT, srcs + HEADERS)


def build(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ_DIR, exist_ok=True)

    def compile_unit(u):
        src = os.path.join(_CSRC, u)
        obj = os.path.join(OBJ_DIR, u.replace(".cu", ".o"))
        if force or _stale(obj, [src] + HEADERS):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            subprocess.run(cmd, check=True)
        return obj

    with ThreadPoolExecutor(len(UNITS)) as ex:
        objs = list(ex.map(compile_unit, UNITS))
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT] + objs + ["-ldl", "-lcublas"], check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
