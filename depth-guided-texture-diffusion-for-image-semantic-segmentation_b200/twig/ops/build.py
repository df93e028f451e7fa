"""Build ``libdgtd_ops.so`` (the C-ABI CUDA extension, ``include/dgtd_ops.h``) in-tree.

The reference builds its ``twig/ops`` extension with ``make.sh`` -> ``setup.py`` ->
``CUDAExtension`` (twig/ops/make.sh, twig/ops/setup.py:47-55).  This library has no ATen or
pybind in it, so it is compiled with plain ``nvcc`` for sm_100a only:

    python -m dgtd_b200.twig.ops.build        (or ``bash twig/ops/make.sh``)

Objects go to ``csrc/build/``; the shared object lands next to this file so that it travels
with the source tree (it is git-ignored).
"""
from __future__ import annotations

import concurrent.futures as cf
import glob
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libdgtd_ops.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xptxas=-v",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3",
]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; libdgtd_ops.so cannot be built")
    return cand


def _digest(path: str) -> str:
    h = hashlib.sha1()
    for dep in sorted(glob.glob(os.path.join(CSRC, "*.cuh")) +
                      [os.path.join(os.path.dirname(PKG), "include", "dgtd_ops.h"), path]):
        with open(dep, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile(src: str, verbose: bool) -> str:
    obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
    stamp = obj + ".sha1"
    dig = _digest(src)
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
        return obj
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", src, "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
    if verbose:
        log = os.path.join(OBJ, os.path.basename(src)[:-3] + ".ptxas.log")
        with open(log, "w") as f:
            f.write(res.stderr)
    with open(stamp, "w") as f:
        f.write(dig)
    return obj


def build(force: bool = False, verbose: bool = True) -> str:
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in glob.glob(os.path.join(OBJ, "*")):
            os.remove(f)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    with cf.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), srcs))
    newest = max(os.path.getmtime(o) for o in objs)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < newest:
        cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-cudart", "shared"]  # share torch's libcudart.so.12
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
