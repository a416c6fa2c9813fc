"""Compile the CUDA sources into ``<package>/liboctm.so`` for sm_100a (in-tree, no JIT cache).

    python -m retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build [--force]

nvcc cross-compiles without a GPU.  The runtime is linked statically so the library only needs the
driver; torch's own cudart shares the primary context, so torch streams and allocations are valid
arguments.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.path.join(PKG, "liboctm.so")
SOURCES = ["common.cu", "label_pass.cu", "contour.cu", "contour_all.cu", "contour_spacing.cu", "surface_dice.cu", "components.cu", "derive.cu", "argmax.cu", "auc.cu", "boundary.cu", "edt3d.cu", "hostpack.cu", "rasterise.cu"]
HEADERS = ["common.cuh", "crack_masks.cuh", "trace_core.h", os.path.join("..", "..", "include", "octm.h")]
NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--fmad=false",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Build liboctm.so if missing or older than its sources; returns its path."""
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        extra = os.environ.get("OCTM_NVCC_EXTRA", "").split()       # debug builds, e.g. -DOCTM_WALK_STATS
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", os.path.join(HERE, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = LIB + ".tmp"
    r = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp, *objs,
                        "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
