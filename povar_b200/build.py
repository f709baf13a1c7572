"""In-tree build of libpovar_b200.so and the `bal` front end with nvcc for sm_100a.

    python -m povar_b200.build [--force] [--verbose]

The built files (povar_b200/lib/libpovar_b200.so, povar_b200/bin/bal) are git-ignored but travel
with gpurun snapshots.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(ROOT, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(ROOT, "lib", "libpovar_b200.so")
BAL = os.path.join(ROOT, "bin", "bal")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall",
          "-Xcompiler", "-Wno-unused-function"]

LIB_SOURCES = [
    "kernels_landmark.cu",
    "kernels_camera.cu",
    "kernels_schur.cu",
    "kernels_chol.cu",
    "kernels_series.cu",
    "kernels_index.cu",
    "kernels_lm.cu",
    "engine.cu",
    "capi.cpp",
    "host/bal_io.cpp",
    "host/ba_log_writer.cpp",
    "host/lm_driver.cpp",
    "host/chol_symbolic.cpp",
]
HEADERS = ["device_math.cuh", "sell_walk.cuh", "povar_internal.h", "engine.h", "lm_step.h", "../../include/povar_b200.h"]
# the LM decision kernels compute what the host driver computes: no contracted multiply-adds (lm_step.h)
EXTRA_FLAGS = {"kernels_lm.cu": ["-fmad=false"]}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libpovar_b200.so cannot be built (there is no CPU fallback)")


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps if os.path.exists(d))


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("build step failed: " + " ".join(cmd))
    if verbose and (res.stdout or res.stderr):
        print(res.stdout + res.stderr)
    return res


def build(force: bool = False, verbose: bool = False, defines=(), suffix: str = "") -> str:
    """`defines` / `suffix`: tuning builds (-D... into lib/libpovar_b200<suffix>.so, selected with POVAR_LIB)."""
    nvcc = _nvcc()
    if suffix:
        return _build_variant(nvcc, list(defines), suffix, verbose)
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    os.makedirs(os.path.dirname(BAL), exist_ok=True)
    headers = [os.path.join(CSRC, h) for h in HEADERS]
    sources = [s for s in LIB_SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src):
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ, src.replace("/", "_") + ".o")
        if not force and _newer(obj, [path] + headers):
            return obj
        cmd = [nvcc] + ARCH + COMMON + EXTRA_FLAGS.get(src, []) + ["-x", "cu", "-Xptxas",
                                                                   "-v" if verbose else "-warn-spills",
                                                                   "-c", path, "-o", obj]
        _run(cmd, verbose)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        objs = list(ex.map(compile_one, sources))

    if force or not _newer(LIB, objs):
        _run([nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-ldl"], verbose)
    main_src = os.path.join(CSRC, "host", "bal_main.cpp")
    if force or not _newer(BAL, [main_src, LIB] + headers):
        _run([nvcc] + ARCH + COMMON + ["-x", "cu", main_src, "-o", BAL, "-L" + os.path.dirname(LIB),
                                      "-lpovar_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN/../lib"],
             verbose)
    return LIB


def _build_variant(nvcc, defines, suffix, verbose):
    obj_dir = OBJ + suffix
    os.makedirs(obj_dir, exist_ok=True)
    lib = LIB.replace(".so", suffix + ".so")
    sources = [s for s in LIB_SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src):
        obj = os.path.join(obj_dir, src.replace("/", "_") + ".o")
        _run([nvcc] + ARCH + COMMON + EXTRA_FLAGS.get(src, []) + ["-D" + d for d in defines] +
             ["-x", "cu", "-Xptxas", "-warn-spills", "-c",
                                                                    os.path.join(CSRC, src), "-o", obj], verbose)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        objs = list(ex.map(compile_one, sources))
    _run([nvcc] + ARCH + ["-shared", "-o", lib] + objs + ["-ldl"], verbose)
    return lib


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
