"""Builds libising_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

One object per translation unit, compiled in parallel and only when stale; the objects live in
csrc/_obj (git-ignored), the linked library next to this file so that it travels with the tree."""
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libising_b200.so")
SOURCES = ["sweep_rows3d.cu", "sweep_rows2d.cu", "sweep_stencil.cu", "sweep_cluster.cu", "sweep_general.cu", "sweep_field.cu", "moves.cu", "strip.cu", "strip_field.cu", "observables.cu", "state_io.cu",
           "api_core.cu", "api_sim.cu", "api_pt.cu", "api_comm.cu", "pt_device.cu", "api_strip.cu", "api_run.cu", "graph.cpp"]
HEADERS = ["kernels.h", "msc_device.cuh", "sweep_phase.cuh", "sweep_rows.cuh", "sweep_rows_launch.cuh", "api_internal.h", "graph.h", "philox.h", "pt_exp.h",
           os.path.join("..", "..", "include", "ising_b200.h")]
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC,-fvisibility=hidden"]


def _mtime(path):
    return os.path.getmtime(path) if os.path.exists(path) else 0.0


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def _compile(src, force, verbose):
    obj = os.path.join(OBJ, os.path.splitext(src)[0] + ".o")
    newest = max(_mtime(os.path.join(CSRC, f)) for f in [src] + HEADERS)
    if not force and _mtime(obj) >= newest:
        return obj, ""
    cmd = [_nvcc()] + FLAGS + (["-Xptxas=-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
    return obj, res.stderr


def build_native(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo ... -> libising_b200.so"""
    newest = max(_mtime(os.path.join(CSRC, f)) for f in SOURCES + HEADERS)
    if not force and _mtime(LIB) >= newest:
        return LIB          # up to date (e.g. the prebuilt library that travelled to the GPU box)
    os.makedirs(OBJ, exist_ok=True)
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
        done = list(pool.map(lambda s: _compile(s, force, verbose), SOURCES))
    objs = [o for o, _ in done]
    if verbose:
        print("".join(log for _, log in done))
    if force or _mtime(LIB) < max(_mtime(o) for o in objs):
        res = subprocess.run([_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs,
                             capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    import sys
    print(build_native(force=True, verbose="-v" in sys.argv))
