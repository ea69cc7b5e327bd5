"""Builds libbrov.so (the sm_100a CUDA engine behind include/brov.h) in-tree with nvcc.

    python -m bluerov2_dynamics_b200.build [--force]

The translation units are compiled in parallel and linked into bluerov2_dynamics_b200/libbrov.so, which
travels to the GPU box with the repository snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
OUT = os.path.join(PKG, "libbrov.so")
BUILD = os.path.join(PKG, "build")
SOURCES = ["brov_api.cu", "brov_kernels_f32.cu", "brov_kernels_f64.cu", "brov_koopman.cu", "brov_pinc.cu", "brov_grad.cu",
           "brov_lin.cu", "brov_cl.cu", "brov_adj.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libbrov.so cannot be built")
    return exe


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    # every source and header of the library, whatever it is called (a header missing from a hand-kept list once let a
    # stale binary through)
    deps = glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) + \
        [os.path.join(PKG, "..", "include", "brov.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force: bool = False, verbose: bool = False, defines=(), out: str = OUT, tag: str = "") -> str:
    """defines/out/tag build a tuning variant next to the default library (see profiles/tune_variants.py)."""
    if not force and not defines and not _stale():
        return OUT
    os.makedirs(BUILD, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(BUILD, src.replace(".cu", tag + ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *[f"-D{d}" for d in defines], "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return out


if __name__ == "__main__":
    path = build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path, os.path.getsize(path), "bytes")
