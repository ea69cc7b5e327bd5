#!/usr/bin/env python3
"""Builds oracle/_ref/: the UNMODIFIED reference, byte-compiled (sourceless byte code, *.refc), for the files of the hot path.

    python oracle/build_ref.py            (or: make -C oracle ref; __graft_entry__.build() runs it when it can)

The reference is pure Python; "building" it is `py_compile` from the sources where they lie under /root/reference
into oracle/_ref/ — no reference source text enters this repository, oracle/_ref/ is git-ignored (it is NOT
gpurun-ignored: like the built libbrov.so it travels to the GPU box, where /root/reference does not exist, and lets
`bench.py --impl reference` and the parity tests execute the reference itself: fossen.BlueROV2.BlueROV2.dynamics and
training/train_tank_brov2_rk4.py's simulate_physics / multistep_rmse_endpoint_physics).
TEST / BASELINE INFRASTRUCTURE: only tests/, __graft_entry__ and bench.py's CPU legs use it (through oracle/ref_loader.py).
"""
import os
import py_compile
import shutil
import sys

REF = os.environ.get("BROV_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
FILES = ["fossen/__init__.py", "fossen/BlueROV2.py", "fossen/BlueROV2_thrust.py", "fossen/BlueROV2_wrench.py",
         "fossen/bluerov_torch.py", "fossen/parameters.py", "Koopman/__init__.py", "Koopman/koopmanEDMDc.py",
         "training/train_tank_brov2_rk4.py", "training/train_tank_brov2_full_comparison.py"]


def build() -> bool:
    if not os.path.isdir(REF):
        # no copy of the reference here: nothing to build, which is not an error (the live-reference tests skip)
        print(f"[build_ref] {REF} not present: keeping whatever oracle/_ref holds")
        return True
    shutil.rmtree(OUT, ignore_errors=True)
    for rel in FILES:
        src = os.path.join(REF, rel)
        dst = os.path.join(OUT, rel[:-3] + ".refc")   # byte code; not named .pyc: snapshot tools tend to skip those
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        py_compile.compile(src, cfile=dst, dfile=src, doraise=True, optimize=0)
    with open(os.path.join(OUT, "BUILT_FROM.txt"), "w") as f:
        f.write(f"py_compile of {REF} ({len(FILES)} files) with Python {sys.version.split()[0]}\n" + "\n".join(FILES) + "\n")
    print(f"[build_ref] {len(FILES)} files -> {OUT}")
    return True


if __name__ == "__main__":
    sys.exit(0 if build() else 1)
