"""CPU-side tests of the closed-loop gradients (no GPU): the C descriptor of brov_closed_loop_vjp and its ctypes mirror
agree, the entry points are exported with the ABI unchanged, and the workspace size is n * (steps * (2 NZ + 2 NU) +
NU * NZ) doubles, 0 for the double-integrator models and empty calls, SIZE_MAX when it does not fit in size_t."""
import ctypes as C
import os
import subprocess

import pytest

from conftest import ROOT


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200.build import build_lib
    build_lib()
    from bluerov2_dynamics_b200 import _lib
    return _lib


def test_closed_loop_vjp_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.ClosedLoopVjpDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_closed_loop_vjp_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_closed_loop_vjp_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct)
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname


def test_closed_loop_vjp_symbols_are_exported(L):
    out = subprocess.run(["nm", "-D", "--defined-only", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = {line.split()[-1] for line in out.splitlines() if line.strip()}
    for s in ("brov_closed_loop_vjp", "brov_closed_loop_vjp_workspace_bytes"):
        assert s in names and s in L._PROTOS
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8


@pytest.mark.parametrize("model,nz,nu", [(0, 30, 8), (1, 12, 6), (2, 13, 6)])
def test_workspace_bytes(L, model, nz, nu):
    f = L.lib.brov_closed_loop_vjp_workspace_bytes
    for n, T in ((1, 1), (7, 13), (65536, 1000)):
        assert f(model, n, T) == n * (T * (2 * nz + 2 * nu) + nu * nz) * 8
    assert f(model, 0, 10) == 0 and f(model, 10, 0) == 0 and f(model, -1, 10) == 0
    size_max = C.c_size_t(-1).value
    n, T = 2 ** 20, 2 ** 30                                      # 2^50 * (steps' and scratch doubles) fits ...
    assert f(model, n, T) == n * (T * (2 * nz + 2 * nu) + nu * nz) * 8 < size_max
    assert f(model, 2 ** 31 - 1, 2 ** 30) == size_max            # ... 2^61 * 2^9 bytes does not
    for di in (3, 4, 5):
        assert f(di, 10, 10) == 0
