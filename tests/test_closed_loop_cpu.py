"""CPU-side tests of the closed-loop rollout (no GPU): the C descriptor of brov_closed_loop and its ctypes mirror
agree, and the entry point is exported with the ABI unchanged."""
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


def test_closed_loop_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.ClosedLoopDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_closed_loop_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_closed_loop_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    # 4 + 4, n / steps / dt, z0 / z_out, three operands with two strides, bounds 2 x 8, weights 30 + 8,
    # traj / u_traj / stride, cost + flag + reserved, health, singular_eps
    assert int(got["size"]) == C.sizeof(ct) == 8 + 24 + 16 + 3 * 24 + 16 * 8 + 38 * 8 + 24 + 16 + 8 + 8
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname


def test_closed_loop_symbol_is_exported(L):
    out = subprocess.run(["nm", "-D", "--defined-only", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert any(line.split()[-1] == "brov_closed_loop" for line in out.splitlines() if line.strip())
    assert "brov_closed_loop" in L._PROTOS
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8
