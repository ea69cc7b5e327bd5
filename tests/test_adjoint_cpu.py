"""CPU-side tests of the reverse-mode rollout gradients (no GPU): the C descriptor of brov_rollout_vjp and its ctypes
mirror agree, the entry points are exported with the ABI unchanged, and the workspace size follows n * steps * NZ."""
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


def test_rollout_vjp_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.RolloutVjpDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_rollout_vjp_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_rollout_vjp_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct) == 4 + 4 + 8 * 3 + 8 * 2 + 8 * 2 + 8 * 2 + 8 * 5 + 8 + 8 + 8
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname


def test_rollout_vjp_symbols_are_exported(L):
    out = subprocess.run(["nm", "-D", "--defined-only", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = {line.split()[-1] for line in out.splitlines() if line.strip()}
    for sym in ("brov_rollout_vjp", "brov_rollout_vjp_workspace_bytes"):
        assert sym in names and sym in L._PROTOS
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8


def test_workspace_bytes(L):
    ws = L.lib.brov_rollout_vjp_workspace_bytes
    assert ws(L.THRUSTER8_LAG3, 65536, 1000) == 65536 * 1000 * 30 * 8
    assert ws(L.WRENCH_EULER12, 37, 60) == 37 * 60 * 12 * 8
    assert ws(L.WRENCH_QUAT13, 37, 60) == 37 * 60 * 13 * 8
    assert ws(L.WRENCH_EULER12, 1 << 21, 180) == (1 << 21) * 180 * 12 * 8 > 2 ** 31
    assert ws(L.WRENCH_EULER12, 0, 60) == 0 and ws(L.WRENCH_EULER12, 5, 0) == 0
    for m in (L.DI_EULER12_U8, L.DI_EULER12_U6, L.DI_QUAT13_U6, 99):
        assert ws(m, 10, 10) == 0
    assert ws(L.THRUSTER8_LAG3, 1 << 40, 1 << 30) == 2 ** 64 - 1   # does not fit in size_t
