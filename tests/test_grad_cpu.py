"""CPU-side tests of the coefficient gradient (no GPU): the C descriptor and its ctypes mirror agree, the workspace
does not grow with the series beyond the carried lag, and coefficient_directions is the Jacobian of
derive_params(with_minv(.)) in the selected physical parameters."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200.build import build_lib
    build_lib()
    from bluerov2_dynamics_b200 import _lib
    return _lib


def test_grad_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.SeGradDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_se_grad_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_se_grad_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct) == 4 + 4 + 8 * 3 + 8 * 3 + 4 + 4 * 4 + 4 + 8 * 3 + 4 + 4 + 8 * 6 + 8 * 3
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8


def test_grad_workspace_bytes(L):
    """Per-block partials of a fixed grid (1024 blocks x 4 horizons x (1 + p + p(p+1)/2) doubles), independent of the
    number of windows, plus the carried-lag rows [n_windows][18] in carry mode; p outside 1..36 needs nothing."""
    f = L.lib.brov_se_grad_workspace_bytes
    part = lambda p: 1024 * 4 * (1 + p + p * (p + 1) // 2) * 8
    assert f(1000, 18, 0) == f(10 ** 6, 18, 0) == part(18)
    assert f(1000, 36, 1) == part(36) + ((1000 * 18 * 8 + 255) // 256) * 256
    assert f(1000, 0, 0) == 0 and f(1000, 37, 0) == 0


def _fd_directions(phys, idx, rebuild):
    from bluerov2_dynamics_b200.engine import derive_params, with_minv
    f = (lambda q: derive_params(with_minv(q))) if rebuild else derive_params
    out = []
    for i in idx:
        h = 1e-6 * max(abs(phys[i]), 1.0)
        d = []
        for s in (h, -h, 2 * h, -2 * h):
            q = phys.copy()
            q[i] += s
            d.append(f(q))
        out.append((8 * (d[0] - d[1]) - (d[2] - d[3])) / (12 * h))
    return np.array(out)


@pytest.mark.parametrize("rebuild", [True, False])
def test_coefficient_directions_match_differences(L, rebuild):
    from bluerov2_dynamics_b200.engine import (PHYS_NAMES, coefficient_directions, default_physical,
                                                parameter_indices)
    rng = np.random.default_rng(3)
    ph = default_physical()
    ph[L.PH_ADDED:L.PH_ADDED + 6] *= rng.uniform(0.7, 1.3, 6)
    ph[L.PH_XB:L.PH_XB + 3] = rng.uniform(-0.02, 0.02, 3)
    ph[L.PH_CURRENT:L.PH_CURRENT + 3] = rng.uniform(-0.1, 0.1, 3)
    params = ["m", "W", "B", "xb", "yb", "zb", "Ix", "Iy", "Iz", "added", "lin", "quad", "current"]
    if not rebuild:
        params += [f"Minv_{a}" for a in "uvwpqr"]
    idx = parameter_indices(params)
    assert len(idx) == (36 if not rebuild else 30) and [PHYS_NAMES[i] for i in idx][:3] == ["m", "W", "B"]
    D = coefficient_directions(ph, params, rebuild_minv=rebuild)
    ref = _fd_directions(ph, idx, rebuild)
    assert D.shape == (len(idx), L.NKP)
    assert np.max(np.abs(D - ref)) <= 1e-9 * max(1.0, np.max(np.abs(ref)))
    # the Minv entries follow the masses only when they are rebuilt
    row_m = D[idx.index(L.PH_M)]
    assert np.any(row_m[0:3] != 0.0) == rebuild and np.all(row_m[3:6] == 0.0)


def test_parameter_selection_is_checked(L):
    from bluerov2_dynamics_b200.engine import coefficient_directions, default_physical, parameter_indices
    assert parameter_indices(["added", "Xu", L.PH_B]) == list(range(9, 15)) + [15, 2]
    assert parameter_indices("quad") == list(range(21, 27))
    for bad in (["Xu_dott"], [L.PH_TLAG1], ["T_lag1"], [37], [-1], ["Xu", "Xu"], []):
        with pytest.raises(ValueError):
            parameter_indices(bad)
    with pytest.raises(ValueError, match="rebuild_minv"):
        coefficient_directions(default_physical(), ["Minv_u"], rebuild_minv=True)
