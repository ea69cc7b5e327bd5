"""CPU-side tests of the coefficient gradients of batched rollouts (no GPU): the C descriptor of brov_rollout_vjp_coef
and its ctypes mirror agree, the entry point is exported with the ABI unchanged, and derive_params_torch equals
derive_params (with and without with_minv) with coefficient_directions as its autograd Jacobian."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200.build import build_lib
    build_lib()
    from bluerov2_dynamics_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def E(L):
    from bluerov2_dynamics_b200 import engine
    return engine


def test_rollout_vjp_coef_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.RolloutVjpCoefDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_rollout_vjp_coef_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_rollout_vjp_coef_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct) == 8 + C.sizeof(L.RolloutVjpDesc) + 8
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname


def test_rollout_vjp_coef_symbol_is_exported(L):
    out = subprocess.run(["nm", "-D", "--defined-only", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = {line.split()[-1] for line in out.splitlines() if line.strip()}
    assert "brov_rollout_vjp_coef" in names and "brov_rollout_vjp_coef" in L._PROTOS
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8


def _vehicles(E, L, k, seed):
    rng = np.random.default_rng(seed)
    ph = np.tile(E.default_physical(), (k, 1))
    ph *= rng.uniform(0.7, 1.3, ph.shape)
    ph[:, L.PH_CURRENT:L.PH_CURRENT + 3] = rng.uniform(-0.2, 0.2, (k, 3))
    ph[: k // 2, L.PH_TLAG1] = 0.0
    return ph


@pytest.mark.parametrize("rebuild_minv", [True, False])
def test_derive_params_torch_equals_derive_params(E, L, rebuild_minv):
    ph = _vehicles(E, L, 16, 3)
    ref = E.derive_params(E.with_minv(ph) if rebuild_minv else ph)
    got = E.derive_params_torch(torch.from_numpy(ph), rebuild_minv=rebuild_minv).numpy()
    assert got.shape == (16, L.NKP)
    # the same operations in the same order: equal up to the last bit, at most one ulp apart
    np.testing.assert_array_max_ulp(got, ref, maxulp=1)
    one = E.derive_params_torch(torch.from_numpy(ph[0]), rebuild_minv=rebuild_minv).numpy()
    np.testing.assert_array_max_ulp(one, ref[0], maxulp=1)


@pytest.mark.parametrize("rebuild_minv", [True, False])
def test_derive_params_torch_jacobian_is_coefficient_directions(E, L, rebuild_minv):
    ph = _vehicles(E, L, 1, 5)[0]
    idx = [i for i in range(L.NPHYS) if i != L.PH_TLAG1 and not (rebuild_minv and L.PH_MINV <= i < L.PH_MINV + 6)]
    J = torch.autograd.functional.jacobian(lambda p: E.derive_params_torch(p, rebuild_minv=rebuild_minv),
                                           torch.from_numpy(ph)).numpy()           # [NKP, NPHYS]
    D = E.coefficient_directions(ph, idx, rebuild_minv=rebuild_minv)              # [p, NKP]
    np.testing.assert_allclose(J[:, idx].T, D, rtol=1e-14, atol=1e-14 * np.abs(D).max())
    assert not J[:, L.PH_TLAG1].any()
