"""CPU-side tests of the extended Kalman filter (no GPU): the C descriptor of brov_ekf and its ctypes mirror agree, the
entry point is exported with the ABI unchanged, and the numpy oracle's sequential scalar updates equal the textbook
joint Kalman update on a linear system."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import ekf_np


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200.build import build_lib
    build_lib()
    from bluerov2_dynamics_b200 import _lib
    return _lib


def test_ekf_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.EkfDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_ekf_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_ekf_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    # 4 + 4, n / steps / dt, z0 / P0, u and y with two strides, q and r with one, four outputs + stride,
    # three statistics + flag + reserved, health, singular_eps
    assert int(got["size"]) == C.sizeof(ct) == 8 + 24 + 16 + 2 * 24 + 2 * 16 + 5 * 8 + 3 * 8 + 8 + 8 + 8
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname


def test_ekf_symbol_is_exported(L):
    out = subprocess.run(["nm", "-D", "--defined-only", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert any(line.split()[-1] == "brov_ekf" for line in out.splitlines() if line.strip())
    assert "brov_ekf" in L._PROTOS
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8


def _joint_kalman(A, x0, P0, Y, q, r):
    """the textbook filter: x- = A x, P- = A P A^T + Q, then one joint update with H the rows of the measured
    components, K = P- H^T S^-1, Joseph form, loglik = log N(nu; 0, S)"""
    x, P = x0.copy(), P0.copy()
    nx = x.shape[0]
    ll = 0.0
    xs, Ps = [], []
    for y in Y:
        x = A @ x
        P = A @ P @ A.T + np.diag(q)
        sel = np.flatnonzero(np.isfinite(y))
        if sel.size:
            H = np.eye(nx)[sel]
            R = np.diag(r[sel])
            nu = y[sel] - H @ x
            S = H @ P @ H.T + R
            K = P @ H.T @ np.linalg.inv(S)
            x = x + K @ nu
            IKH = np.eye(nx) - K @ H
            P = IKH @ P @ IKH.T + K @ R @ K.T
            ll -= 0.5 * (nu @ np.linalg.solve(S, nu) + np.linalg.slogdet(S)[1] + sel.size * np.log(2 * np.pi))
        xs.append(x)
        Ps.append(P)
    return np.array(xs), np.array(Ps), ll


def test_sequential_scalar_updates_equal_the_joint_kalman_update():
    rng = np.random.default_rng(0)
    nx, N, T = 6, 5, 40
    A = np.eye(nx) + 0.05 * rng.standard_normal((nx, nx))
    q = rng.uniform(0.01, 0.1, nx)
    r = rng.uniform(0.05, 0.5, nx)
    x0 = rng.standard_normal((N, nx))
    M = rng.standard_normal((N, nx, nx))
    P0 = M @ np.swapaxes(M, 1, 2) + np.eye(nx)
    Y = rng.standard_normal((T, N, nx))
    Y[rng.random((T, N, nx)) < 0.4] = np.nan
    Y[7, 2] = np.nan                                      # a step with nothing measured
    out = ekf_np.ekf(lambda x, a, u: (x @ A.T, a), lambda x, a, u: np.broadcast_to(A, (x.shape[0], nx, nx)),
                     x0, None, P0, np.zeros((T, N, 1)), Y, q, r, wrap=())
    for i in range(N):
        xs, Ps, ll = _joint_kalman(A, x0[i], P0[i], Y[:, i], q, r)
        assert np.max(np.abs(out["x_traj"][:, i] - xs)) <= 1e-12 * max(1.0, np.max(np.abs(xs)))
        assert np.max(np.abs(out["P_traj"][:, i] - Ps)) <= 1e-12 * max(1.0, np.max(np.abs(Ps)))
        assert abs(out["loglik"][i] - ll) <= 1e-12 * max(1.0, abs(ll))
        assert out["count"][i] == np.isfinite(Y[:, i]).sum()
    assert np.array_equal(out["P"], np.swapaxes(out["P"], 1, 2))
