"""CPU-side tests of the candidate sweep (no GPU): the C descriptor and its ctypes mirror agree, the multi-rank
candidate split assembles the same table as one rank, and the Minv helper rebuilds diag(inv(M)) as the reference does."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200.build import build_lib
    build_lib()
    from bluerov2_dynamics_b200 import _lib
    return _lib


def test_sweep_desc_layout_matches_the_ctypes_mirror(L, tmp_path):
    ct = L.SeSweepDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "brov.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(brov_se_sweep_desc));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(brov_se_sweep_desc, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct) == 4 + 4 + 8 * 3 + 8 * 3 + 4 + 4 * 4 + 4 + 8 * 4 + 4 + 4 + 8 * 6
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname
    assert L.ABI_VERSION == 8 and L.lib.brov_abi_version() == 8


def test_sweep_workspace_bytes(L):
    """Partial sums per candidate and window block of 128, plus the carried-lag rows [n_windows][18] in carry mode."""
    f = L.lib.brov_se_sweep_workspace_bytes
    assert f(0, 1000, 0) == 0
    assert f(3, 1000, 0) == 3 * 8 * 4 * 8
    assert f(3, 1000, 1) == 3 * 8 * 4 * 8 + ((1000 * 18 * 8 + 255) // 256) * 256
    assert f(-1, -5, 1) == 0


def test_with_minv_matches_the_reference_formula(L):
    from bluerov2_dynamics_b200.engine import default_physical, with_minv
    from oracle import fossen_np as O
    rng = np.random.default_rng(4)
    ph = np.tile(default_physical(), (16, 1))
    ph[:, L.PH_M] *= rng.uniform(0.8, 1.2, 16)
    ph[:, L.PH_I:L.PH_I + 3] *= rng.uniform(0.8, 1.2, (16, 3))
    ph[:, L.PH_ADDED:L.PH_ADDED + 6] *= rng.uniform(0.5, 1.5, (16, 6))
    got = with_minv(ph)
    names = ["Xu_dot", "Yv_dot", "Zw_dot", "Kp_dot", "Mq_dot", "Nr_dot"]
    p = dict(m=ph[:, L.PH_M], Ix=ph[:, L.PH_I], Iy=ph[:, L.PH_I + 1], Iz=ph[:, L.PH_I + 2],
             **{k: ph[:, L.PH_ADDED + j] for j, k in enumerate(names)})
    assert np.array_equal(got[:, L.PH_MINV:L.PH_MINV + 6], O.minv_diag(p))
    keep = np.r_[0:L.PH_MINV, L.PH_MINV + 6:L.NPHYS]
    assert np.array_equal(got[:, keep], ph[:, keep])          # nothing else changes, the input is not modified
    assert np.array_equal(with_minv(default_physical()), default_physical())


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch
import torch.distributed as dist
from bluerov2_dynamics_b200 import dist as D
P = 37
table = np.random.default_rng(9).normal(size=(P, 4))
def local_fn(lo, hi):
    # stand-in for Engine.multistep_se_sweep on candidates [lo, hi): a per-candidate row of squared-error sums
    return torch.from_numpy(table[lo:hi] ** 2)
one = D.sharded_sweep(local_fn, P, 0, 1)          # world size 1, before the process group exists
rank, world, _ = D.init_from_env("gloo")
got = D.sharded_sweep(local_fn, P, rank, world)
assert got.shape == (P, 4) and torch.equal(got, one) and np.array_equal(one.numpy(), table ** 2)
if rank == 0:
    print("SWEEP_OK")
dist.barrier()
dist.destroy_process_group()
"""


def test_sharded_sweep_world_size_2_gloo(tmp_path):
    """Two gloo ranks score their halves of the candidates; the all-reduced table equals the one-rank table bit for
    bit."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29631", str(script)],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "SWEEP_OK" in r.stdout
