"""GPU tests of the step Jacobians (brov_linearize through Engine.linearize): the primal trajectory equals the rollout,
J agrees with central differences of one-step rollouts and of the numpy oracle, the first-order remainder falls
quadratically, the lag rows and the position columns have their exact structure, results are reproducible, chainable
and independent of the neighbouring vehicles and of the input layout, the health counters and argument checks work,
and outputs above 2^31 elements are indexed correctly."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import fossen_np as O

pytestmark = pytest.mark.gpu

DT = 0.02
MODELS = ("thruster8", "wrench12", "quat13")
CASES = [(m, i, c) for m in MODELS for i in ("rk4", "euler") for c in (False, True)]
IDS = [f"{m}-{i}-{'current' if c else 'still'}" for m, i, c in CASES]
CURRENT = (0.12, -0.07, 0.05)


@pytest.fixture(scope="module")
def B():
    import bluerov2_dynamics_b200 as b
    return b


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200 import _lib
    return _lib


def _engine(B, model, current=False):
    return B.Engine(model, "f64", current=CURRENT if current else None)


def _normwise(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _point(e, n, seed):
    """n vehicles at moderate angles with nonzero velocities (z [n, NZ]) and inputs u [n, NU]."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, e.nx))
    x[:, :3] = rng.uniform(-2, 2, (n, 3))
    ang = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.5, 0.5, n), rng.uniform(-3, 3, n)], axis=1)
    nu = np.concatenate([rng.choice([-1, 1], (n, 3)) * rng.uniform(0.1, 0.6, (n, 3)),
                         rng.choice([-1, 1], (n, 3)) * rng.uniform(0.05, 0.4, (n, 3))], axis=1)
    if e.nx == 13:
        x[:, 3:7] = O.euler_to_quat(ang[:, 0], ang[:, 1], ang[:, 2])
        x[:, 7:] = nu
    else:
        x[:, 3:6] = ang
        x[:, 6:] = nu
    if e.model == "thruster8":
        L24 = rng.uniform(-0.5, 0.5, (n, 24))
        z = np.concatenate([x, e.project_lag(L24).cpu().numpy()], axis=1)
        u = rng.uniform(-0.8, 0.8, (n, 8))
    else:
        z = x
        u = np.concatenate([rng.uniform(-8, 8, (n, 3)), rng.uniform(-1, 1, (n, 3))], axis=1)
    return z, u


def _phi(e, z, u, integ):
    """one step of the engine's rollout in projected lag coordinates: z [M, NZ], u [M, NU] -> z' [M, NZ] (numpy)"""
    z = np.asarray(z, float)
    thr = e.model == "thruster8"
    r = e.rollout(z[:, :e.nx], np.asarray(u, float)[None], dt=DT, integrator=integ,
                  lag0=z[:, e.nx:] if thr else None, lag_repr="projected")
    out = r.xT.cpu().numpy()
    return np.concatenate([out, r.lag.cpu().numpy()], axis=1) if thr else out


def _fd_jacobian(e, z, u, integ, phi, h=1e-5):
    """central differences of phi over every column of [z | u]: [n, NZ, NC]"""
    n, nz = z.shape
    nc = nz + u.shape[1]
    w = np.concatenate([z, u], axis=1)
    W = np.repeat(w[:, None, None, :], 2, axis=1).repeat(nc, axis=2)          # [n, 2, nc, nc]
    hs = h * np.maximum(1.0, np.abs(w))                                          # [n, nc]
    idx = np.arange(nc)
    W[:, 0, idx, idx] += hs
    W[:, 1, idx, idx] -= hs
    W = W.reshape(-1, nc)
    out = phi(W[:, :nz], W[:, nz:]).reshape(n, 2, nc, nz)
    return np.transpose((out[:, 0] - out[:, 1]) / (2 * hs[:, :, None]), (0, 2, 1))


def _J(res):
    return torch.cat([res.A, res.B], dim=-1)


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_primal_trajectory_equals_rollout(B, model, integ, cur):
    e = _engine(B, model, cur)
    n, T = 37, 200
    z0, _ = _point(e, n, 1)
    rng = np.random.default_rng(2)
    U = np.stack([O.smooth_inputs(rng, T, e.nu, scale=0.5 if model == "thruster8" else 3.0) for _ in range(n)], axis=1)
    res = e.linearize(z0[:, :e.nx], U, dt=DT, integrator=integ, lag0=z0[:, e.nx:] if model == "thruster8" else None,
                      lag_repr="projected")
    r = e.rollout(z0[:, :e.nx], U, dt=DT, integrator=integ, stride=1, lag_repr="projected",
                  lag0=z0[:, e.nx:] if model == "thruster8" else None)
    zt = res.z_traj.cpu().numpy()
    assert _normwise(zt[:, :, :e.nx], r.traj.cpu().numpy()) <= 1e-12
    assert torch.equal(res.z, res.z_traj[-1])
    if model == "thruster8":
        assert _normwise(zt[-1, :, e.nx:], r.lag.cpu().numpy()) <= 1e-12


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_jacobian_matches_central_differences(B, model, integ, cur):
    e = _engine(B, model, cur)
    z, u = _point(e, 256, 3)
    res = e.linearize(z[:, :e.nx], u, dt=DT, integrator=integ, lag0=z[:, e.nx:] if model == "thruster8" else None,
                      lag_repr="projected")
    J = _J(res)[0].cpu().numpy()
    assert J.shape == (256, e.nz, e.nz + e.nu)
    fd = _fd_jacobian(e, z, u, integ, lambda zz, uu: _phi(e, zz, uu, integ))
    assert _normwise(J, fd) <= 1e-7
    # every column on its own, including the lag and input columns
    for j in range(J.shape[2]):
        assert np.max(np.abs(J[:, :, j] - fd[:, :, j])) <= 1e-7 * max(np.max(np.abs(J)), 1.0), j


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_first_order_remainder_falls_quadratically(B, model, integ, cur):
    e = _engine(B, model, cur)
    n = 16
    z, u = _point(e, n, 4)
    res = e.linearize(z[:, :e.nx], u, dt=DT, integrator=integ, lag0=z[:, e.nx:] if model == "thruster8" else None,
                      lag_repr="projected")
    J = _J(res)[0].cpu().numpy()
    rng = np.random.default_rng(5)
    v = rng.standard_normal((n, e.nz + e.nu))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    base = _phi(e, z, u, integ)
    rem = []
    for eps in (1e-3, 1e-4):
        w = np.concatenate([z, u], axis=1) + eps * v
        p = _phi(e, w[:, :e.nz], w[:, e.nz:], integ)
        rem.append(np.linalg.norm(p - base - eps * np.einsum("nij,nj->ni", J, v), axis=1))
    ratio = rem[0] / rem[1]
    assert np.all((ratio >= 50) & (ratio <= 200)), ratio


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_exact_structure(B, model, integ, cur):
    e = _engine(B, model, cur)
    z, u = _point(e, 100, 6)
    T = 3
    U = np.repeat(u[None], T, axis=0) * np.linspace(1.0, 0.5, T)[:, None, None]
    res = e.linearize(z[:, :e.nx], U, dt=DT, integrator=integ, lag0=z[:, e.nx:] if model == "thruster8" else None,
                      lag_repr="projected")
    A = res.A.cpu().numpy()
    Bm = res.B.cpu().numpy()
    eye = np.eye(e.nz)
    # positions enter no right-hand side: unit columns, bit for bit
    assert np.array_equal(A[..., :, :3], np.broadcast_to(eye[:, :3], A[..., :, :3].shape))
    if model != "thruster8":
        return
    nx = e.nx
    assert np.array_equal(A[..., nx:, :nx], np.zeros_like(A[..., nx:, :nx]))
    Ad, Bd = B.lag_discretize(DT)
    nsub = 4 if integ == "rk4" else 1
    lagA = np.linalg.matrix_power(Ad, nsub)
    lagB = sum(np.linalg.matrix_power(Ad, j) for j in range(nsub)) @ Bd
    assert _normwise(A[..., nx:, nx:], np.broadcast_to(np.kron(np.eye(6), lagA), A[..., nx:, nx:].shape)) <= 1e-14
    alloc = B.default_allocation()[0]
    a, b, c, d, f = -140.3, 389.9, -404.1, 176.0, 8.9
    s = U * U
    Fp = (((9 * a * s + 7 * b) * s + 5 * c) * s + 3 * d) * s + f                     # [T, n, 8]
    ref = np.einsum("k,ci,tni->tncki", lagB, alloc, Fp).reshape(T, 100, 18, 8)
    assert _normwise(Bm[..., nx:, :], ref) <= 1e-14


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_state_and_input_columns_match_the_numpy_oracle(B, model, integ, cur):
    e = _engine(B, model, cur)
    n = 64
    z, u = _point(e, n, 7)
    m = O.Model(model, DT, O.default_params(current=CURRENT if cur else (0.0, 0.0, 0.0)))
    thr = model == "thruster8"
    rng = np.random.default_rng(8)
    L24 = rng.uniform(-0.5, 0.5, (n, 8, 3))
    if thr:
        z[:, e.nx:] = e.project_lag(L24).cpu().numpy()
    res = e.linearize(z[:, :e.nx], u, dt=DT, integrator=integ, lag0=L24.reshape(n, 24) if thr else None)
    J = _J(res)[0].cpu().numpy()
    alloc = O.thruster_geometry()[2]
    nx, nz, nc = e.nx, e.nz, e.nz + e.nu
    cols = list(range(nx)) + list(range(nz, nc))
    rep = 2 * len(cols)

    def phi(zz, uu):
        # the per-thruster lag is held at L24 for every perturbed copy (only x and u are perturbed); Z' = P L'
        xo, lo = O.step(m, integ, zz[:, :nx], uu, np.repeat(L24, rep, axis=0) if thr else None)
        return np.concatenate([xo, np.einsum("ci,nik->nck", alloc, lo).reshape(-1, 18)], axis=1) if thr else xo

    w = np.concatenate([z, u], axis=1)
    W = np.repeat(w[:, None, :], rep, axis=1)
    hs = 1e-5 * np.maximum(1.0, np.abs(w[:, cols]))
    for q, cq in enumerate(cols):
        W[:, 2 * q, cq] += hs[:, q]
        W[:, 2 * q + 1, cq] -= hs[:, q]
    W = W.reshape(-1, nc)
    out = phi(W[:, :nz], W[:, nz:]).reshape(n, len(cols), 2, nz)
    fd = np.transpose((out[:, :, 0] - out[:, :, 1]) / (2 * hs[:, :, None]), (0, 2, 1))
    assert _normwise(J[:, :, cols], fd) <= 1e-7


@pytest.mark.parametrize("model", MODELS)
def test_chaining_reproducibility_permutation_and_layouts(B, model):
    e = _engine(B, model, True)
    thr = model == "thruster8"
    n, T = 101, 6                                    # ragged: not a multiple of the vehicles per block
    z, u = _point(e, n, 9)
    rng = np.random.default_rng(10)
    U = u[None] + 0.1 * rng.standard_normal((T, n, e.nu))
    lag0 = z[:, e.nx:] if thr else None
    kw = dict(dt=DT, integrator="rk4", lag_repr="projected")
    r = e.linearize(z[:, :e.nx], U, lag0=lag0, **kw)
    J = _J(r)
    # run to run
    r2 = e.linearize(z[:, :e.nx], U, lag0=lag0, **kw)
    assert torch.equal(J, _J(r2)) and torch.equal(r.z, r2.z) and torch.equal(r.z_traj, r2.z_traj)
    # T steps in one call = two chained calls
    a = e.linearize(z[:, :e.nx], U[:2], lag0=lag0, **kw)
    b = e.linearize(a.z[:, :e.nx], U[2:], lag0=a.z[:, e.nx:] if thr else None, **kw)
    assert torch.equal(J, torch.cat([_J(a), _J(b)])) and torch.equal(r.z, b.z)
    assert torch.equal(r.z_traj, torch.cat([a.z_traj, b.z_traj]))
    # a vehicle's block does not depend on its neighbours
    perm = rng.permutation(n)
    p = e.linearize(z[perm, :e.nx], U[:, perm], lag0=lag0[perm] if thr else None, **kw)
    assert torch.equal(_J(p), J[:, perm]) and torch.equal(p.z, r.z[perm])
    # N = 1
    one = e.linearize(z[5:6, :e.nx], U[:, 5:6], lag0=lag0[5:6] if thr else None, **kw)
    assert torch.equal(_J(one), J[:, 5:6])
    # the three input layouts agree
    us = U[:, 0]
    t1 = e.linearize(z[:, :e.nx], np.repeat(us[:, None], n, axis=1), lag0=lag0, **kw)
    t2 = e.linearize(z[:, :e.nx], us, lag0=lag0, u_layout="shared", **kw)
    assert torch.equal(_J(t1), _J(t2)) and torch.equal(t1.z, t2.z)
    c1 = e.linearize(z[:, :e.nx], np.repeat(u[None], T, axis=0), lag0=lag0, **kw)
    c2 = e.linearize(z[:, :e.nx], (u, T), lag0=lag0, u_layout="const", **kw)
    assert torch.equal(_J(c1), _J(c2)) and torch.equal(c1.z, c2.z)
    # a 2-D U is one step; want_traj=False and jac_out give the same J
    s1 = e.linearize(z[:, :e.nx], u, lag0=lag0, want_traj=False, **kw)
    out = torch.empty((1, n, e.nz, e.nz + e.nu), dtype=torch.float64, device="cuda")
    s2 = e.linearize(z[:, :e.nx], u, lag0=lag0, jac_out=out, **kw)
    assert s1.z_traj is None and torch.equal(_J(s1), out) and s2.A.data_ptr() == out.data_ptr()
    assert torch.equal(_J(s1), _J(c1)[:1])


@pytest.mark.parametrize("model", MODELS)
def test_health_counters(B, model):
    e = _engine(B, model)
    n = 50
    z, u = _point(e, n, 11)
    lag0 = z[:, e.nx:] if model == "thruster8" else None
    r = e.linearize(z[:, :e.nx], u, dt=DT, lag0=lag0, lag_repr="projected", health=True)
    assert r.health.tolist() == [0, 0]
    x = z[:, :e.nx].copy()
    x[[3, 17], 6 if e.nx == 12 else 7] = np.nan
    if e.nx == 12:
        x[[4, 20, 41], 4] = np.pi / 2 - 1e-4       # |cos theta| = 1e-4 < 1e-3
    r = e.linearize(x, u, dt=DT, lag0=lag0, lag_repr="projected", health=True)
    assert r.health.tolist() == [2, 3 if e.nx == 12 else 0]


def test_unsupported_and_invalid_calls(B, L):
    z, u = _point(_engine(B, "thruster8"), 4, 12)
    x = z[:, :12]
    with pytest.raises(B.BrovError, match="-4"):
        B.Engine("thruster8", "f32").linearize(x, u)
    di = B.Engine("di12_u8", "f64")
    di.set_di_gains(np.full((8, 3), 0.1), np.full((8, 3), 0.1))
    with pytest.raises(B.BrovError, match="-4"):
        di.linearize(x, u)
    w = B.Engine("wrench12", "f64")
    w.set_wrench_lag1(True, 0.1)
    with pytest.raises(B.BrovError, match="-4"):
        w.linearize(x, u[:, :6])
    e = B.Engine("thruster8", "f64")
    e.set_vehicle_physical(np.tile(B.default_physical(), (4, 1)))
    with pytest.raises(B.BrovError, match="-4"):
        e.linearize(x, u)
    e.set_vehicle_physical(None)
    e.linearize(x, u)                                # fine again once the table is cleared
    with pytest.raises(B.BrovError, match="-1"):
        e.linearize(x, np.zeros((0, 4, 8)))          # steps < 1
    with pytest.raises(B.BrovError, match="-1"):
        e.linearize(x, u, dt=-0.02)
    with pytest.raises(ValueError):
        e.linearize(x, u[:, :6])
    with pytest.raises(ValueError):
        e.linearize(x, u, jac_out=torch.empty((1, 4, 30, 37), dtype=torch.float64, device="cuda"))
    # the C ABI: NULL jac, n = 0 is a no-op
    zt = e.tensor(z)
    ut = e.tensor(u)
    d = L.LinearizeDesc()
    d.struct_size = C.sizeof(L.LinearizeDesc)
    d.n, d.steps, d.dt = 4, 1, DT
    d.z0_dev, d.u_dev, d.u_stride_t, d.u_stride_n = zt.data_ptr(), ut.data_ptr(), 0, 8
    assert L.lib.brov_linearize(e._h, C.byref(d), None) == -1
    d.n = 0
    d.jac_dev = zt.data_ptr()
    assert L.lib.brov_linearize(e._h, C.byref(d), None) == 0
    d.struct_size = 8
    assert L.lib.brov_linearize(e._h, C.byref(d), None) == -1


def test_full_size_output_above_2_31_elements(B):
    e = _engine(B, "thruster8")
    n, T = 65536, 32
    assert T * n * 30 * 38 > 2 ** 31
    z, u = _point(e, n, 13)
    rng = np.random.default_rng(14)
    U = torch.as_tensor(u[None] + 0.05 * rng.standard_normal((T, n, 8)), device="cuda")
    r = e.linearize(z[:, :12], U, dt=DT, lag0=z[:, 12:], lag_repr="projected", want_traj=False)
    pick = np.array([0, 1, 2, 12345, 56491, n - 2, n - 1])
    s = e.linearize(z[pick, :12], U[:, pick], dt=DT, lag0=z[pick, 12:], lag_repr="projected", want_traj=False)
    assert torch.equal(r.A[:, pick], s.A) and torch.equal(r.B[:, pick], s.B) and torch.equal(r.z[pick], s.z)
    del r
    torch.cuda.empty_cache()
