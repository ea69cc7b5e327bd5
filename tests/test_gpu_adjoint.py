"""GPU tests of the reverse-mode rollout gradients (brov_rollout_vjp through Engine.rollout_vjp / rollout_diff): the
result equals the exact chain over Engine.linearize's Jacobians, directional derivatives agree with central differences
of the rollout and of the numpy oracle, torch.autograd.gradcheck passes, position has its exact structure, results are
bit-reproducible under repeats, permutation, input layouts and chaining, and edge sizes, health counters, refusals and
arrays above 2^31 elements behave."""
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


def _problem(e, n, T, seed):
    """z0 [n, NZ] at moderate angles with nonzero velocities, smooth inputs U [T, n, NU] (numpy)"""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, e.nx))
    x[:, :3] = rng.uniform(-2, 2, (n, 3))
    ang = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.5, 0.5, n), rng.uniform(-3, 3, n)], axis=1)
    nu = np.concatenate([rng.uniform(-0.6, 0.6, (n, 3)), rng.uniform(-0.4, 0.4, (n, 3))], axis=1)
    if e.nx == 13:
        x[:, 3:7] = O.euler_to_quat(ang[:, 0], ang[:, 1], ang[:, 2])
        x[:, 7:] = nu
    else:
        x[:, 3:6] = ang
        x[:, 6:] = nu
    thr = e.model == "thruster8"
    if thr:
        z = np.concatenate([x, e.project_lag(rng.uniform(-0.5, 0.5, (n, 24))).cpu().numpy()], axis=1)
    else:
        z = x
    U = np.stack([O.smooth_inputs(rng, T, e.nu, scale=0.5 if thr else 3.0) for _ in range(n)], axis=1)
    return z, U


def _vjp(e, z0, U, integ="rk4", **kw):
    thr = e.model == "thruster8"
    return e.rollout_vjp(z0[:, :e.nx], U, dt=DT, integrator=integ, lag0=z0[:, e.nx:] if thr else None,
                         lag_repr="projected", **kw)


def _gz0(e, r):
    return torch.cat([r.gx0, r.glag0], dim=1) if e.model == "thruster8" else r.gx0


@pytest.mark.parametrize("stride", [1, 7])
@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_gradient_equals_the_exact_chain_over_linearize(B, model, integ, cur, stride):
    e = _engine(B, model, cur)
    n, T = 37, 60
    z0, U = _problem(e, n, T, 1)
    rng = np.random.default_rng(2)
    gtraj = rng.standard_normal((T // stride, n, e.nx))
    gzT = rng.standard_normal((n, e.nz))
    r = _vjp(e, z0, U, integ, gtraj=gtraj, gzT=gzT, stride=stride)
    lin = e.linearize(z0[:, :e.nx], U, dt=DT, integrator=integ, lag0=z0[:, e.nx:] if model == "thruster8" else None,
                      lag_repr="projected")
    lam = e.tensor(gzT).clone()
    gt = e.tensor(gtraj)
    gU = torch.empty((T, n, e.nu), dtype=torch.float64, device=e.device)
    for k in range(T - 1, -1, -1):
        if (k + 1) % stride == 0:
            lam[:, :e.nx] += gt[(k + 1) // stride - 1]
        gU[k] = torch.einsum("nzu,nz->nu", lin.B[k], lam)
        lam = torch.einsum("nzy,nz->ny", lin.A[k], lam)
    assert _normwise(_gz0(e, r).cpu(), lam.cpu()) <= 1e-12
    assert _normwise(r.gU.cpu(), gU.cpu()) <= 1e-12
    assert _normwise(r.z.cpu(), lin.z.cpu()) <= 1e-13


def _loss_rollout(e, z0, U, gtraj, gzT, stride, integ):
    thr = e.model == "thruster8"
    r = e.rollout(z0[:, :e.nx], U, dt=DT, integrator=integ, lag0=z0[:, e.nx:] if thr else None, lag_repr="projected",
                  stride=stride)
    zT = torch.cat([r.xT, r.lag], dim=1) if thr else r.xT
    return (r.traj * gtraj).sum(dim=(0, 2)) + (zT * gzT).sum(dim=1)   # per vehicle


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_directional_derivatives_match_central_differences(B, model, integ, cur):
    e = _engine(B, model, cur)
    n, T, stride = 16, 40, 5
    thr = model == "thruster8"
    z0, U = _problem(e, n, T, 3)
    rng = np.random.default_rng(4)
    gtraj = rng.standard_normal((T // stride, n, e.nx))
    gzT = rng.standard_normal((n, e.nz))
    dz = rng.standard_normal(z0.shape)
    dU = rng.standard_normal(U.shape) * (0.1 if thr else 1.0)
    r = _vjp(e, z0, U, integ, gtraj=gtraj, gzT=gzT, stride=stride)
    ad = ((_gz0(e, r).cpu().numpy() * dz).sum(1) + (r.gU.cpu().numpy() * dU).sum((0, 2)))
    # central differences of Engine.rollout
    h = 1e-6
    gt, gT = e.tensor(gtraj), e.tensor(gzT)
    lp = _loss_rollout(e, z0 + h * dz, U + h * dU, gt, gT, stride, integ).cpu().numpy()
    lm = _loss_rollout(e, z0 - h * dz, U - h * dU, gt, gT, stride, integ).cpu().numpy()
    fd = (lp - lm) / (2 * h)
    assert np.max(np.abs(ad - fd) / np.maximum(np.abs(fd), 1.0)) <= 1e-6
    # and independently of the numpy oracle (per-thruster lag; Z = P L, the gradient in per-thruster coordinates)
    m = O.Model(model, DT, O.default_params(current=CURRENT if cur else (0.0, 0.0, 0.0)))
    L0 = rng.uniform(-0.5, 0.5, (n, 24)) if thr else None
    dL = rng.standard_normal((n, 24)) if thr else None
    r2 = e.rollout_vjp(z0[:, :e.nx], U, gtraj=gtraj, gzT=gzT, stride=stride, dt=DT, integrator=integ, lag0=L0,
                       lag_repr="thruster")
    ad2 = (r2.gx0.cpu().numpy() * dz[:, :e.nx]).sum(1) + (r2.gU.cpu().numpy() * dU).sum((0, 2))
    if thr:
        ad2 = ad2 + (r2.glag0.cpu().numpy() * dL).sum(1)
        P = O.thruster_geometry()[2]

    def loss_np(s):
        snaps, xT, lagT = O.rollout(m, integ, z0[:, :e.nx] + s * dz[:, :e.nx], U + s * dU,
                                    lag0=(L0 + s * dL) if thr else None, stride=stride)
        out = (snaps * gtraj).sum((0, 2)) + (xT * gzT[:, :e.nx]).sum(1)
        if thr:
            out = out + (np.einsum("ci,nik->nck", P, lagT).reshape(n, 18) * gzT[:, e.nx:]).sum(1)
        return out

    fd2 = (loss_np(h) - loss_np(-h)) / (2 * h)
    assert np.max(np.abs(ad2 - fd2) / np.maximum(np.abs(fd2), 1.0)) <= 1e-6


@pytest.mark.parametrize("model", MODELS)
def test_rollout_diff_passes_gradcheck(B, model):
    e = _engine(B, model, True)
    n, T, stride = 2, 6, 2
    z0, U = _problem(e, n, T, 5)
    x0 = e.tensor(z0[:, :e.nx]).clone().requires_grad_(True)
    Ut = e.tensor(U).clone().requires_grad_(True)
    thr = model == "thruster8"
    lag0 = e.tensor(z0[:, e.nx:]).clone().requires_grad_(True) if thr else None

    def f(x0, Ut, *lag):
        traj, xT, lagT = e.rollout_diff(x0, Ut, lag0=lag[0] if lag else None, dt=DT, integrator="rk4", stride=stride)
        return (traj, xT, lagT) if thr else (traj, xT)

    inputs = (x0, Ut, lag0) if thr else (x0, Ut)
    assert torch.autograd.gradcheck(f, inputs, eps=1e-6, atol=1e-6, rtol=1e-5)


def test_thruster_lag_gradient_in_per_thruster_coordinates(B):
    e = _engine(B, "thruster8")
    n, T = 5, 30
    z0, U = _problem(e, n, T, 6)
    rng = np.random.default_rng(7)
    L24 = rng.uniform(-0.5, 0.5, (n, 24))
    gzT = rng.standard_normal((n, e.nz))
    rt = e.rollout_vjp(z0[:, :12], U, gzT=gzT, dt=DT, lag0=L24, lag_repr="thruster")
    rp = e.rollout_vjp(z0[:, :12], U, gzT=gzT, dt=DT, lag0=e.project_lag(L24), lag_repr="projected")
    P = e.tensor(e._alloc)
    want = torch.einsum("ci,nck->nik", P, rp.glag0.reshape(n, 6, 3)).reshape(n, 24)
    assert torch.equal(rt.glag0, want)
    # central differences in the per-thruster lag
    d = rng.standard_normal((n, 24))
    h = 1e-6

    def loss(s):
        r = e.rollout(z0[:, :12], U, dt=DT, lag0=e.project_lag(L24 + s * d), lag_repr="projected")
        zT = torch.cat([r.xT, r.lag], dim=1).cpu().numpy()
        return (zT * gzT).sum(1)

    fd = (loss(h) - loss(-h)) / (2 * h)
    ad = (rt.glag0.cpu().numpy() * d).sum(1)
    assert np.max(np.abs(ad - fd) / np.maximum(np.abs(fd), 1.0)) <= 1e-6


@pytest.mark.parametrize("model", MODELS)
def test_position_gradient_is_the_sum_of_its_cotangents(B, model):
    e = _engine(B, model, True)
    n, T, stride = 33, 50, 5
    z0, U = _problem(e, n, T, 8)
    rng = np.random.default_rng(9)
    gtraj = rng.standard_normal((T // stride, n, e.nx))
    gzT = rng.standard_normal((n, e.nz))
    r = _vjp(e, z0, U, gtraj=gtraj, gzT=gzT, stride=stride)
    # the reverse sweep adds the cotangents in the order it meets them and leaves the position rows otherwise alone
    want = gzT[:, :3].copy()
    for j in range(T // stride - 1, -1, -1):
        want = want + gtraj[j, :, :3]
    assert np.max(np.abs(r.gx0[:, :3].cpu().numpy() - want)) <= 1e-15


@pytest.mark.parametrize("model", MODELS)
def test_bit_for_bit_repeats_permutation_layouts_and_chaining(B, model):
    e = _engine(B, model, True)
    n, T, stride = 45, 42, 7
    thr = model == "thruster8"
    z0, U = _problem(e, n, T, 10)
    rng = np.random.default_rng(11)
    gtraj = rng.standard_normal((T // stride, n, e.nx))
    gzT = rng.standard_normal((n, e.nz))
    r1 = _vjp(e, z0, U, gtraj=gtraj, gzT=gzT, stride=stride)
    r2 = _vjp(e, z0, U, gtraj=gtraj, gzT=gzT, stride=stride)
    assert torch.equal(_gz0(e, r1), _gz0(e, r2)) and torch.equal(r1.gU, r2.gU) and torch.equal(r1.z, r2.z)
    perm = rng.permutation(n)
    rp = _vjp(e, z0[perm], U[:, perm], gtraj=gtraj[:, perm], gzT=gzT[perm], stride=stride)
    pt = torch.as_tensor(perm, device=e.device)
    assert torch.equal(_gz0(e, rp), _gz0(e, r1)[pt]) and torch.equal(rp.gU, r1.gU[:, pt])
    # shared and constant inputs against the expanded per-vehicle series
    Us = U[:, 0]
    rs = _vjp(e, z0, Us, gtraj=gtraj, gzT=gzT, stride=stride, u_layout="shared")
    re_ = _vjp(e, z0, np.ascontiguousarray(np.broadcast_to(Us[:, None], U.shape)), gtraj=gtraj, gzT=gzT, stride=stride)
    assert torch.equal(_gz0(e, rs), _gz0(e, re_)) and torch.equal(rs.gU, re_.gU)
    Uc = U[0]
    rc = _vjp(e, z0, (Uc, T), gtraj=gtraj, gzT=gzT, stride=stride, u_layout="const")
    rce = _vjp(e, z0, np.ascontiguousarray(np.broadcast_to(Uc[None], U.shape)), gtraj=gtraj, gzT=gzT, stride=stride)
    assert torch.equal(_gz0(e, rc), _gz0(e, rce)) and torch.equal(rc.gU, rce.gU)
    # two chained calls at t1 (a multiple of the stride) against one call
    t1 = 21
    first = _vjp(e, z0, U[:t1])                           # z at t1
    zt1 = first.z.cpu().numpy()
    second = _vjp(e, zt1, U[t1:], gtraj=gtraj[t1 // stride:], gzT=gzT, stride=stride)
    head = _vjp(e, z0, U[:t1], gtraj=gtraj[:t1 // stride], gzT=_gz0(e, second), stride=stride)
    assert torch.equal(_gz0(e, head), _gz0(e, r1))
    assert torch.equal(torch.cat([head.gU, second.gU]), r1.gU)
    assert torch.equal(second.z, r1.z)
    if thr:
        assert r1.glag0.shape == (n, 18)


@pytest.mark.parametrize("model", MODELS)
def test_edge_sizes(B, model):
    e = _engine(B, model)
    z0, U = _problem(e, 300, 9, 12)
    rng = np.random.default_rng(13)
    gzT = rng.standard_normal((300, e.nz))
    ref = _vjp(e, z0, U, gzT=gzT)
    for n in (1, 127, 128, 129, 257):
        r = _vjp(e, z0[:n], U[:, :n], gzT=gzT[:n])
        assert torch.equal(_gz0(e, r), _gz0(e, ref)[:n]) and torch.equal(r.gU, ref.gU[:, :n])
    # T = 1 against the one-step linearization
    r = _vjp(e, z0, U[:1], gzT=gzT)
    lin = e.linearize(z0[:, :e.nx], U[:1], lag0=z0[:, e.nx:] if model == "thruster8" else None, lag_repr="projected",
                      dt=DT)
    g = e.tensor(gzT)
    assert _normwise(_gz0(e, r).cpu(), torch.einsum("nzy,nz->ny", lin.A[0], g).cpu()) <= 1e-12
    # stride > T: no snapshot, no trajectory term
    r = _vjp(e, z0, U, gtraj=np.zeros((0, 300, e.nx)), gzT=gzT, stride=20)
    assert torch.equal(_gz0(e, r), _gz0(e, ref))
    # n = 0 is a no-op
    r = _vjp(e, z0[:0], U[:, :0])
    assert r.gU.shape == (9, 0, e.nu)


@pytest.mark.parametrize("model", MODELS)
def test_health_counts_non_finite_inputs_and_singular_pitch(B, model):
    e = _engine(B, model)
    n, T = 40, 12
    z0, U = _problem(e, n, T, 14)
    U[5, 3, 2] = np.nan
    r = _vjp(e, z0, U, gzT=np.ones((n, e.nz)), health=True)
    assert int(r.health[0]) == 1
    assert bool(torch.isfinite(r.gU[:, [i for i in range(n) if i != 3]]).all())
    if model != "quat13":
        z0, U = _problem(e, n, T, 14)
        z0[7, 4] = np.pi / 2 - 1e-4
        r = _vjp(e, z0, U, gzT=np.ones((n, e.nz)), health=True, singular_eps=1e-3)
        assert int(r.health[1]) >= 1


def _desc(L, e, n, T, z0, U, gz0, gU, ws, wsb):
    d = L.RolloutVjpDesc()
    d.struct_size = C.sizeof(L.RolloutVjpDesc)
    d.integrator = L.RK4
    d.n, d.steps, d.dt = n, T, DT
    d.z0_dev, d.u_dev = z0.data_ptr(), U.data_ptr()
    d.u_stride_t, d.u_stride_n = n * e.nu, e.nu
    d.gz0_dev, d.gu_dev = gz0.data_ptr(), gU.data_ptr()
    d.workspace_dev, d.workspace_bytes = ws.data_ptr(), wsb
    return d


def test_refusals(B, L):
    n, T = 4, 3
    e = B.Engine("thruster8", "f32")
    with pytest.raises(B.BrovError, match="fp64"):
        e.rollout_vjp(torch.zeros(n, 12), torch.zeros(T, n, 8))
    e = B.Engine("di12_u8", "f64")
    with pytest.raises(B.BrovError, match="double-integrator"):
        e.rollout_vjp(torch.zeros(n, 12), torch.zeros(T, n, 8))
    e = B.Engine("wrench12", "f64")
    e.set_wrench_lag1(True, 0.1)
    with pytest.raises(B.BrovError, match="first-order"):
        e.rollout_vjp(torch.zeros(n, 12), torch.zeros(T, n, 6))
    e = B.Engine("thruster8", "f64")
    e.set_vehicle_physical(np.repeat(B.default_physical()[None], n, axis=0))
    with pytest.raises(B.BrovError, match="per-vehicle"):
        e.rollout_vjp(torch.zeros(n, 12), torch.zeros(T, n, 8))
    e = B.Engine("thruster8", "f64")
    dev = e.device
    z0 = torch.zeros(n, 30, dtype=torch.float64, device=dev)
    U = torch.zeros(T, n, 8, dtype=torch.float64, device=dev)
    gz0 = torch.empty(n, 30, dtype=torch.float64, device=dev)
    gU = torch.empty(T, n, 8, dtype=torch.float64, device=dev)
    need = L.lib.brov_rollout_vjp_workspace_bytes(L.THRUSTER8_LAG3, n, T)
    assert need == n * T * 30 * 8
    ws = torch.empty(need // 8, dtype=torch.float64, device=dev)
    gt = torch.zeros(T, n, 12, dtype=torch.float64, device=dev)
    sentinel = gz0.clone()

    def run(**kw):
        d = _desc(L, e, n, T, z0, U, gz0, gU, ws, need)
        for k, v in kw.items():
            setattr(d, k, v)
        return L.lib.brov_rollout_vjp(e._h, C.byref(d), None)

    assert run() == 0
    torch.cuda.synchronize()
    sentinel = gz0.clone()
    assert run(workspace_bytes=need - 1) == -1
    assert run(workspace_dev=None) == -1
    assert run(gtraj_dev=gt.data_ptr(), stride=0) == -1
    assert run(steps=0) == -1
    assert run(n=-1) == -1
    assert run(dt=0.0) == -1
    assert run(u_stride_t=-1) == -1
    assert run(gu_dev=None) == -1
    assert run(gz0_dev=None) == -1
    assert run(integrator=7) == -1
    assert run(struct_size=8) == -1
    torch.cuda.synchronize()
    assert torch.equal(gz0, sentinel)
    assert run(n=0) == 0
    assert L.lib.brov_rollout_vjp_workspace_bytes(L.DI_EULER12_U8, n, T) == 0


def test_more_than_2_31_elements_in_gU_and_the_workspace(B):
    e = _engine(B, "wrench12")
    n, T = 1 << 21, 180
    assert T * n * 6 > 2 ** 31 and T * n * 12 > 2 ** 31
    rng = np.random.default_rng(15)
    zs, Us = _problem(e, 8, T, 16)
    idx = np.array([0, 1, 777_777, 1_234_567, n - 2, n - 1])
    z0 = torch.zeros((n, 12), dtype=torch.float64, device=e.device)
    z0[:, 6] = 0.1
    z0[torch.as_tensor(idx, device=e.device)] = e.tensor(zs[:6])
    U = torch.zeros((T, n, 6), dtype=torch.float64, device=e.device)
    U[:, torch.as_tensor(idx, device=e.device)] = e.tensor(Us[:, :6])
    gzT = torch.zeros((n, 12), dtype=torch.float64, device=e.device)
    gsel = rng.standard_normal((6, 12))
    gzT[torch.as_tensor(idx, device=e.device)] = e.tensor(gsel)
    r = e.rollout_vjp(z0, U, gzT=gzT, dt=DT)
    small = _vjp(e, zs[:6], Us[:, :6], gzT=gsel)
    it = torch.as_tensor(idx, device=e.device)
    assert torch.equal(r.gx0[it], small.gx0)
    assert torch.equal(r.gU[:, it], small.gU)
    assert torch.equal(r.z[it], small.z)
