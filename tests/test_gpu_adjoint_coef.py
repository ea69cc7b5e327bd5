"""GPU tests of the coefficient gradients of batched rollouts (brov_rollout_vjp_coef through
Engine.rollout_vjp(coef=True) and Engine.rollout_diff(kp=...)): gkp agrees with central differences in the coefficients
and with the forward-mode gradient of multistep_se_grad, the state and input gradients are those of rollout_vjp,
per-vehicle tables give each vehicle its own gradient, results are bit-reproducible under repeats, permutation, input
layouts and chaining, torch autograd reaches the coefficients and the physical vector, the engine's coefficients
survive, and health counters and refusals behave."""
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
NKPG = 34   # KP_ILAG1: the entries from there on have no gradient


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
    z = np.concatenate([x, e.project_lag(rng.uniform(-0.5, 0.5, (n, 24))).cpu().numpy()], axis=1) if thr else x
    U = np.stack([O.smooth_inputs(rng, T, e.nu, scale=0.5 if thr else 3.0) for _ in range(n)], axis=1)
    return z, U


def _cot(e, n, T, stride, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((T // stride, n, e.nx)), rng.standard_normal((n, e.nz))


def _vjp(e, z0, U, integ="rk4", **kw):
    thr = e.model == "thruster8"
    return e.rollout_vjp(z0[:, :e.nx], U, dt=DT, integrator=integ, lag0=z0[:, e.nx:] if thr else None,
                         lag_repr="projected", **kw)


def _gz0(e, r):
    return torch.cat([r.gx0, r.glag0], dim=1) if e.model == "thruster8" else r.gx0


def _loss(e, z0, U, integ, stride, gt, gT):
    """L of every vehicle from Engine.rollout, float64 numpy [n]"""
    thr = e.model == "thruster8"
    r = e.rollout(z0[:, :e.nx], U, dt=DT, integrator=integ, lag0=z0[:, e.nx:] if thr else None, stride=stride,
                  lag_repr="projected", want_lag=thr)
    zT = torch.cat([r.xT, r.lag], dim=1) if thr else r.xT
    out = (zT.cpu().numpy() * gT).sum(1)
    if gt is not None and gt.shape[0]:
        out += (r.traj.cpu().numpy() * gt).sum(axis=(0, 2))
    return out


def _phys(B, L, k, seed, current=True):
    rng = np.random.default_rng(seed)
    ph = np.tile(B.default_physical(), (k, 1))
    idx = list(range(L.PH_ADDED, L.PH_ADDED + 6)) + list(range(L.PH_LIN, L.PH_QUAD + 6))
    ph[:, idx] *= rng.uniform(0.7, 1.3, (k, len(idx)))
    if current:
        ph[:, L.PH_CURRENT:L.PH_CURRENT + 3] = rng.uniform(-0.15, 0.15, (k, 3))
    return B.with_minv(ph)


@pytest.mark.parametrize("stride", [1, 7])
@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_gkp_against_central_differences(B, L, model, integ, cur, stride):
    e = _engine(B, model, cur)
    T = 42
    z0, U = _problem(e, 1, T, 11)
    gt, gT = _cot(e, 1, T, stride, 12)
    kp0 = B.derive_params(e.phys)
    r = _vjp(e, z0, U, integ, gtraj=gt, gzT=gT, stride=stride, coef=True)
    g = r.gkp.cpu().numpy()[0]
    assert g.shape == (L.NKP,) and not g[NKPG:].any()
    # one rollout of a table: the base vehicle and 4 x 34 copies with kp +- h e_j and kp +- 2h e_j; the Richardson
    # combination of the two central differences is accurate to O(h^4), so h can be large enough that the rounding
    # of L (~1e-16 |L| / h) stays far below the 1e-6 tolerance
    h = 1e-4 * np.maximum(np.abs(kp0[:NKPG]), 0.1)
    table = np.repeat(kp0[None], 1 + 4 * NKPG, axis=0)
    for j in range(NKPG):
        for q, s in enumerate((1, -1, 2, -2)):
            table[1 + 4 * j + q, j] += s * h[j]
    m = table.shape[0]
    with e._coefficients(torch.from_numpy(table).to(e.device)):
        Lv = _loss(e, np.repeat(z0, m, 0), np.repeat(U, m, 1), integ, stride, np.repeat(gt, m, 1),
                   np.repeat(gT, m, 0))
    d1 = (Lv[1::4] - Lv[2::4]) / (2 * h)
    d2 = (Lv[3::4] - Lv[4::4]) / (4 * h)
    fd = (4 * d1 - d2) / 3
    scale = np.maximum(np.abs(fd), 1e-4 * np.abs(fd).max())
    err = np.abs(g[:NKPG] - fd) / scale
    assert err.max() <= 1e-6, (int(err.argmax()), err.max(), g[:NKPG], fd)


@pytest.mark.parametrize("rebuild_minv", [True, False])
@pytest.mark.parametrize("model", MODELS)
def test_gkp_against_forward_mode(B, L, model, rebuild_minv):
    e = _engine(B, model, True)
    H = 30
    ph = _phys(B, L, 1, 21)[0]
    kp = B.derive_params(B.with_minv(ph) if rebuild_minv else ph)
    z0, U = _problem(e, 1, H + 1, 22)
    X = np.zeros((H + 1, e.nx))
    X[0] = z0[0, :e.nx]
    X[1:] = X[0] + 0.01 * np.random.default_rng(23).standard_normal((H, e.nx))
    Us = U[:, 0]
    params = ["added", "lin", "quad", "current"]
    ref = e.multistep_se_grad(X, Us, [H], ph, params, dt=DT, integrator="rk4", rebuild_minv=rebuild_minv)
    x0 = torch.from_numpy(X[:1]).to(e.device)
    with e._coefficients(torch.from_numpy(kp).to(e.device)):
        xH = e.rollout(x0, Us[:H], dt=DT, integrator="rk4").xT.cpu().numpy()
        gzT = np.zeros((1, e.nz))
        gzT[0, :e.nx] = 2.0 * (xH[0] - X[H])
        r = e.rollout_vjp(x0, Us[:H], gzT=gzT, dt=DT, integrator="rk4", coef=True)
    D = B.coefficient_directions(ph, params, rebuild_minv=rebuild_minv)
    got = D @ r.gkp.cpu().numpy()[0]
    assert _normwise(got, ref.grad.cpu().numpy()[0]) <= 1e-9


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_state_and_input_gradients_equal_rollout_vjp(B, model, integ, cur):
    e = _engine(B, model, cur)
    n, T, stride = 33, 40, 4
    z0, U = _problem(e, n, T, 31)
    gt, gT = _cot(e, n, T, stride, 32)
    a = _vjp(e, z0, U, integ, gtraj=gt, gzT=gT, stride=stride)
    b = _vjp(e, z0, U, integ, gtraj=gt, gzT=gT, stride=stride, coef=True)
    # the coef build evaluates the same expressions, but the coefficient cotangent reuses some of their products
    # (e_i nur_i, the current's rotation, the quaternion's R entries), and the compiler does not fuse a product with a
    # second use into an FMA: with a current and for quat13, gx0 and gU agree to rounding rather than bit for bit
    for x, y in ((_gz0(e, a), _gz0(e, b)), (a.gU, b.gU), (a.z, b.z)):
        assert _normwise(y.cpu(), x.cpu()) <= 1e-13


@pytest.mark.parametrize("integ", ["rk4", "euler"])
@pytest.mark.parametrize("model", MODELS)
def test_per_vehicle_table(B, L, model, integ):
    e = _engine(B, model)
    n, T, stride = 45, 36, 6
    z0, U = _problem(e, n, T, 41)
    gt, gT = _cot(e, n, T, stride, 42)
    ph = _phys(B, L, n, 43)
    ph[::3, L.PH_CURRENT:L.PH_CURRENT + 3] = 0.0
    e.set_vehicle_physical(ph)
    t = _vjp(e, z0, U, integ, gtraj=gt, gzT=gT, stride=stride, coef=True)
    # repeats: bit for bit
    t2 = _vjp(e, z0, U, integ, gtraj=gt, gzT=gT, stride=stride, coef=True)
    for x, y in ((t.gkp, t2.gkp), (_gz0(e, t), _gz0(e, t2)), (t.gU, t2.gU)):
        assert torch.equal(x, y)
    # vehicle i of the table call = a shared-coefficient call with table column i
    kp = B.derive_params(ph)
    for i in (0, 1, n - 1):
        with e._coefficients(torch.from_numpy(kp[i]).to(e.device)):
            s = _vjp(e, z0[i:i + 1], U[:, i:i + 1], integ, gtraj=gt[:, i:i + 1], gzT=gT[i:i + 1], stride=stride,
                     coef=True)
        assert _normwise(t.gkp[i].cpu(), s.gkp[0].cpu()) <= 1e-14
        assert _normwise(_gz0(e, t)[i].cpu(), _gz0(e, s)[0].cpu()) <= 1e-14
        assert _normwise(t.gU[:, i].cpu(), s.gU[:, 0].cpu()) <= 1e-14
    # vehicle permutation with the table columns permuted: bit for bit
    perm = np.random.default_rng(44).permutation(n)
    e.set_vehicle_physical(ph[perm])
    p = _vjp(e, z0[perm], U[:, perm], integ, gtraj=gt[:, perm], gzT=gT[perm], stride=stride, coef=True)
    pt = torch.from_numpy(perm).to(e.device)
    assert torch.equal(p.gkp, t.gkp[pt]) and torch.equal(_gz0(e, p), _gz0(e, t)[pt]) and torch.equal(p.gU, t.gU[:, pt])
    # shared and constant input layouts: bit for bit with the same inputs laid out per vehicle
    e.set_vehicle_physical(ph)
    Us = U[:, 0]
    a = _vjp(e, z0, Us, integ, gtraj=gt, gzT=gT, stride=stride, coef=True, u_layout="shared")
    b = _vjp(e, z0, np.repeat(Us[:, None], n, 1), integ, gtraj=gt, gzT=gT, stride=stride, coef=True)
    assert torch.equal(a.gkp, b.gkp) and torch.equal(a.gU, b.gU)
    c = _vjp(e, z0, (U[0], T), integ, gtraj=gt, gzT=gT, stride=stride, coef=True, u_layout="const")
    d = _vjp(e, z0, np.repeat(U[:1], T, 0), integ, gtraj=gt, gzT=gT, stride=stride, coef=True)
    assert torch.equal(c.gkp, d.gkp) and torch.equal(c.gU, d.gU)


@pytest.mark.parametrize("model", MODELS)
def test_chaining(B, L, model):
    e = _engine(B, model, True)
    n, T, stride, t1 = 29, 48, 6, 18
    z0, U = _problem(e, n, T, 51)
    gt, gT = _cot(e, n, T, stride, 52)
    full = _vjp(e, z0, U, "rk4", gtraj=gt, gzT=gT, stride=stride, coef=True)
    first = _vjp(e, z0, U[:t1], "rk4", coef=True)                     # z_{t1}
    zm = first.z.cpu().numpy()
    late = _vjp(e, zm, U[t1:], "rk4", gtraj=gt[t1 // stride:], gzT=gT, stride=stride, coef=True)
    early = _vjp(e, z0, U[:t1], "rk4", gtraj=gt[:t1 // stride], gzT=_gz0(e, late), stride=stride, coef=True)
    assert torch.equal(_gz0(e, early), _gz0(e, full))
    assert torch.equal(torch.cat([early.gU, late.gU]), full.gU)
    assert _normwise((early.gkp + late.gkp).cpu(), full.gkp.cpu()) <= 1e-13


@pytest.mark.parametrize("model", MODELS)
def test_rollout_diff_gradcheck(B, L, model):
    e = _engine(B, model)
    n, T = 2, 6
    z0, U = _problem(e, n, T, 61)
    dev = e.device
    x0 = torch.from_numpy(z0[:, :e.nx]).to(dev)
    Ut = torch.from_numpy(U).to(dev)
    kp0 = torch.from_numpy(B.derive_params(_phys(B, L, n, 62))).to(dev)

    def f(kp):
        traj, xT, lagT = e.rollout_diff(x0, Ut, dt=DT, stride=2, kp=kp)
        return (traj, xT) if lagT is None else (traj, xT, lagT)

    assert torch.autograd.gradcheck(f, (kp0[0].clone().requires_grad_(),), eps=1e-6, atol=1e-6, rtol=1e-5)
    assert torch.autograd.gradcheck(f, (kp0.clone().requires_grad_(),), eps=1e-6, atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("model", MODELS)
def test_physical_gradient_through_derive_params_torch(B, L, model):
    e = _engine(B, model)
    n, T = 3, 30
    z0, U = _problem(e, n, T, 71)
    dev = e.device
    x0 = torch.from_numpy(z0[:, :e.nx]).to(dev)
    Ut = torch.from_numpy(U).to(dev)
    w = torch.from_numpy(np.random.default_rng(72).standard_normal((n, e.nx))).to(dev)
    ph0 = _phys(B, L, 1, 73)[0]
    ph = torch.from_numpy(ph0).to(dev).requires_grad_()
    _, xT, _ = e.rollout_diff(x0, Ut, dt=DT, stride=0, kp=B.derive_params_torch(ph))
    (xT * w).sum().backward()
    g = ph.grad.cpu().numpy()
    base = e.phys.copy()
    sel = [L.PH_M, L.PH_B, L.PH_XB + 2, L.PH_ADDED, L.PH_ADDED + 4, L.PH_LIN + 1, L.PH_QUAD + 2, L.PH_CURRENT]
    for i in sel:
        hh = 1e-6 * max(abs(ph0[i]), 0.1)
        vals = []
        for s in (1, -1):
            p = ph0.copy()
            p[i] += s * hh
            e.set_physical(B.with_minv(p))
            vals.append(float((e.rollout(x0, Ut, dt=DT).xT * w).sum()))
        fd = (vals[0] - vals[1]) / (2 * hh)
        assert abs(g[i] - fd) <= 1e-6 * max(abs(fd), 1e-3 * np.abs(g).max()), (i, g[i], fd)
    e.set_physical(base)


@pytest.mark.parametrize("table", [False, True])
def test_engine_coefficients_are_restored(B, L, table):
    e = _engine(B, "thruster8", True)
    n, T = 8, 12
    z0, U = _problem(e, n, T, 81)
    dev = e.device
    x0 = torch.from_numpy(z0[:, :e.nx]).to(dev)
    Ut = torch.from_numpy(U).to(dev)
    if table:
        e.set_vehicle_physical(_phys(B, L, n, 82))

    def probe():
        return e.rollout(x0, Ut, dt=DT, stride=3).traj.clone()

    ref = probe()
    kps = [torch.from_numpy(B.derive_params(_phys(B, L, 1, 83)[0])).to(dev),
           torch.from_numpy(B.derive_params(_phys(B, L, n, 84))).to(dev)]
    for kp in kps:
        k = kp.clone().requires_grad_()
        traj, xT, lagT = e.rollout_diff(x0, Ut, dt=DT, stride=3, kp=k)
        assert torch.equal(probe(), ref)
        assert not torch.equal(traj, ref)
        (traj.sum() + xT.sum() + lagT.sum()).backward()
        assert torch.equal(probe(), ref) and k.grad is not None
        with pytest.raises(ValueError):
            e.rollout_diff(x0, Ut[:, :n - 1], dt=DT, stride=3, kp=k)
        assert torch.equal(probe(), ref)
    with pytest.raises(ValueError):
        e.rollout_diff(x0, Ut, dt=DT, stride=3, kp=kps[0].float())


def test_health_counts_non_finite(B, L):
    e = _engine(B, "wrench12")
    n, T = 130, 10
    z0, U = _problem(e, n, T, 91)
    z0[5, 7] = np.nan
    r = _vjp(e, z0, U, "rk4", gzT=np.ones((n, e.nz)), coef=True, health=True)
    assert int(r.health[0]) == 1 and not torch.isfinite(r.gkp[5]).all()
    z0[5, 7] = 0.1
    ph = _phys(B, L, n, 92)
    ph[77, L.PH_LIN] = np.inf
    e.set_vehicle_physical(ph)
    r = _vjp(e, z0, U, "rk4", gzT=np.ones((n, e.nz)), coef=True, health=True)
    assert int(r.health[0]) == 1
    assert torch.isfinite(r.gkp[torch.arange(n, device=e.device) != 77]).all()


def _coef_desc(L, e, n, T, bufs, need):
    z0, U, gz0, gU, ws, gkp = bufs
    d = L.RolloutVjpDesc()
    d.struct_size = C.sizeof(L.RolloutVjpDesc)
    d.integrator = L.RK4
    d.n, d.steps, d.dt = n, T, DT
    d.z0_dev, d.u_dev = z0.data_ptr(), U.data_ptr()
    d.u_stride_t, d.u_stride_n = n * U.shape[2], U.shape[2]
    d.gz0_dev, d.gu_dev = gz0.data_ptr(), gU.data_ptr()
    d.workspace_dev, d.workspace_bytes = ws.data_ptr(), need
    dc = L.RolloutVjpCoefDesc()
    dc.struct_size = C.sizeof(L.RolloutVjpCoefDesc)
    dc.vjp = d
    dc.gkp_dev = gkp.data_ptr()
    return dc


def test_refusals(B, L):
    n, T = 4, 3
    nkp = L.NKP

    def bufs(nz, nu, dtype=torch.float64):
        dev = torch.device("cuda", torch.cuda.current_device())
        return (torch.zeros(n, nz, dtype=dtype, device=dev), torch.zeros(T, n, nu, dtype=dtype, device=dev),
                torch.full((n, nz), 7.0, dtype=dtype, device=dev), torch.full((T, n, nu), 7.0, dtype=dtype, device=dev),
                torch.empty(n * T * nz, dtype=torch.float64, device=dev),
                torch.full((nkp, n), 7.0, dtype=torch.float64, device=dev))

    def refused(e, nz, nu, match, edit=None, dtype=torch.float64, code=None):
        b = bufs(nz, nu, dtype)
        dc = _coef_desc(L, e, n, T, b, n * T * nz * 8)
        if edit:
            edit(dc)
        rc = L.lib.brov_rollout_vjp_coef(e._h, C.byref(dc), None)
        torch.cuda.synchronize()
        assert rc != 0 and match in L.lib.brov_last_error().decode(), (rc, L.lib.brov_last_error())
        for t in (b[2], b[3], b[5]):
            assert bool((t == 7.0).all())

    refused(B.Engine("thruster8", "f32"), 30, 8, "fp64", dtype=torch.float32)
    refused(B.Engine("di12_u8", "f64"), 12, 8, "double-integrator")
    e = B.Engine("wrench12", "f64")
    e.set_wrench_lag1(True, 0.1)
    refused(e, 12, 6, "first-order")
    e = B.Engine("thruster8", "f64")
    e.set_vehicle_physical(np.repeat(B.default_physical()[None], n + 1, axis=0))
    refused(e, 30, 8, "vehicle table has 5 rows")
    e = B.Engine("thruster8", "f64")
    refused(e, 30, 8, "gkp", edit=lambda dc: setattr(dc, "gkp_dev", None))
    refused(e, 30, 8, "size mismatch", edit=lambda dc: setattr(dc, "struct_size", dc.struct_size - 8))
    refused(e, 30, 8, "size mismatch", edit=lambda dc: setattr(dc.vjp, "struct_size", dc.vjp.struct_size + 8))
    refused(e, 30, 8, "workspace", edit=lambda dc: setattr(dc.vjp, "workspace_bytes", 8))
    # the table of n rows is accepted, and rollout_vjp without coef keeps refusing it
    e.set_vehicle_physical(np.repeat(B.default_physical()[None], n, axis=0))
    r = e.rollout_vjp(torch.zeros(n, 12), torch.zeros(T, n, 8), coef=True)
    assert r.gkp.shape == (n, nkp)
    with pytest.raises(B.BrovError, match="per-vehicle"):
        e.rollout_vjp(torch.zeros(n, 12), torch.zeros(T, n, 8))
