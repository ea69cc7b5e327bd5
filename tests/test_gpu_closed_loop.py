"""GPU tests of the closed-loop rollout (brov_closed_loop through Engine.closed_loop): the recorded inputs replay through
the open-loop rollout, an independent closed loop on the numpy oracle agrees, the accumulated LQR cost tends to the
Riccati form, a TVLQR built on linearize tracks per-vehicle nominals, operand layouts / chunking / permutation / run
order / a 2 pi goal offset / edge sizes leave results unchanged, per-vehicle coefficient tables match shared-coefficient
calls, the health counters and argument checks work, and operands above 2^31 elements are indexed correctly."""
import ctypes as C
import functools

import numpy as np
import pytest
import scipy.linalg
import torch

from oracle import fossen_np as O

pytestmark = pytest.mark.gpu

DT = 0.02
MODELS = ("thruster8", "wrench12", "quat13")
CASES = [(m, i, c) for m in MODELS for i in ("rk4", "euler") for c in (False, True)]
IDS = [f"{m}-{i}-{'current' if c else 'still'}" for m, i, c in CASES]
CURRENT = (0.12, -0.07, 0.05)
TOL = {"f64": 1e-12, "f32": 1e-5}
WRENCH_BOUND = np.array([25.0, 25.0, 25.0, 2.0, 2.0, 2.0])


@pytest.fixture(scope="module")
def B():
    import bluerov2_dynamics_b200 as b
    return b


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200 import _lib
    return _lib


def _engine(B, model, current=False, dtype="f64"):
    return B.Engine(model, dtype, current=CURRENT if current else None)


def _normwise(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _np(t):
    return t.double().cpu().numpy()


def _bounds(model):
    return (-1.0, 1.0) if model == "thruster8" else (-WRENCH_BOUND, WRENCH_BOUND)


@functools.lru_cache(maxsize=None)
def _lqr(model, integ, cur):
    """hover trim at 1 m depth (minimum-norm Newton on Phi(z, u) = z) and a discrete LQR about it:
    (z*, u*, K, P, Q, R), numpy fp64"""
    import bluerov2_dynamics_b200 as b
    e = b.Engine(model, "f64", current=CURRENT if cur else None)
    nx, nz, nu = e.nx, e.nz, e.nu
    z = np.zeros(nz)
    z[2] = 1.0
    if nx == 13:
        z[3] = 1.0
    u = np.zeros(nu)
    thr = model == "thruster8"
    for _ in range(20):
        r = e.linearize(z[None, :nx], u[None], dt=DT, integrator=integ, lag0=z[None, nx:] if thr else None,
                        lag_repr="projected", want_traj=False)
        F = r.z[0].cpu().numpy() - z
        if np.linalg.norm(F) < 1e-13:
            break
        M = np.concatenate([r.A[0, 0].cpu().numpy() - np.eye(nz), r.B[0, 0].cpu().numpy()], axis=1)
        s = np.linalg.lstsq(M, -F, rcond=None)[0]
        z += s[:nz]
        u += s[nz:]
    r = e.linearize(z[None, :nx], u[None], dt=DT, integrator=integ, lag0=z[None, nx:] if thr else None,
                    lag_repr="projected", want_traj=False)
    A, Bm = r.A[0, 0].cpu().numpy(), r.B[0, 0].cpu().numpy()
    ang = 3 if nx == 12 else 4
    Q = np.diag([10.0] * 3 + [5.0] * ang + [1.0] * 6 + [1e-6] * (nz - nx))
    R = (0.5 if thr else 0.01) * np.eye(nu)
    P = scipy.linalg.solve_discrete_are(A, Bm, Q, R)
    K = np.linalg.solve(R + Bm.T @ P @ Bm, Bm.T @ P @ A)
    return z, u, K, P, Q, R


def _start(e, zs, n, seed, scale=1.0):
    """n vehicles about the trim zs: position, attitude and rate perturbations (z [n, NZ], numpy)"""
    rng = np.random.default_rng(seed)
    z = np.tile(zs, (n, 1))
    z[:, 0:3] += scale * rng.uniform(-0.5, 0.5, (n, 3))
    if e.nx == 12:
        z[:, 3:6] += scale * rng.uniform(-0.3, 0.3, (n, 3))
        z[:, 6:12] += scale * rng.uniform(-0.2, 0.2, (n, 6))
    else:
        ang = scale * rng.uniform(-0.3, 0.3, (n, 3))
        z[:, 3:7] = O.euler_to_quat(ang[:, 0], ang[:, 1], ang[:, 2])
        z[:, 7:13] += scale * rng.uniform(-0.2, 0.2, (n, 6))
    return z


def _cl(e, z0, K, zr, ur, **kw):
    lo, hi = _bounds(e.model)
    kw.setdefault("u_min", lo)
    kw.setdefault("u_max", hi)
    thr = e.model == "thruster8"
    return e.closed_loop(z0[:, :e.nx], K, zr, ur, lag0=z0[:, e.nx:] if thr else None, lag_repr="projected", **kw)


@pytest.mark.parametrize("dtype", ("f64", "f32"))
@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_recorded_inputs_replay_through_the_rollout(B, model, integ, cur, dtype):
    e = _engine(B, model, cur, dtype)
    zs, us, K, *_ = _lqr(model, integ, cur)
    n, T = 300, 200
    z0 = _start(e, zs, n, 1)
    r = _cl(e, z0, K, zs, us, steps=T, dt=DT, integrator=integ, stride=1, want_u=True, health=True)
    assert r.health.tolist() == [0, 0]
    thr = model == "thruster8"
    o = e.rollout(z0[:, :e.nx], r.u_traj, dt=DT, integrator=integ, stride=1, lag_repr="projected",
                  lag0=z0[:, e.nx:] if thr else None)
    err = _normwise(_np(r.z_traj[:, :, :e.nx]), _np(o.traj))
    bitwise = torch.equal(r.z_traj[:, :, :e.nx], o.traj)
    print(f"{model} {integ} current={cur} {dtype}: replay normwise {err:.3e}, bitwise {bitwise}")
    assert err <= TOL[dtype]
    if thr:
        assert _normwise(_np(r.z[:, e.nx:]), _np(o.lag)) <= TOL[dtype]
    # zero gain: the open-loop rollout of clamp(u_ref), here a time-varying shared reference that leaves the bounds
    rng = np.random.default_rng(2)
    lo, hi = _bounds(model)
    Ur = us + 3.0 * np.asarray(hi) * O.smooth_inputs(rng, T, e.nu, sigma=0.2)
    r0 = _cl(e, z0, np.zeros_like(K), zs, Ur, dt=DT, integrator=integ, stride=1, want_u=True)
    Uc = np.clip(Ur, lo, hi)
    assert np.any(Uc != Ur)
    assert torch.equal(r0.u_traj, e.tensor(np.broadcast_to(Uc[:, None], (T, n, e.nu))))
    o0 = e.rollout(z0[:, :e.nx], Uc, dt=DT, integrator=integ, stride=1, lag_repr="projected",
                   lag0=z0[:, e.nx:] if thr else None)
    assert _normwise(_np(r0.z_traj[:, :, :e.nx]), _np(o0.traj)) <= TOL[dtype]


@pytest.mark.parametrize("dtype", ("f64", "f32"))
@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_agrees_with_a_closed_loop_on_the_numpy_oracle(B, model, integ, cur, dtype):
    e = _engine(B, model, cur, dtype)
    zs, us, K, *_ = _lqr(model, integ, cur)
    n, T = 48, 500
    thr = model == "thruster8"
    rng = np.random.default_rng(3)
    x = _start(e, zs, n, 4, scale=1.6)[:, :e.nx]
    m = O.Model(model, DT, O.default_params(current=CURRENT if cur else (0.0, 0.0, 0.0)))
    lo, hi = _bounds(model)
    if thr:
        # per-thruster lag about the trim's steady state, projected for the kernel
        Lag = np.tile(e.rollout(np.zeros((1, 12)), (us[None], 2000), dt=DT, integrator=integ,
                                u_layout="const").lag.cpu().numpy().reshape(1, 8, 3), (n, 1, 1))
        Lag += rng.uniform(-0.05, 0.05, Lag.shape)
        alloc = O.thruster_geometry()[2]
        z0 = np.concatenate([x, np.einsum("ci,nik->nck", alloc, Lag).reshape(n, 18)], axis=1)
    else:
        Lag = None
        z0 = x
    r = _cl(e, z0, K, zs, us, steps=T, dt=DT, integrator=integ, stride=1, want_u=True)
    zt = np.zeros((T, n, e.nz))
    clamped = 0
    for k in range(T):
        z = np.concatenate([x, np.einsum("ci,nik->nck", alloc, Lag).reshape(n, 18)], axis=1) if thr else x
        dz = z - zs
        if e.nx == 12:
            dz[:, 3:6] -= 2 * np.pi * np.rint(dz[:, 3:6] / (2 * np.pi))
        v = us - dz @ K.T
        u = np.clip(v, lo, hi)
        clamped += int(np.sum(u != v))
        x, Lag = O.step(m, integ, x, u, Lag)
        zt[k] = np.concatenate([x, np.einsum("ci,nik->nck", alloc, Lag).reshape(n, 18)], axis=1) if thr else x
    assert clamped > 0
    tol = 1e-10 if dtype == "f64" else 1e-4
    err = _normwise(_np(r.z_traj), zt)
    print(f"{model} {integ} current={cur} {dtype}: oracle normwise {err:.3e}, {clamped} clamped channel-steps")
    assert err <= tol


def test_lqr_cost_tends_to_the_riccati_form(B):
    e = _engine(B, "thruster8")
    zs, us, K, P, Q, R = _lqr("thruster8", "rk4", False)
    rng = np.random.default_rng(5)
    d = rng.standard_normal((8, e.nz))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    dev = []
    for eps in (1e-2, 1e-3, 1e-4):
        z0 = zs + eps * d
        r = _cl(e, z0, K, zs, us, steps=6000, dt=DT, cost_q=np.diag(Q), cost_r=np.diag(R))
        ratio = _np(r.cost) / np.einsum("ni,ij,nj->n", eps * d, P, eps * d)
        dev.append(np.abs(ratio - 1))
    dev = np.array(dev)
    print("|cost / dz'P dz - 1| at eps = 1e-2, 1e-3, 1e-4:", dev.max(1))
    assert np.all(dev[0] < 0.1)
    assert np.all(dev[2] < 1e-3)
    # the worst vehicle's deviation falls in proportion to eps; no vehicle's falls slower than that
    worst = dev.max(1)
    assert np.all((worst[:-1] / worst[1:] > 5) & (worst[:-1] / worst[1:] < 20)), worst
    assert np.all(dev[:-1] / dev[1:] > 3), dev


def test_tvlqr_about_per_vehicle_nominals(B):
    e = _engine(B, "thruster8")
    zs, us, K0, P0, Q, R = _lqr("thruster8", "rk4", False)
    n, T = 64, 250
    rng = np.random.default_rng(6)
    zn0 = _start(e, zs, n, 7, scale=0.3)
    Un = np.clip(us + O.smooth_inputs(rng, T, 8, n=n, sigma=0.05), -0.9, 0.9)
    lin = e.linearize(zn0[:, :12], Un, dt=DT, lag0=zn0[:, 12:], lag_repr="projected")
    znom = torch.cat([e.tensor(zn0)[None], lin.z_traj[:-1]])              # [T, n, NZ]: z at the start of step k
    A, Bm = lin.A, lin.B
    Qt, Rt = e.tensor(Q), e.tensor(R)
    Pk = Qt.expand(n, -1, -1).clone()
    Ks = torch.empty((T, n, 8, e.nz), dtype=torch.float64, device="cuda")
    for k in range(T - 1, -1, -1):                                         # batched backward Riccati pass
        BtP = Bm[k].transpose(1, 2) @ Pk
        Kk = torch.linalg.solve(Rt + BtP @ Bm[k], BtP @ A[k])
        Ks[k] = Kk
        Acl = A[k] - Bm[k] @ Kk
        Pk = Qt + A[k].transpose(1, 2) @ Pk @ Acl
        Pk = 0.5 * (Pk + Pk.transpose(1, 2))
    Ut = e.tensor(Un)
    on = _cl(e, zn0, Ks, znom, Ut, dt=DT, u_min=-1.0, u_max=1.0)
    assert _normwise(_np(on.z), _np(lin.z)) <= 1e-10
    zp = zn0.copy()
    zp[:, 0:3] += rng.uniform(-0.15, 0.15, (n, 3))
    zp[:, 3:6] += rng.uniform(-0.1, 0.1, (n, 3))
    zp[:, 6:12] += rng.uniform(-0.1, 0.1, (n, 6))
    cl = _cl(e, zp, Ks, znom, Ut, dt=DT, u_min=-1.0, u_max=1.0)
    ol = e.rollout(zp[:, :12], Ut, dt=DT, lag0=zp[:, 12:], lag_repr="projected")
    e_cl = torch.linalg.norm(cl.z[:, :12] - lin.z[:, :12], dim=1)
    e_ol = torch.linalg.norm(ol.xT - lin.z[:, :12], dim=1)
    print(f"TVLQR final error: median closed {e_cl.median():.3e}, open {e_ol.median():.3e}")
    assert torch.all(e_cl < e_ol)


@pytest.mark.parametrize("model", MODELS)
def test_layouts_chunks_reproducibility_permutation_and_edges(B, model):
    e = _engine(B, model, True)
    zs, us, K, *_ = _lqr(model, "rk4", True)
    thr = model == "thruster8"
    n, T = 1000, 40
    z0 = _start(e, zs, n, 8)
    kw = dict(dt=DT, integrator="rk4", stride=1, want_u=True, cost_q=0.5, cost_r=0.25, health=True)
    ref = _cl(e, z0, K, zs, us, steps=T, **kw)
    # the four layouts of every operand, holding the same values
    Kt, zt, ut = e.tensor(K), e.tensor(zs), e.tensor(us)
    forms = {"const_shared": lambda t: t, "shared": lambda t: t.expand(T, *t.shape),
             "const": lambda t: t.expand(n, *t.shape), "tnc": lambda t: t.expand(T, n, *t.shape)}
    for kl, kf in forms.items():
        for rl, rf in forms.items():
            r = _cl(e, z0, kf(Kt), rf(zt), rf(ut), steps=T, k_layout=kl, ref_layout=rl, **kw)
            for a, b in ((r.z, ref.z), (r.z_traj, ref.z_traj), (r.u_traj, ref.u_traj), (r.cost, ref.cost)):
                assert torch.equal(a, b), (kl, rl)
    # run to run
    r2 = _cl(e, z0, K, zs, us, steps=T, **kw)
    assert torch.equal(r2.z, ref.z) and torch.equal(r2.cost, ref.cost) and torch.equal(r2.z_traj, ref.z_traj)
    # two chunks carrying z and the cost = one call (time-varying references sliced between them)
    rng = np.random.default_rng(9)
    Zr = zs + 0.05 * rng.standard_normal((T, n, e.nz))
    Ur = us + 0.05 * rng.standard_normal((T, e.nu))
    one = _cl(e, z0, K, Zr, Ur, **kw)
    a = _cl(e, z0, K, Zr[:15], Ur[:15], **kw)
    zc = _np(a.z)
    b = _cl(e, zc, K, Zr[15:], Ur[15:], cost=a.cost, cost_accumulate=True, **kw)
    assert torch.equal(b.z, one.z) and torch.equal(b.cost, one.cost)
    assert torch.equal(torch.cat([a.z_traj, b.z_traj]), one.z_traj)
    # permuting the vehicles permutes the results (per-vehicle operands permuted with them)
    perm = rng.permutation(n)
    p = _cl(e, z0[perm], K, Zr[:, perm], Ur, **kw)
    assert torch.equal(p.z, one.z[perm]) and torch.equal(p.cost, one.cost[perm])
    assert torch.equal(p.z_traj, one.z_traj[:, perm])
    # edge sizes: N = 1 and ragged N give the rows of the large call
    for m in (1, 129):
        s = _cl(e, z0[:m], K, Zr[:, :m], Ur, **kw)
        assert torch.equal(s.z, one.z[:m]) and torch.equal(s.z_traj, one.z_traj[:, :m])
    # steps = 0 copies z0 (cost zeroed); n = 0 is a no-op
    s0 = _cl(e, z0, K, zs, us, steps=0, cost_q=1.0)
    assert torch.equal(s0.z, e.tensor(z0)) and torch.all(s0.cost == 0)
    s00 = _cl(e, z0[:0], K, zs, us, steps=5)
    assert s00.z.shape == (0, e.nz)
    # a yaw goal offset by 2 pi (Euler-angle models) gives the same trajectory
    if e.nx == 12:
        zs2 = zs.copy()
        zs2[5] += 2 * np.pi
        w = _cl(e, z0, K, zs2, us, steps=T, **kw)
        assert _normwise(_np(w.z_traj), _np(ref.z_traj)) <= 1e-12


@pytest.mark.parametrize("dtype", ("f64", "f32"))
@pytest.mark.parametrize("model", MODELS)
def test_per_vehicle_coefficients_match_shared_calls(B, model, dtype):
    zs, us, K, *_ = _lqr(model, "rk4", False)
    e = _engine(B, model, False, dtype)
    n, T = 6, 120
    z0 = _start(e, zs, n, 10)
    rng = np.random.default_rng(11)
    table = np.tile(B.default_physical(), (n, 1))
    for grp in ("added", "lin", "quad"):
        idx = B.engine.PARAM_GROUPS[grp]
        table[:, idx] *= rng.uniform(0.8, 1.2, (n, len(idx)))
    table[2:4, 33:36] = CURRENT                       # some rows with an ocean current
    table = B.with_minv(table)
    e.set_vehicle_physical(table)
    r = _cl(e, z0, K, zs, us, steps=T, dt=DT, stride=10)
    e.set_vehicle_physical(None)
    for i in range(n):
        e.set_physical(table[i])
        s = _cl(e, z0[i:i + 1], K, zs, us, steps=T, dt=DT, stride=10)
        assert _normwise(_np(r.z_traj[:, i:i + 1]), _np(s.z_traj)) <= TOL[dtype], i


@pytest.mark.parametrize("model", MODELS)
def test_health_counters(B, model):
    e = _engine(B, model)
    zs, us, K, *_ = _lqr(model, "rk4", False)
    n = 50
    z0 = _start(e, zs, n, 12)
    r = _cl(e, z0, K, zs, us, steps=10, dt=DT, health=True)
    assert r.health.tolist() == [0, 0]
    z0[[3, 17], 7] = np.nan
    if e.nx == 12:
        z0[[4, 20, 41], 4] = np.pi / 2 - 1e-4         # |cos theta| = 1e-4 < 1e-3
    r = _cl(e, z0, K, zs, us, steps=1, dt=DT, health=True, stride=1, want_u=True)
    assert r.health.tolist()[0] == 2 and r.health.tolist()[1] == (3 if e.nx == 12 else 0)
    assert torch.all(torch.isnan(r.u_traj[0, [3, 17]]))          # the clamp does not hide a NaN
    assert torch.all(torch.isnan(r.z[[3, 17]]).any(1))


def test_unsupported_and_invalid_calls(B, L):
    zs, us, K, *_ = _lqr("thruster8", "rk4", False)
    x = np.tile(zs[:12], (4, 1))
    di = B.Engine("di12_u8", "f64")
    di.set_di_gains(np.full((8, 3), 0.1), np.full((8, 3), 0.1))
    d = L.ClosedLoopDesc()
    d.struct_size = C.sizeof(L.ClosedLoopDesc)
    assert L.lib.brov_closed_loop(di._h, C.byref(d), None) == -4
    w = B.Engine("wrench12", "f64")
    w.set_wrench_lag1(True, 0.1)
    assert L.lib.brov_closed_loop(w._h, C.byref(d), None) == -4
    e = B.Engine("thruster8", "f64")
    z = e.tensor(np.tile(zs, (4, 1)))
    zo = torch.empty_like(z)
    Kt, zr, ur = e.tensor(K), e.tensor(zs), e.tensor(us)

    def desc(**kw):
        d = L.ClosedLoopDesc()
        d.struct_size = C.sizeof(L.ClosedLoopDesc)
        d.n, d.steps, d.dt = 4, 3, DT
        d.z0_dev, d.z_out_dev = z.data_ptr(), zo.data_ptr()
        d.K_dev, d.z_ref_dev, d.u_ref_dev = Kt.data_ptr(), zr.data_ptr(), ur.data_ptr()
        for r in range(8):
            d.u_min[r], d.u_max[r] = -1.0, 1.0
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    def rc(**kw):
        return L.lib.brov_closed_loop(e._h, C.byref(desc(**kw)), None)

    assert rc() == 0
    assert rc(struct_size=8) == -1
    assert rc(n=-1) == -1
    assert rc(steps=-1) == -1
    assert rc(dt=0.0) == -1 and rc(dt=-0.02) == -1
    assert rc(integrator=7) == -1
    for s in ("K_stride_t", "K_stride_n", "z_ref_stride_t", "z_ref_stride_n", "u_ref_stride_t", "u_ref_stride_n"):
        assert rc(**{s: -1}) == -1, s
    for p in ("K_dev", "z_ref_dev", "u_ref_dev"):
        assert rc(**{p: None}) == -1, p
        assert rc(**{p: None, "steps": 0}) == 0, p
        assert rc(**{p: None, "n": 0}) == 0, p
    d = desc()
    d.u_min[5] = 2.0
    assert L.lib.brov_closed_loop(e._h, C.byref(d), None) == -1
    d = desc()
    d.u_max[0] = float("nan")
    assert L.lib.brov_closed_loop(e._h, C.byref(d), None) == -1
    d = desc()
    d.u_min[7] = float("nan")
    assert L.lib.brov_closed_loop(e._h, C.byref(d), None) == -1
    assert rc(traj_dev=zo.data_ptr(), stride=0) == -1
    assert rc(u_traj_dev=zo.data_ptr(), stride=0) == -1
    e.set_vehicle_physical(np.tile(B.default_physical(), (5, 1)))
    assert rc() == -1                                  # table of 5 rows, call of 4
    e.set_vehicle_physical(None)
    with pytest.raises(B.BrovError, match="-1"):
        e.closed_loop(x, K, zs, us, steps=5, dt=-0.02)
    with pytest.raises(ValueError):
        e.closed_loop(x, K, zs, us)                    # no time-varying operand and no steps=
    with pytest.raises(ValueError):
        e.closed_loop(x, np.tile(K, (3, 1, 1)), np.tile(zs, (4, 1)), us)   # T = 3 against T = 4
    with pytest.raises(ValueError):
        e.closed_loop(x, K[:, :12], zs, us, steps=5)


def test_stride_beyond_int_range_takes_no_snapshot(B, L):
    # a 64-bit stride past INT_MAX is a snapshot interval longer than any call: 3 steps take none, and the trajectory
    # buffer (sized here for 3 snapshots) stays as it was
    zs, us, K, *_ = _lqr("thruster8", "rk4", False)
    e = B.Engine("thruster8", "f64")
    n, steps = 4, 3
    z = e.tensor(np.tile(zs, (n, 1)))
    zo = torch.empty_like(z)
    Kt, zr, ur = e.tensor(K), e.tensor(zs), e.tensor(us)
    traj = torch.full((steps, n, e.nz), float("nan"), device="cuda", dtype=torch.float64)
    d = L.ClosedLoopDesc()
    d.struct_size = C.sizeof(L.ClosedLoopDesc)
    d.n, d.steps, d.dt = n, steps, DT
    d.z0_dev, d.z_out_dev = z.data_ptr(), zo.data_ptr()
    d.K_dev, d.z_ref_dev, d.u_ref_dev = Kt.data_ptr(), zr.data_ptr(), ur.data_ptr()
    for r in range(8):
        d.u_min[r], d.u_max[r] = -1.0, 1.0
    d.traj_dev, d.stride = traj.data_ptr(), 2 ** 32 + 1
    assert L.lib.brov_closed_loop(e._h, C.byref(d), None) == 0
    torch.cuda.synchronize()
    assert torch.isnan(traj).all()
    assert torch.isfinite(zo).all()


def test_full_size_per_vehicle_gains_above_2_31_elements(B):
    e = _engine(B, "thruster8")
    zs, us, K, *_ = _lqr("thruster8", "rk4", False)
    n, T = 65536, 140
    assert T * n * 8 * 30 > 2 ** 31
    z0 = _start(e, zs, n, 13)
    g = torch.Generator(device="cuda").manual_seed(14)
    Kt = e.tensor(K).expand(T, n, 8, 30).clone()
    Kt += 1e-3 * torch.randn(Kt.shape, dtype=torch.float64, device="cuda", generator=g)
    r = _cl(e, z0, Kt, zs, us, dt=DT, cost_q=1.0, health=True)
    assert r.health.tolist()[0] == 0
    m = 300
    s = _cl(e, z0[-m:], Kt[:, -m:], zs, us, dt=DT, cost_q=1.0)
    assert torch.equal(r.z[-m:], s.z) and torch.equal(r.cost[-m:], s.cost)
    del Kt, r
    torch.cuda.empty_cache()
