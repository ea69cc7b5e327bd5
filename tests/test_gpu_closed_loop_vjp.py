"""GPU tests of the reverse-mode gradients of closed-loop rollouts (brov_closed_loop_vjp through Engine.closed_loop_vjp /
closed_loop_diff): the result equals the explicit Jacobian chain over Engine.linearize with the feedback law formed in
torch, directional derivatives agree with central differences of Engine.closed_loop in every operand layout, the clamp
and the angle wrap have the derivative of the computed function, layouts, repeats, permutations and chaining behave as
the ABI states, per-vehicle tables match single-vehicle calls, gradcheck passes, and health counters, refusals, edge
sizes and a gain gradient above 2^31 elements behave."""
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
LAYOUTS = ("const_shared", "shared", "const", "tnc")
TWO_PI = 2.0 * np.pi


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


def _t(e, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device=e.device)


def _problem(e, n, T, seed):
    """z0 [n, NZ], per-(step, vehicle) K [T, n, NU, NZ], z_ref [T, n, NZ], u_ref [T, n, NU] (numpy), bounds [NU] and
    cost weights: moderate angles and velocities, references near z0, gains that saturate some channels"""
    rng = np.random.default_rng(seed)
    nz, nu, nx = e.nz, e.nu, e.nx
    x = np.zeros((n, nx))
    x[:, :3] = rng.uniform(-1, 1, (n, 3))
    ang = np.stack([rng.uniform(-0.4, 0.4, n), rng.uniform(-0.4, 0.4, n), rng.uniform(-3, 3, n)], axis=1)
    nu_ = np.concatenate([rng.uniform(-0.4, 0.4, (n, 3)), rng.uniform(-0.3, 0.3, (n, 3))], axis=1)
    if nx == 13:
        x[:, 3:7] = O.euler_to_quat(ang[:, 0], ang[:, 1], ang[:, 2])
        x[:, 7:] = nu_
    else:
        x[:, 3:6] = ang
        x[:, 6:] = nu_
    z0 = x
    if e.model == "thruster8":
        z0 = np.concatenate([x, e.project_lag(rng.uniform(-0.5, 0.5, (n, 24))).cpu().numpy()], axis=1)
    uscale = 1.0 if e.model == "thruster8" else 20.0
    K0 = rng.normal(0, 0.3 * uscale, (nu, nz)) / np.sqrt(nz)
    K = K0 + rng.normal(0, 0.05 * uscale, (T, n, nu, nz)) / np.sqrt(nz)
    zr = z0[None] + rng.normal(0, 0.2, (T, n, nz))
    if nx == 13:
        zr[..., 3:7] /= np.linalg.norm(zr[..., 3:7], axis=-1, keepdims=True)
    ur = rng.uniform(-0.4, 0.4, (T, n, nu)) * uscale
    bound = uscale * np.where(np.arange(nu) % 3 == 0, 0.35, 1.0)
    q = rng.uniform(0.5, 2.0, nz)
    r = rng.uniform(0.5, 2.0, nu) / uscale ** 2
    return z0, K, zr, ur, -bound, bound, q, r


def _layout(a, layout, T, n):
    """the operand a [T, n, ...] in `layout` (its first step / vehicle where a dimension is shared)"""
    return {"const_shared": a[0, 0], "shared": a[:, 0], "const": a[0], "tnc": a}[layout]


def _expand(a, layout, T, n):
    """operand in `layout` back to [T, n, ...]"""
    inner = a.shape[{"const_shared": 0, "shared": 1, "const": 1, "tnc": 2}[layout]:]
    lead = {"const_shared": (1, 1), "shared": (T, 1), "const": (1, n), "tnc": (T, n)}[layout]
    return a.reshape(lead + tuple(inner)).expand((T, n) + tuple(inner))


def _wrap(e, d):
    if e.nx == 12:
        d = d.clone()
        d[..., 3:6] = d[..., 3:6] - TWO_PI * torch.round(d[..., 3:6] / TWO_PI)
    return d


def _lin_chain(e, z0, K, zr, ur, lo, hi, q, r, gtraj, gzT, gc, stride, integ):
    """the explicit chain: linearize step by step with u_k formed in torch, then the transposed recursion"""
    T, n = K.shape[0], K.shape[1]
    nx, nz = e.nx, e.nz
    lo_t, hi_t, q_t, r_t = _t(e, lo), _t(e, hi), _t(e, q), _t(e, r)
    z = z0.clone()
    rec, sat = [], []
    for k in range(T):
        dz = _wrap(e, z - zr[k])
        v = ur[k] - torch.einsum("nrj,nj->nr", K[k], dz)
        m = ((v >= lo_t) & (v <= hi_t)).to(torch.float64)
        u = torch.minimum(torch.maximum(v, lo_t), hi_t)
        lag = z[:, nx:] if e.model == "thruster8" else None
        res = e.linearize(z[:, :nx].contiguous(), u.contiguous(), dt=DT, integrator=integ, lag0=lag,
                          lag_repr="projected", u_layout="step", want_traj=False)
        rec.append((res.A[0].clone(), res.B[0].clone(), dz, u, m))
        sat.append(1.0 - float(m.mean()))
        z = res.z.clone()
    lam = gzT.clone() if gzT is not None else torch.zeros((n, nz), dtype=torch.float64, device=e.device)
    if gtraj is not None and T % stride == 0:
        lam = lam + gtraj[T // stride - 1]
    gK, gzr, gur = torch.zeros_like(K), torch.zeros_like(zr), torch.zeros_like(ur)
    g2 = (2.0 * gc)[:, None]
    for k in range(T - 1, -1, -1):
        A, Bm, dz, u, m = rec[k]
        gu = torch.einsum("nzr,nz->nr", Bm, lam)
        gcu = g2 * r_t * (u - ur[k])
        gv = m * (gu + gcu)
        gK[k] = -gv[:, :, None] * dz[:, None, :]
        gdz = -torch.einsum("nrj,nr->nj", K[k], gv) + g2 * q_t * dz
        gzr[k] = -gdz
        gur[k] = gv - gcu
        lam = torch.einsum("nij,ni->nj", A, lam) + gdz
        if gtraj is not None and k > 0 and k % stride == 0:
            lam = lam + gtraj[k // stride - 1]
    return lam, gK, gzr, gur, z, float(np.mean(sat))


def _cotangents(e, n, T, stride, seed):
    rng = np.random.default_rng(seed)
    gt = _t(e, rng.normal(size=(T // stride, n, e.nz)))
    gT = _t(e, rng.normal(size=(n, e.nz)))
    gc = _t(e, rng.uniform(0.2, 1.0, n))
    return gt, gT, gc


def _call(e, z0, K, zr, ur, lo, hi, q, r, integ="rk4", kl="tnc", rl="tnc", **kw):
    nx = e.nx
    lag = z0[:, nx:] if e.model == "thruster8" else None
    return e.closed_loop_vjp(z0[:, :nx], K, zr, ur, dt=DT, integrator=integ, lag0=lag, lag_repr="projected",
                             k_layout=kl, ref_layout=rl, u_min=lo, u_max=hi, cost_q=q, cost_r=r, **kw)


def _gz0(e, res):
    return torch.cat([res.gx0, res.glag0], 1) if res.glag0 is not None else res.gx0


@pytest.mark.parametrize("stride", [1, 7])
@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_gradients_equal_the_explicit_chain_over_linearize(B, model, integ, cur, stride):
    e = _engine(B, model, cur)
    n, T = 5, 21
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 11)
    z0, K, zr, ur = _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur)
    gt, gT, gc = _cotangents(e, n, T, stride, 3)
    res = _call(e, z0, K, zr, ur, lo, hi, q, r, integ, gtraj=gt, gzT=gT, gcost=gc, stride=stride, health=True)
    lam, gK, gzr, gur, zT, sat = _lin_chain(e, z0, K, zr, ur, lo, hi, q, r, gt, gT, gc, stride, integ)
    assert 0.02 < sat < 0.9        # saturation is active on some channels, not on all
    assert _normwise(res.z.cpu(), zT.cpu()) < 1e-13
    assert _normwise(_gz0(e, res).cpu(), lam.cpu()) < 1e-12
    assert _normwise(res.gK.cpu(), gK.cpu()) < 1e-12
    assert _normwise(res.gz_ref.cpu(), gzr.cpu()) < 1e-12
    assert _normwise(res.gu_ref.cpu(), gur.cpu()) < 1e-12
    assert res.health.tolist() == [0, 0]


def _loss(e, z0, K, zr, ur, lo, hi, q, r, integ, kl, rl, gt, gT, gc, stride, T):
    nx = e.nx
    c = e.closed_loop(z0[:, :nx], K, zr, ur, dt=DT, integrator=integ, lag0=z0[:, nx:] if e.model == "thruster8" else None,
                      lag_repr="projected", k_layout=kl, ref_layout=rl, u_min=lo, u_max=hi, stride=stride,
                      cost_q=q, cost_r=r, steps=T)
    tot = (c.z * gT).sum() + (gc * c.cost).sum()
    if gt is not None:
        tot = tot + (c.z_traj * gt).sum()
    return float(tot)


def _margin(e, z0, K, zr, ur, lo, hi, integ, kl, rl, T, n):
    """the smallest distance of any v_k from a clamp bound along the closed loop"""
    nx = e.nx
    c = e.closed_loop(z0[:, :nx], K, zr, ur, dt=DT, integrator=integ, lag0=z0[:, nx:] if e.model == "thruster8" else None,
                      lag_repr="projected", k_layout=kl, ref_layout=rl, u_min=lo, u_max=hi, stride=1, steps=T)
    zs = torch.cat([z0[None], c.z_traj[:-1]], 0)
    Kx, zrx, urx = _expand(K, kl, T, n), _expand(zr, rl, T, n), _expand(ur, rl, T, n)
    v = urx - torch.einsum("tnrj,tnj->tnr", Kx, _wrap(e, zs - zrx))
    return float(torch.minimum((v - _t(e, lo)).abs(), (v - _t(e, hi)).abs()).min())


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_directional_derivatives_match_central_differences_in_every_layout(B, model, integ, cur):
    e = _engine(B, model, cur)
    n, T, stride = 3, 14, 7
    h = 1e-5
    for lay in LAYOUTS:
        for seed in range(40, 60):
            z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, seed)
            z0, K, zr, ur = _t(e, z0), _t(e, _layout(K, lay, T, n)), _t(e, _layout(zr, lay, T, n)), _t(e, _layout(ur, lay, T, n))
            if _margin(e, z0, K, zr, ur, lo, hi, integ, lay, lay, T, n) > 50 * h:
                break
        else:
            pytest.fail("no seed keeps every v_k away from the clamp bounds")
        gt, gT, gc = _cotangents(e, n, T, stride, seed)
        res = _call(e, z0, K, zr, ur, lo, hi, q, r, integ, lay, lay, gtraj=gt, gzT=gT, gcost=gc, stride=stride, steps=T)
        rng = np.random.default_rng(seed + 100)
        ops = {"z0": (z0, _gz0(e, res)), "K": (K, res.gK), "z_ref": (zr, res.gz_ref), "u_ref": (ur, res.gu_ref)}
        for name, (base, grad) in ops.items():
            dirn = _t(e, rng.normal(size=tuple(base.shape)))
            if name == "z0" and e.nx == 13:
                dirn[:, 3:7] = 0.0      # leave the unit quaternion on its sphere

            def f(s):
                args = dict(z0=z0, K=K, zr=zr, ur=ur)
                args[{"z0": "z0", "K": "K", "z_ref": "zr", "u_ref": "ur"}[name]] = base + s * dirn
                return _loss(e, args["z0"], args["K"], args["zr"], args["ur"], lo, hi, q, r, integ, lay, lay, gt, gT,
                             gc, stride, T)

            d1 = (f(h) - f(-h)) / (2 * h)
            d2 = (f(h / 2) - f(-h / 2)) / h
            fd = (4 * d2 - d1) / 3
            an = float((grad * dirn).sum())
            assert abs(an - fd) <= 1e-6 * max(abs(fd), 1.0), (lay, name, an, fd)


def _saturated(e, n, T, seed):
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, seed)
    ur = np.where(np.arange(e.nu) % 2 == 0, 50.0, -50.0) * np.abs(hi) * np.ones_like(ur)
    return z0, K * 1e-3, zr, ur, lo, hi, q, r


@pytest.mark.parametrize("model", MODELS)
def test_clamp_saturated_everywhere(B, model):
    e = _engine(B, model)
    n, T = 4, 12
    z0, K, zr, ur, lo, hi, q, r = _saturated(e, n, T, 5)
    z0, K, zr, ur = _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur)
    gt, gT, gc = _cotangents(e, n, T, 1, 6)
    res = _call(e, z0, K, zr, ur, lo, hi, q, r, gtraj=gt, gzT=gT, gcost=gc, stride=1)
    assert (res.gK == 0).all()
    u = torch.where(ur > 0, _t(e, hi), _t(e, lo))
    expect = -2.0 * gc[None, :, None] * _t(e, r) * (u - ur)
    assert _normwise(res.gu_ref.cpu(), expect.cpu()) < 1e-14
    res0 = _call(e, z0, K, zr, ur, lo, hi, q, r, gtraj=gt, gzT=gT, stride=1)
    assert (res0.gK == 0).all() and (res0.gu_ref == 0).all()


@pytest.mark.parametrize("model", ("thruster8", "wrench12"))
def test_yaw_reference_offset_by_a_turn_gives_the_same_gradients(B, model):
    e = _engine(B, model)
    n, T = 4, 15
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 8)
    zr2 = zr.copy()
    zr2[..., 5] += TWO_PI
    zr2[..., 3] -= TWO_PI
    gt, gT, gc = _cotangents(e, n, T, 5, 9)
    a = _call(e, _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur), lo, hi, q, r, gtraj=gt, gzT=gT, gcost=gc, stride=5)
    b = _call(e, _t(e, z0), _t(e, K), _t(e, zr2), _t(e, ur), lo, hi, q, r, gtraj=gt, gzT=gT, gcost=gc, stride=5)
    for x, y in ((_gz0(e, a), _gz0(e, b)), (a.gK, b.gK), (a.gz_ref, b.gz_ref), (a.gu_ref, b.gu_ref)):
        assert _normwise(y.cpu(), x.cpu()) < 1e-12


@pytest.mark.parametrize("model", MODELS)
def test_layouts_repeats_permutation_and_chaining(B, model):
    e = _engine(B, model)
    n, T, stride = 37, 14, 7
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 21)
    z0 = _t(e, z0)
    gt, gT, gc = _cotangents(e, n, T, stride, 22)
    kw = dict(gtraj=gt, gzT=gT, gcost=gc, stride=stride)
    # equal values in every layout: bit-identical gz0; shared gradients = sums of the tnc gradient
    Kb, zrb, urb = K[:1, :1].repeat(T, 0).repeat(n, 1), zr[:1, :1].repeat(T, 0).repeat(n, 1), ur[:1, :1].repeat(T, 0).repeat(n, 1)
    full = _call(e, z0, _t(e, Kb), _t(e, zrb), _t(e, urb), lo, hi, q, r, **kw)
    dims = {"const_shared": (0, 1), "shared": (1,), "const": (0,), "tnc": ()}
    for lay in LAYOUTS:
        res = _call(e, z0, _t(e, _layout(Kb, lay, T, n)), _t(e, _layout(zrb, lay, T, n)), _t(e, _layout(urb, lay, T, n)),
                    lo, hi, q, r, kl=lay, rl=lay, steps=T, **kw)
        assert torch.equal(_gz0(e, res), _gz0(e, full)), lay
        for g, gf in ((res.gK, full.gK), (res.gz_ref, full.gz_ref), (res.gu_ref, full.gu_ref)):
            want = gf.sum(dim=dims[lay]) if dims[lay] else gf
            assert _normwise(g.cpu(), want.cpu()) < 1e-13, lay
    # repeats
    K, zr, ur = _t(e, K), _t(e, zr), _t(e, ur)
    a = _call(e, z0, K, zr, ur, lo, hi, q, r, **kw)
    b = _call(e, z0, K, zr, ur, lo, hi, q, r, **kw)
    for x, y in ((_gz0(e, a), _gz0(e, b)), (a.gK, b.gK), (a.gz_ref, b.gz_ref), (a.gu_ref, b.gu_ref), (a.z, b.z)):
        assert torch.equal(x, y)
    # permutation of the vehicles permutes gz0 and the per-vehicle gradients bit for bit
    p = torch.as_tensor(np.random.default_rng(3).permutation(n), device=e.device)
    c = _call(e, z0[p], K[:, p], zr[:, p], ur[:, p], lo, hi, q, r, gtraj=gt[:, p], gzT=gT[p], gcost=gc[p], stride=stride)
    assert torch.equal(_gz0(e, c), _gz0(e, a)[p])
    for x, y in ((c.gK, a.gK[:, p]), (c.gz_ref, a.gz_ref[:, p]), (c.gu_ref, a.gu_ref[:, p])):
        assert torch.equal(x, y)
    # chaining at t1 = 7: gz0 and the time-sliced gradients bit for bit, constant sums to rounding
    t1 = 7
    s1 = t1 // stride
    late = _call(e, _first_z(e, z0, K, zr, ur, lo, hi, q, r, t1), K[t1:], zr[t1:], ur[t1:], lo, hi, q, r,
                 gtraj=gt[s1:], gzT=gT, gcost=gc, stride=stride)
    early = _call(e, z0, K[:t1], zr[:t1], ur[:t1], lo, hi, q, r, gtraj=gt[:s1], gzT=_gz0(e, late).contiguous(), gcost=gc,
                  stride=stride)
    assert torch.equal(_gz0(e, early), _gz0(e, a))
    for x, y in ((torch.cat([early.gK, late.gK]), a.gK), (torch.cat([early.gz_ref, late.gz_ref]), a.gz_ref),
                 (torch.cat([early.gu_ref, late.gu_ref]), a.gu_ref)):
        assert torch.equal(x, y)
    const = dict(kl="const", rl="const")
    one = _call(e, z0, K[0], zr[0], ur[0], lo, hi, q, r, steps=T, **const, **kw)
    c2 = _call(e, _first_z(e, z0, K[0], zr[0], ur[0], lo, hi, q, r, t1, "const"), K[0], zr[0], ur[0], lo, hi, q, r,
               steps=T - t1, gtraj=gt[s1:], gzT=gT, gcost=gc, stride=stride, **const)
    c1 = _call(e, z0, K[0], zr[0], ur[0], lo, hi, q, r, steps=t1, gtraj=gt[:s1], gzT=_gz0(e, c2).contiguous(), gcost=gc,
               stride=stride, **const)
    assert torch.equal(_gz0(e, c1), _gz0(e, one))
    for x, y in ((c1.gK + c2.gK, one.gK), (c1.gz_ref + c2.gz_ref, one.gz_ref), (c1.gu_ref + c2.gu_ref, one.gu_ref)):
        assert _normwise(x.cpu(), y.cpu()) < 1e-13


def _first_z(e, z0, K, zr, ur, lo, hi, q, r, t1, lay="tnc"):
    """z_{t1}: the z_out of a vjp call over the first t1 steps (the primal the adjoint differentiates)"""
    if lay == "tnc":
        return _call(e, z0, K[:t1], zr[:t1], ur[:t1], lo, hi, q, r, want=()).z
    return _call(e, z0, K, zr, ur, lo, hi, q, r, kl=lay, rl=lay, steps=t1, want=()).z


@pytest.mark.parametrize("model", MODELS)
def test_per_vehicle_table_matches_single_vehicle_calls(B, L, model):
    e = _engine(B, model)
    n, T = 6, 12
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 31)
    rng = np.random.default_rng(4)
    ph = np.tile(e.phys, (n, 1))
    for s in (L.PH_ADDED, L.PH_LIN, L.PH_QUAD):
        ph[:, s:s + 6] *= rng.uniform(0.7, 1.3, (n, 6))
    gt, gT, gc = _cotangents(e, n, T, 4, 5)
    e.set_vehicle_physical(ph)
    try:
        res = _call(e, _t(e, z0), _t(e, K[0]), _t(e, zr[0]), _t(e, ur[0]), lo, hi, q, r, kl="const", rl="const", steps=T,
                    gtraj=gt, gzT=gT, gcost=gc, stride=4)
    finally:
        e.set_vehicle_physical(None)
    base = e.phys.copy()
    try:
        for i in range(n):
            e.set_physical(ph[i])
            one = _call(e, _t(e, z0[i:i + 1]), _t(e, K[0, i:i + 1]), _t(e, zr[0, i:i + 1]), _t(e, ur[0, i:i + 1]), lo, hi,
                        q, r, kl="const", rl="const", steps=T, gtraj=gt[:, i:i + 1].contiguous(), gzT=gT[i:i + 1],
                        gcost=gc[i:i + 1], stride=4)
            for x, y in ((_gz0(e, one)[0], _gz0(e, res)[i]), (one.gK[0], res.gK[i]), (one.gz_ref[0], res.gz_ref[i]),
                         (one.gu_ref[0], res.gu_ref[i])):
                assert _normwise(y.cpu(), x.cpu()) < 1e-14
    finally:
        e.set_physical(base)


@pytest.mark.parametrize("lay", LAYOUTS)
@pytest.mark.parametrize("model", MODELS)
def test_closed_loop_diff_passes_gradcheck(B, model, lay):
    e = _engine(B, model)
    n, T = 2, 4
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 61)
    lo, hi = 100 * lo, 100 * hi              # no clamp within gradcheck's steps
    x0 = _t(e, z0[:, :e.nx]).requires_grad_()
    lag = _t(e, z0[:, e.nx:]).requires_grad_() if model == "thruster8" else None
    Kt = _t(e, _layout(K, lay, T, n)).requires_grad_()
    zrt = _t(e, _layout(zr, lay, T, n)).requires_grad_()
    urt = _t(e, _layout(ur, lay, T, n)).requires_grad_()
    steps = T if lay in ("const_shared", "const") else None

    def f(x0, Kt, zrt, urt, *lag_):
        zt, z, cost = e.closed_loop_diff(x0, Kt, zrt, urt, lag0=lag_[0] if lag_ else None, steps=steps, dt=DT, stride=2,
                                         k_layout=lay, ref_layout=lay, u_min=lo, u_max=hi, cost_q=q, cost_r=r)
        return zt, z, cost

    inputs = (x0, Kt, zrt, urt) + ((lag,) if lag is not None else ())
    assert torch.autograd.gradcheck(f, inputs, eps=1e-6, atol=1e-6, rtol=1e-5, fast_mode=True)


@pytest.mark.parametrize("model", MODELS)
def test_edge_sizes(B, model):
    e = _engine(B, model)
    T = 9
    nmax = 130
    z0, K, zr, ur, lo, hi, q, r = _problem(e, nmax, T, 71)
    gt, gT, gc = _cotangents(e, nmax, T, 3, 72)
    z0, K, zr, ur = _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur)
    big = _call(e, z0, K, zr, ur, lo, hi, q, r, gtraj=gt, gzT=gT, gcost=gc, stride=3)
    for n in (1, 127, 129):
        res = _call(e, z0[:n], K[:, :n].contiguous(), zr[:, :n].contiguous(), ur[:, :n].contiguous(), lo, hi, q, r,
                    gtraj=gt[:, :n].contiguous(), gzT=gT[:n], gcost=gc[:n], stride=3)
        assert torch.equal(_gz0(e, res), _gz0(e, big)[:n])
        assert torch.equal(res.gK, big.gK[:, :n])
        assert torch.equal(res.gz_ref, big.gz_ref[:, :n])
        assert torch.equal(res.gu_ref, big.gu_ref[:, :n])
    empty = e.closed_loop_vjp(z0[:0, :e.nx], K[0, 0], zr[0, 0], ur[0, 0], steps=T, lag0=z0[:0, e.nx:] if model == "thruster8"
                              else None, lag_repr="projected")
    assert empty.gx0.shape == (0, e.nx)


@pytest.mark.parametrize("model", ("thruster8", "wrench12"))
def test_health_counts_non_finite_and_singular_vehicles(B, model):
    e = _engine(B, model)
    n, T = 8, 10
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 81)
    z0[2, 0] = np.nan
    z0[5, 4] = np.pi / 2 - 1e-5
    res = _call(e, _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur), lo, hi, q, r, gzT=_t(e, np.ones((n, e.nz))), health=True)
    h = res.health.tolist()
    assert h[0] >= 1 and h[1] >= 1
    assert not torch.isfinite(_gz0(e, res)[2]).all()
    assert torch.isfinite(_gz0(e, res)[0]).all()


def _desc(L, e, n, T, bufs):
    d = L.ClosedLoopVjpDesc()
    d.struct_size = C.sizeof(L.ClosedLoopVjpDesc)
    d.integrator = L.RK4
    d.n, d.steps, d.dt = n, T, DT
    d.z0_dev = bufs["z0"].data_ptr()
    d.K_dev = bufs["K"].data_ptr()
    d.z_ref_dev = bufs["zr"].data_ptr()
    d.u_ref_dev = bufs["ur"].data_ptr()
    for j in range(8):
        d.u_min[j], d.u_max[j] = -1.0, 1.0
    d.gz0_dev = bufs["gz0"].data_ptr()
    d.gK_dev = bufs["gK"].data_ptr()
    d.workspace_dev = bufs["ws"].data_ptr()
    d.workspace_bytes = bufs["ws"].numel() * 8
    return d


def test_refusals(B, L):
    e = B.Engine("thruster8", "f64")
    n, T = 4, 5
    wsb = L.lib.brov_closed_loop_vjp_workspace_bytes(L.THRUSTER8_LAG3, n, T)
    bufs = dict(z0=torch.zeros((n, 30), dtype=torch.float64, device="cuda"),
                K=torch.zeros((8, 30), dtype=torch.float64, device="cuda"),
                zr=torch.zeros(30, dtype=torch.float64, device="cuda"), ur=torch.zeros(8, dtype=torch.float64, device="cuda"),
                gz0=torch.zeros((n, 30), dtype=torch.float64, device="cuda"),
                gK=torch.zeros((8, 30), dtype=torch.float64, device="cuda"),
                ws=torch.zeros(wsb // 8, dtype=torch.float64, device="cuda"))

    def rc(eng, **over):
        d = _desc(L, eng, n, T, bufs)
        for k, v in over.items():
            if k in ("u_min", "u_max"):
                getattr(d, k)[0] = v
            else:
                setattr(d, k, v)
        return L.lib.brov_closed_loop_vjp(eng._h, C.byref(d), None)

    assert rc(e) == 0
    torch.cuda.synchronize()
    EINVAL, EUNSUP = -1, -4
    assert rc(e, struct_size=8) == EINVAL
    assert rc(e, steps=0) == EINVAL
    assert rc(e, n=-1) == EINVAL
    assert rc(e, dt=0.0) == EINVAL
    assert rc(e, integrator=7) == EINVAL
    assert rc(e, K_stride_t=-1) == EINVAL
    assert rc(e, u_min=2.0) == EINVAL
    assert rc(e, u_max=float("nan")) == EINVAL
    assert rc(e, gtraj_dev=bufs["gz0"].data_ptr(), stride=0) == EINVAL
    assert rc(e, workspace_bytes=wsb // 4) == EINVAL
    assert rc(e, workspace_dev=None) == EINVAL
    assert rc(e, gz0_dev=None) == EINVAL
    assert rc(e, K_dev=None) == EINVAL
    assert rc(e, K_stride_n=8) == EINVAL                         # rows of distinct vehicles would overlap in gK
    assert rc(e, n=0, z0_dev=None, gz0_dev=None) == 0
    # a workspace size that wraps modulo 2^64 in unchecked arithmetic (n * steps * 38 doubles) is still refused
    assert rc(e, n=452_144_348, steps=1_073_640_831) == EINVAL
    e.set_vehicle_physical(np.tile(e.phys, (n + 1, 1)))
    try:
        assert rc(e) == EINVAL
    finally:
        e.set_vehicle_physical(None)
    e32 = B.Engine("thruster8", "f32")
    assert rc(e32) == EUNSUP
    edi = B.Engine("di12_u6", "f64")
    assert rc(edi) == EUNSUP
    ew = B.Engine("wrench12", "f64")
    ew.set_wrench_lag1(True, 0.1)
    assert rc(ew) == EUNSUP


def test_gain_gradient_above_2_31_elements(B):
    e = _engine(B, "thruster8")
    n, T = 8192, 1093                                           # T * n * 240 > 2^31
    assert T * n * 240 > 2 ** 31
    z0, K1, zr, ur, lo, hi, q, r = _problem(e, 2, 2, 91)
    rng = np.random.default_rng(92)
    z0 = _t(e, np.tile(z0[:1], (n, 1)) + rng.normal(0, 0.05, (n, e.nz)))
    Kb = _t(e, K1[0, 0])
    K = Kb.expand(T, n, 8, 30).contiguous()
    zr_, ur_ = _t(e, zr[0, 0]), _t(e, ur[0, 0])
    gT = _t(e, rng.normal(size=(n, e.nz)))
    res = _call(e, z0, K, zr_, ur_, lo, hi, q, r, kl="tnc", rl="const_shared", gzT=gT, want=("K",))
    del K
    for i in (0, n - 1):
        one = _call(e, z0[i:i + 1], Kb.expand(T, 1, 8, 30).contiguous(), zr_, ur_, lo, hi, q, r, kl="tnc",
                    rl="const_shared", gzT=gT[i:i + 1], want=("K",))
        assert torch.equal(res.gK[:, i:i + 1], one.gK)
        assert torch.equal(_gz0(e, res)[i], _gz0(e, one)[0])


def test_health_counts_a_non_finite_gain_gradient_entry(B):
    """|dz_j| ~ 1e300 in a state column the gain does not read, and a large cotangent: z, gz0, the dz cotangent and
    dL/du_ref stay finite, only -gv dz_j overflows, and the vehicle is counted"""
    e = _engine(B, "wrench12")
    n, T = 2, 3
    z0, K, zr, ur, lo, hi, q, r = _problem(e, n, T, 95)
    K[..., 0] = 0.0
    zr[:, 0, 0] = 1e300
    gT = np.full((n, e.nz), 1e12)
    res = _call(e, _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur), 1e3 * lo, 1e3 * hi, q, r, gzT=_t(e, gT), health=True,
                want=("K", "u_ref"))
    assert torch.isfinite(res.z).all() and torch.isfinite(_gz0(e, res)).all() and torch.isfinite(res.gu_ref).all()
    assert not torch.isfinite(res.gK[:, 0]).all() and torch.isfinite(res.gK[:, 1]).all()
    assert res.health.tolist()[0] == 1
    # without the gain gradient there is no such entry
    res = _call(e, _t(e, z0), _t(e, K), _t(e, zr), _t(e, ur), 1e3 * lo, 1e3 * hi, q, r, gzT=_t(e, gT), health=True,
                want=("u_ref",))
    assert res.health.tolist()[0] == 0
