"""GPU tests of the coefficient gradient (brov_multistep_se_grad through Engine.multistep_se_grad) and the
Levenberg-Marquardt calibration built on it: the primal sums equal the evaluator's, the gradient agrees with
differences of the sweep, of per-window rollouts and of the numpy oracle, the Gauss-Newton matrix is symmetric and
positive semidefinite, the outputs are reproducible, linear in the directions and additive over window shards, and a
calibration recovers the vehicle that generated a series."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import fossen_np as O

pytestmark = pytest.mark.gpu

DT = 0.02
HS = [1, 10, 100]
P18 = ["added", "lin", "quad"]


@pytest.fixture(scope="module")
def B():
    import bluerov2_dynamics_b200 as b
    return b


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200 import _lib
    return _lib


def _series(B, model, rows, seed, integ="rk4", phys=None, noise=1e-3):
    """A recorded series: a rollout of the default (or given) vehicle under smooth random inputs, plus noise."""
    rng = np.random.default_rng(seed)
    e = B.Engine(model, "f64")
    if phys is not None:
        e.set_physical(phys)
    U = O.smooth_inputs(rng, rows, e.nu, scale=0.5) if model == "thruster8" else O.smooth_inputs(rng, rows, 6, scale=3.0)
    x0 = np.zeros((1, e.nx))
    if e.nx == 13:
        x0[0, 3] = 1.0
    x0[0, :3] = rng.uniform(-1, 1, 3)
    r = e.rollout(x0, U[:rows - 1], dt=DT, integrator=integ, stride=1, u_layout="shared")
    X = np.concatenate([x0, r.traj[:, 0, :].cpu().numpy()])
    return X + noise * rng.standard_normal(X.shape), U


def _perturbed(B, L, seed, spread=0.3, current=False):
    """The defaults with the 18 hydrodynamic coefficients (and buoyancy, optionally a current) perturbed."""
    rng = np.random.default_rng(seed)
    ph = B.default_physical()
    for col in (L.PH_ADDED, L.PH_LIN, L.PH_QUAD):
        ph[col:col + 6] *= rng.uniform(1 - spread, 1 + spread, 6)
    ph[L.PH_B] *= rng.uniform(0.98, 1.02)
    if current:
        ph[L.PH_CURRENT:L.PH_CURRENT + 3] = rng.uniform(-0.1, 0.1, 3)
    return B.with_minv(ph)


@pytest.fixture(scope="module")
def series(B):
    return {m: _series(B, m, 1501, i) for i, m in enumerate(("thruster8", "wrench12", "quat13"))}


def _params(L, ph):
    """physical vector -> parameter dict of the numpy oracle (oracle/fossen_np.py)"""
    from oracle import c_oracle as CO
    p = dict(m=ph[L.PH_M], W=ph[L.PH_W], B=ph[L.PH_B], xb=ph[L.PH_XB], yb=ph[L.PH_XB + 1], zb=ph[L.PH_XB + 2],
             Ix=ph[L.PH_I], Iy=ph[L.PH_I + 1], Iz=ph[L.PH_I + 2], Minv=ph[L.PH_MINV:L.PH_MINV + 6].copy(),
             current=ph[L.PH_CURRENT:L.PH_CURRENT + 3].copy())
    for names, col in ((CO._PH_NAMES_ADDED, L.PH_ADDED), (CO._PH_NAMES_LIN, L.PH_LIN), (CO._PH_NAMES_QUAD, L.PH_QUAD)):
        for j, k in enumerate(names):
            p[k] = ph[col + j]
    return p


def _normwise(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _sweep_fd(B, e, X, U, hs, ph, idx, integ, lag_mode, rel=1e-4):
    """Central differences of the sweep's sums in the physical entries idx, Richardson-extrapolated (h and 2h)."""
    scale = np.where(ph[idx] != 0.0, np.abs(ph[idx]), 1.0)
    table = []
    for j, i in enumerate(idx):
        h = rel * scale[j]
        for s in (h, -h, 2 * h, -2 * h):
            q = ph.copy()
            q[i] += s
            table.append(B.with_minv(q))
    out = []
    for part in ([[h] for h in hs] if lag_mode == "carry" else [hs]):
        se, _ = e.multistep_se_sweep(X, U, part, np.array(table), dt=DT, integrator=integ, lag_mode=lag_mode)
        out.append(se.cpu().numpy()[:, :len(part)])
    s = np.concatenate(out, axis=1).reshape(len(idx), 4, len(hs))
    h = (rel * scale)[:, None]
    d1 = (s[:, 0] - s[:, 1]) / (2 * h)
    d2 = (s[:, 2] - s[:, 3]) / (4 * h)
    return ((4 * d1 - d2) / 3).T                      # [nH, p]


def _raw(B, L, e, X, U, hs, kp, dirs, carry=0, window0=0, row0=0, n_windows=None, any_current=0, health=None):
    """Direct C-ABI call with arbitrary directions: (se [4], grad [4, p], gn [4, p, p], counts, rc)."""
    X, U = e.tensor(X), e.tensor(U)
    rows = X.shape[0]
    nwin = rows - (window0 - row0) - hs[0] if n_windows is None else n_windows
    p = dirs.shape[0]
    kp_t = torch.as_tensor(kp, dtype=torch.float64, device="cuda")
    d_t = torch.as_tensor(np.ascontiguousarray(dirs), dtype=torch.float64, device="cuda")
    se = torch.zeros(4, dtype=torch.float64, device="cuda")
    gr = torch.zeros((4, max(p, 1)), dtype=torch.float64, device="cuda")
    gn = torch.zeros((4, max(p, 1), max(p, 1)), dtype=torch.float64, device="cuda")
    ws = torch.empty(max(L.lib.brov_se_grad_workspace_bytes(max(nwin, 0), max(min(p, 36), 1), carry), 1),
                     dtype=torch.uint8, device="cuda")
    cnt = (C.c_longlong * 4)()
    d = L.SeGradDesc()
    d.struct_size = C.sizeof(L.SeGradDesc)
    d.integrator, d.rows, d.n_windows, d.dt = L.RK4, rows, nwin, DT
    d.X_dev, d.U_dev = X.data_ptr(), U.data_ptr()
    d.n_horizons = len(hs)
    for i, h in enumerate(hs):
        d.horizons[i] = h
    d.lag_carry, d.window0, d.row0 = carry, window0, row0
    d.kp_dev, d.any_current, d.n_dirs, d.dirs_dev = kp_t.data_ptr(), any_current, p, d_t.data_ptr()
    d.se_out_dev, d.grad_out_dev, d.gn_out_dev = se.data_ptr(), gr.data_ptr(), gn.data_ptr()
    d.count_out = cnt
    d.health_dev = health.data_ptr() if health is not None else None
    d.workspace_dev, d.workspace_bytes = ws.data_ptr(), ws.numel()
    rc = L.lib.brov_multistep_se_grad(e._h, C.byref(d), None)
    torch.cuda.synchronize()
    return se.cpu().numpy(), gr.cpu().numpy(), gn.cpu().numpy(), list(cnt), rc


# ------------------------------------------------------------------------------------------------ 1. primal
@pytest.mark.parametrize("integ", ["rk4", "euler"])
@pytest.mark.parametrize("model,lag_mode", [("thruster8", "reset"), ("thruster8", "carry"), ("wrench12", "reset"),
                                            ("quat13", "reset")])
def test_primal_equals_the_evaluator(B, L, series, model, lag_mode, integ):
    X, U = series[model]
    ph = _perturbed(B, L, 1, current=(model == "wrench12"))
    e = B.Engine(model, "f64")
    r = e.multistep_se_grad(X, U, HS, ph, P18, dt=DT, integrator=integ, lag_mode=lag_mode)
    e.set_physical(ph)
    ref = []
    for part in ([[h] for h in HS] if lag_mode == "carry" else [HS]):
        se, cnt = e.multistep_se(X, U, part, dt=DT, integrator=integ, lag_mode=lag_mode, time_slices=1)
        ref += list(se.cpu().numpy()[:len(part)])
    assert r.counts == [1500, 1491, 1401] and r.names[:2] == ["Xu_dot", "Yv_dot"]
    assert _normwise(r.se.cpu().numpy(), ref) <= 1e-12
    assert r.grad.shape == (3, 18) and r.gn.shape == (3, 18, 18)


# ------------------------------------------------------------------------------------------------ 2. vs differences
@pytest.mark.parametrize("integ", ["rk4", "euler"])
@pytest.mark.parametrize("model,lag_mode", [("thruster8", "reset"), ("thruster8", "carry"), ("wrench12", "reset"),
                                            ("quat13", "reset")])
def test_gradient_matches_sweep_differences(B, L, series, model, lag_mode, integ):
    X, U = series[model]
    X, U = X[:601], U[:601]
    cur = model == "wrench12"
    ph = _perturbed(B, L, 2, current=cur)
    e = B.Engine(model, "f64")
    params = P18[:2] + (["B", "quad", "current_n", "current_e"] if cur else ["B", "quad"])
    r = e.multistep_se_grad(X, U, HS, ph, params, dt=DT, integrator=integ, lag_mode=lag_mode)
    fd = _sweep_fd(B, e, X, U, HS, ph, r.index, integ, lag_mode)
    g = r.grad.cpu().numpy()
    for h in range(3):
        assert _normwise(g[h], fd[h]) <= 1e-6, (HS[h], _normwise(g[h], fd[h]))


# ------------------------------------------------------------------------------------------------ 3. per window
@pytest.mark.parametrize("model", ["thruster8", "quat13"])
def test_gradient_and_gn_match_per_window_rollout_differences(B, L, series, model):
    """64 windows in reset mode: J_w by central differences of Engine.rollout with the windows as vehicles; the
    host-assembled sum_w 2 r_w J_w and sum_w J_w^T J_w agree with the kernel's."""
    X, U = series[model]
    H, nw = 10, 64
    X, U = X[:nw + H], U[:nw + H]
    ph = _perturbed(B, L, 3)
    e = B.Engine(model, "f64")
    r = e.multistep_se_grad(X, U, [H], ph, P18, dt=DT)
    assert r.counts == [nw]
    Useq = np.stack([U[k:k + H] for k in range(nw)], axis=1)          # [H, nw, NU] time-major
    idx = r.index

    def ends(q):
        e.set_physical(B.with_minv(q))
        return e.rollout(X[:nw], Useq, dt=DT, integrator="rk4", want_lag=False).xT.cpu().numpy()

    res = ends(ph) - X[H:H + nw]
    J = np.zeros((nw, e.nx, len(idx)))
    for j, i in enumerate(idx):
        hh = 1e-5 * max(abs(ph[i]), 1.0)
        d = []
        for s in (hh, -hh, 2 * hh, -2 * hh):
            q = ph.copy()
            q[i] += s
            d.append(ends(q))
        J[:, :, j] = (8 * (d[0] - d[1]) - (d[2] - d[3])) / (12 * hh)
    g = 2 * np.einsum("wx,wxj->j", res, J)
    G = np.einsum("wxi,wxj->ij", J, J)
    assert _normwise(r.grad.cpu().numpy()[0], g) <= 1e-6
    assert _normwise(r.gn.cpu().numpy()[0], G) <= 1e-6


# ------------------------------------------------------------------------------------------------ 4. numpy oracle
@pytest.mark.parametrize("lag_mode", ["reset", "carry"])
def test_gradient_matches_oracle_differences(B, L, series, lag_mode):
    X, U = series["thruster8"]
    X, U = X[:300], U[:300]
    ph = _perturbed(B, L, 4)
    e = B.Engine("thruster8", "f64")
    params = ["Xu_dot", "Zw_dot", "Xu", "Zw", "Xu_abs", "Nr_abs", "B"]
    hs = [1, 10]
    r = e.multistep_se_grad(X, U, hs, ph, params, dt=DT, lag_mode=lag_mode)
    g = r.grad.cpu().numpy()
    for j, i in enumerate(r.index):
        hh = 1e-4 * max(abs(ph[i]), 1.0)
        vals = []
        for s in (hh, -hh, 2 * hh, -2 * hh):
            q = ph.copy()
            q[i] += s
            res = O.multistep_se(O.Model("thruster8", DT, _params(L, B.with_minv(q))), "rk4", X, U, hs, lag_mode=lag_mode)
            vals.append(np.array([res[h][0] for h in hs]))
        fd = (8 * (vals[0] - vals[1]) - (vals[2] - vals[3])) / (12 * hh)
        for k in range(len(hs)):
            assert abs(g[k, j] - fd[k]) <= 1e-5 * np.max(np.abs(g[k])) + 1e-12, (r.names[j], hs[k], g[k, j], fd[k])


# ------------------------------------------------------------------------------------------------ 5-6. structure
def test_gn_structure_reproducibility_independence_permutation(B, L, series):
    X, U = series["wrench12"]
    ph = _perturbed(B, L, 5, current=True)
    params = P18 + ["B", "current_n", "current_e", "current_d"]
    e = B.Engine("wrench12", "f64")
    r1 = e.multistep_se_grad(X, U, HS, ph, params, dt=DT)
    G = r1.gn.cpu().numpy()
    for h in range(3):
        assert np.array_equal(G[h], G[h].T)
        ev = np.linalg.eigvalsh(G[h])
        assert ev[0] >= -1e-12 * ev[-1], (ev[0], ev[-1])
    r2 = e.multistep_se_grad(X, U, HS, ph, params, dt=DT)
    assert torch.equal(r1.se, r2.se) and torch.equal(r1.grad, r2.grad) and torch.equal(r1.gn, r2.gn)
    other = B.default_physical()
    other[L.PH_QUAD:L.PH_QUAD + 6] *= 3.0
    e.set_physical(B.with_minv(other))
    r3 = e.multistep_se_grad(X, U, HS, ph, params, dt=DT)
    assert torch.equal(r1.grad, r3.grad) and torch.equal(r1.gn, r3.gn)
    perm = list(np.random.default_rng(0).permutation(len(r1.index)))
    rp = e.multistep_se_grad(X, U, HS, ph, [r1.index[i] for i in perm], dt=DT)
    pt = torch.as_tensor(perm, device=r1.grad.device)
    assert torch.equal(rp.grad, r1.grad[:, pt]) and torch.equal(rp.gn, r1.gn[:, pt][:, :, pt])


def test_outputs_are_linear_in_the_directions(B, L, series):
    X, U = series["thruster8"]
    e = B.Engine("thruster8", "f64")
    ph = _perturbed(B, L, 6)
    kp = B.derive_params(ph)
    D = B.coefficient_directions(ph, ["Xu_abs", "Zw_dot"])
    a, b = 0.7, -1.9
    dirs = np.stack([D[0], D[1], a * D[0] + b * D[1]])
    se, g, G, cnt, rc = _raw(B, L, e, X, U, HS, kp, dirs)
    assert rc == 0
    for h in range(3):
        assert abs(g[h, 2] - (a * g[h, 0] + b * g[h, 1])) <= 1e-12 * np.max(np.abs(g[h]))
        ref = a * a * G[h, 0, 0] + 2 * a * b * G[h, 0, 1] + b * b * G[h, 1, 1]
        assert abs(G[h, 2, 2] - ref) <= 1e-12 * np.max(np.abs(G[h]))
        assert abs(G[h, 0, 2] - (a * G[h, 0, 0] + b * G[h, 0, 1])) <= 1e-12 * np.max(np.abs(G[h]))


@pytest.mark.parametrize("carry", [0, 1])
def test_window_shards_add_up_to_the_whole(B, L, series, carry):
    X, U = series["thruster8"]
    e = B.Engine("thruster8", "f64")
    ph = _perturbed(B, L, 7)
    kp, D = B.derive_params(ph), B.coefficient_directions(ph, P18)
    hs = [10] if carry else HS
    whole = _raw(B, L, e, X, U, hs, kp, D, carry=carry)
    assert whole[4] == 0
    n = whole[3][0]
    cut = 700
    if carry:
        row0 = (cut * hs[0] - e.carry_steps(DT, "rk4")) // hs[0]
        a = _raw(B, L, e, X[:cut + hs[0]], U[:cut + hs[0]], hs, kp, D, carry=1, n_windows=cut)
        b = _raw(B, L, e, X[row0:], U[row0:], hs, kp, D, carry=1, window0=cut, row0=row0, n_windows=n - cut)
    else:
        a = _raw(B, L, e, X[:cut + hs[-1]], U[:cut + hs[-1]], hs, kp, D, n_windows=cut)
        b = _raw(B, L, e, X[cut:], U[cut:], hs, kp, D)
    assert a[4] == 0 and b[4] == 0
    for k in range(3):
        assert _normwise(a[k] + b[k], whole[k]) <= 1e-12, k


# ------------------------------------------------------------------------------------------------ 7. edges, errors
def test_edge_cases_and_errors(B, L, series):
    X, U = series["thruster8"]
    e = B.Engine("thruster8", "f64")
    ph = B.default_physical()
    kp, D = B.derive_params(ph), B.coefficient_directions(ph, P18)
    assert _raw(B, L, e, X, U, HS, kp, np.zeros((0, 36)))[4] == -1
    assert _raw(B, L, e, X, U, HS, kp, np.zeros((37, 36)))[4] == -1
    assert _raw(B, L, e, X, U, [10, 5], kp, D)[4] == -1
    for eng in (B.Engine("thruster8", "f32"), B.Engine("di12_u8", "f64")):
        with pytest.raises(B.BrovError):
            eng.multistep_se_grad(X[:, :eng.nx], U, HS, ph, P18, dt=DT)
        assert _raw(B, L, eng, X, U, HS, kp, D)[4] == -4
    w = B.Engine("wrench12", "f64")
    w.set_wrench_lag1(True)
    Xw, Uw = series["wrench12"]
    with pytest.raises(B.BrovError, match="wrench lag"):
        w.multistep_se_grad(Xw, Uw, HS, ph, P18, dt=DT)
    r = e.multistep_se_grad(X[:50], U[:50], [50, 60], ph, P18, dt=DT)     # rows <= H: nothing to score
    assert r.counts == [0, 0] and not torch.any(r.se) and not torch.any(r.grad) and not torch.any(r.gn)
    Xb = X.copy()
    Xb[400, 7] = np.nan
    hc = torch.zeros(2, dtype=torch.int64, device=e.device)
    rb = e.multistep_se_grad(Xb, U, HS, ph, P18, dt=DT, health_out=hc)
    assert hc[0].item() > 0 and not np.isfinite(rb.se[0].item())
    with pytest.raises(ValueError):
        e.multistep_se_grad(X, U, HS, ph, ["T_lag1"], dt=DT)


# ------------------------------------------------------------------------------------------------ 8-9. calibration
@pytest.mark.parametrize("model,integ,hs,lag_mode", [("thruster8", "rk4", (1,), "carry"),
                                                     ("quat13", "euler", (1, 10, 100), "reset")])
def test_calibration_recovers_the_generating_vehicle(B, L, model, integ, hs, lag_mode):
    """Noise-free series of a vehicle with all 18 coefficients perturbed by up to 30 %.  The thruster model is fitted
    at H = 1 with the carried lag: there the reference's shared lag state equals that of the continuous series, so the
    generating vehicle scores zero (at H = 10 / 100 the carried lag replays overlapping windows and does not)."""
    from bluerov2_dynamics_b200.evaluators import calibrate_physical
    truth = _perturbed(B, L, 8)
    truth[L.PH_B] = B.default_physical()[L.PH_B]
    X, U = _series(B, model, 3001, 9, integ=integ, phys=truth, noise=0.0)
    res = calibrate_physical(X, U, DT, B.default_physical(), P18, horizons=hs, model=model, integrator=integ,
                             lag_mode=lag_mode, max_iter=50, tol=1e-14)
    G = res.gn
    ev, vec = np.linalg.eigh(G)
    print(f"{model}: {res.iterations} iterations, cost {res.cost0:.3e} -> {res.cost:.3e}, cond(G) {ev[-1] / max(ev[0], 1e-300):.3e}")
    assert res.iterations <= 50
    assert res.cost <= 1e-10 * res.cost0
    idx = B.parameter_indices(P18)
    scale = np.where(truth[idx] != 0.0, np.abs(truth[idx]), 1.0)
    err = np.abs(res.theta - truth[idx]) / scale
    assert np.max(err) <= 1e-4, dict(zip(res.names, err))


def test_calibration_with_noise_beats_the_sweep(B, L):
    from bluerov2_dynamics_b200.evaluators import calibrate_physical
    truth = _perturbed(B, L, 10)
    truth[L.PH_B] = B.default_physical()[L.PH_B]
    X, U = _series(B, "thruster8", 6001, 11, phys=truth, noise=1e-3)
    res = calibrate_physical(X, U, DT, B.default_physical(), P18, model="thruster8", max_iter=50)
    e = B.Engine("thruster8", "f64")
    rng = np.random.default_rng(12)
    table = np.tile(B.default_physical(), (300, 1))
    for col in (L.PH_ADDED, L.PH_LIN, L.PH_QUAD):
        table[:, col:col + 6] *= rng.uniform(0.7, 1.3, (300, 6))
    table = B.with_minv(table)
    sweep = e.multistep_rmse_sweep(X, U, [10], table, dt=DT, lag_mode="carry")[:, 0]
    at_truth = e.multistep_rmse_sweep(X, U, [10], truth[None], dt=DT, lag_mode="carry")[0, 0]
    print(f"H=10 rmse: fit {res.rmse[10]:.6e}, truth {at_truth:.6e}, best of 300 {np.min(sweep):.6e}")
    assert res.rmse[10] <= np.min(sweep)
    assert res.rmse[10] <= 1.01 * at_truth


# ------------------------------------------------------------------------------------------------ 10. full size
def test_full_size_tank_series(B, L):
    X, U = _series(B, "thruster8", 45823, seed=13)
    e = B.Engine("thruster8", "f64")
    ph = _perturbed(B, L, 14)
    Xt, Ut = e.tensor(X), e.tensor(U)
    r = e.multistep_se_grad(Xt, Ut, HS, ph, P18, dt=DT)
    assert r.counts == [45822, 45813, 45723]
    pick = [0, 8, 15]
    fd = _sweep_fd(B, e, Xt, Ut, HS, ph, [r.index[i] for i in pick], "rk4", "reset")
    g = r.grad.cpu().numpy()[:, pick]
    for h in range(3):
        assert _normwise(g[h], fd[h]) <= 1e-6, (HS[h], g[h], fd[h])
        ev = np.linalg.eigvalsh(r.gn.cpu().numpy()[h])
        assert ev[0] >= -1e-12 * ev[-1]
