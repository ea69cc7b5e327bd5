"""GPU tests of the candidate sweep (brov_multistep_se_sweep through Engine.multistep_se_sweep): every candidate's
squared-error sums equal those of the single-vehicle evaluator with that candidate's coefficients, agree with the CPU
oracles, carry the lag the reference's single model object carries, single out the vehicle that generated a series,
stay independent of the other candidates and of the engine's own coefficients, and refuse what they do not support."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import fossen_np as O

pytestmark = pytest.mark.gpu

DT = 0.02
HS = [1, 10, 100]


@pytest.fixture(scope="module")
def B():
    import bluerov2_dynamics_b200 as b
    return b


@pytest.fixture(scope="module")
def L():
    from bluerov2_dynamics_b200 import _lib
    return _lib


def _candidates(B, L, P, seed, spread=0.3, current=False):
    """P physical vectors around the defaults: added masses, linear / quadratic damping, buoyancy (and an ocean
    current); diag(Minv) rebuilt from the perturbed masses."""
    rng = np.random.default_rng(seed)
    ph = np.tile(B.default_physical(), (P, 1))
    for col in (L.PH_ADDED, L.PH_LIN, L.PH_QUAD):
        ph[:, col:col + 6] *= rng.uniform(1 - spread, 1 + spread, (P, 6))
    ph[:, L.PH_B] *= rng.uniform(0.98, 1.02, P)
    if current:
        ph[:, L.PH_CURRENT:L.PH_CURRENT + 3] = rng.uniform(-0.1, 0.1, (P, 3))
    return B.with_minv(ph)


def _params(L, ph):
    """physical vector -> parameter dict of the oracles (oracle/fossen_np.py)"""
    from oracle import c_oracle as CO
    p = dict(m=ph[L.PH_M], W=ph[L.PH_W], B=ph[L.PH_B], xb=ph[L.PH_XB], yb=ph[L.PH_XB + 1], zb=ph[L.PH_XB + 2],
             Ix=ph[L.PH_I], Iy=ph[L.PH_I + 1], Iz=ph[L.PH_I + 2], Minv=ph[L.PH_MINV:L.PH_MINV + 6].copy(),
             current=ph[L.PH_CURRENT:L.PH_CURRENT + 3].copy())
    for names, col in ((CO._PH_NAMES_ADDED, L.PH_ADDED), (CO._PH_NAMES_LIN, L.PH_LIN), (CO._PH_NAMES_QUAD, L.PH_QUAD)):
        for j, k in enumerate(names):
            p[k] = ph[col + j]
    return p


def _series(B, model, rows, seed, integ="rk4", phys=None, noise=1e-3):
    """A recorded series of `model`: a rollout of the default (or given) vehicle under smooth random inputs, plus
    measurement noise.  Returns (X [rows, NX], U [rows, NU]) as float64 numpy arrays."""
    rng = np.random.default_rng(seed)
    e = B.Engine(model, "f64")
    if phys is not None:
        e.set_physical(phys)
    # gentle commands: the vehicle stays far from theta = +-pi/2, where rounding differences grow without bound
    U = O.smooth_inputs(rng, rows, e.nu, scale=0.5) if model == "thruster8" else O.smooth_inputs(rng, rows, 6, scale=3.0)
    x0 = np.zeros((1, e.nx))
    if e.nx == 13:
        x0[0, 3] = 1.0
    x0[0, :3] = rng.uniform(-1, 1, 3)
    r = e.rollout(x0, U[:rows - 1], dt=DT, integrator=integ, stride=1, u_layout="shared")
    X = np.concatenate([x0, r.traj[:, 0, :].cpu().numpy()])
    if e.nx == 12:
        assert np.max(np.abs(X[:, 4])) < 1.0
    return X + noise * rng.standard_normal(X.shape), U


@pytest.fixture(scope="module")
def series(B):
    return {m: _series(B, m, 3001, i) for i, m in enumerate(("thruster8", "wrench12", "quat13"))}


def _per_candidate(e, X, U, hs, ph, integ, lag_mode="reset"):
    out = []
    for c in range(ph.shape[0]):
        e.set_physical(ph[c])
        se, _ = e.multistep_se(X, U, hs, dt=DT, integrator=integ, lag_mode=lag_mode, time_slices=1)
        out.append(se.cpu().numpy())
    return np.array(out)


def _rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


# ------------------------------------------------------------------------------------------------ 1. equality
@pytest.mark.parametrize("dtype,tol", [("f64", 1e-12), ("f32", 1e-5)])
@pytest.mark.parametrize("integ", ["rk4", "euler"])
@pytest.mark.parametrize("model", ["thruster8", "wrench12", "quat13"])
def test_sweep_equals_the_single_vehicle_evaluator(B, L, series, model, integ, dtype, tol, record_property):
    X, U = series[model]
    ph = _candidates(B, L, 37, seed=11, current=(model == "wrench12"))
    e = B.Engine(model, dtype)
    se, cnt = e.multistep_se_sweep(X, U, HS, ph, dt=DT, integrator=integ)
    assert se.shape == (37, L.MAX_H) and cnt == [3000, 2991, 2901]
    got = se.cpu().numpy()
    ref = _per_candidate(e, X, U, HS, ph, integ)
    assert np.all(got[:, 3] == 0.0)
    assert _rel(got[:, :3], ref[:, :3]) <= tol
    record_property("bitwise", bool(np.array_equal(got, ref)))
    print(f"{model} {integ} {dtype}: bitwise equal to multistep_se(time_slices=1): {np.array_equal(got, ref)}")


# ------------------------------------------------------------------------------------------------ 2. oracle parity
def test_sweep_against_c_oracle(B, L, series):
    import subprocess
    from conftest import ROOT
    from oracle import c_oracle as CO
    if not CO.available():
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s"], check=True)
    X, U = series["thruster8"]
    X, U = X[:1201], U[:1201]
    ph = _candidates(B, L, 8, seed=12)
    se, _ = B.Engine("thruster8", "f64").multistep_se_sweep(X, U, HS, ph, dt=DT, integrator="rk4")
    got = se.cpu().numpy()
    for c in range(8):
        for j, H in enumerate(HS):
            ref, _, _ = CO.multistep_se("thruster8", "rk4", DT, X, U, H, params=_params(L, ph[c]))
            assert abs(got[c, j] - ref) <= 1e-10 * abs(ref), (c, H, got[c, j], ref)


# ------------------------------------------------------------------------------------------------ 3. carried lag
@pytest.mark.parametrize("integ", ["rk4", "euler"])
def test_sweep_carry_mode(B, L, series, integ):
    X, U = series["thruster8"]
    X, U = X[:160], U[:160]
    ph = _candidates(B, L, 4, seed=13)
    e = B.Engine("thruster8", "f64")
    for H in (1, 10):
        se, cnt = e.multistep_se_sweep(X, U, [H], ph, dt=DT, integrator=integ, lag_mode="carry")
        got = se.cpu().numpy()[:, 0]
        assert cnt == [160 - H]
        ref_engine = _per_candidate(e, X, U, [H], ph, integ, lag_mode="carry")[:, 0]
        assert _rel(got, ref_engine) <= 1e-12
        for c in range(4):
            ref = O.multistep_se(O.Model("thruster8", DT, _params(L, ph[c])), integ, X, U, [H], lag_mode="carry")[H][0]
            assert abs(got[c] - ref) <= 1e-10 * abs(ref), (H, c, got[c], ref)
        # the carried lag is not the reset lag: the modes differ
        reset, _ = e.multistep_se_sweep(X, U, [H], ph, dt=DT, integrator=integ, lag_mode="reset")
        assert not np.allclose(reset.cpu().numpy()[:, 0], got, rtol=1e-6)


# ------------------------------------------------------------------------------------------------ 4. truth recovery
def test_sweep_recovers_the_vehicle_that_generated_the_series(B, L):
    ph = _candidates(B, L, 64, seed=14)
    truth = 17
    X, U = _series(B, "wrench12", 2001, seed=5, integ="rk4", phys=ph[truth], noise=0.0)
    se, _ = B.Engine("wrench12", "f64").multistep_se_sweep(X, U, HS, ph, dt=DT, integrator="rk4")
    s = se.cpu().numpy()[:, :3]
    for j in range(3):
        assert int(np.argmin(s[:, j])) == truth
        assert s[truth, j] < 1e-20 * np.median(s[:, j]), (HS[j], s[truth, j], np.median(s[:, j]))
    # thruster model, Euler, H = 1, carried lag: window k starts from the lag of the continuous series at row k
    X, U = _series(B, "thruster8", 2001, seed=6, integ="euler", phys=ph[truth], noise=0.0)
    se, _ = B.Engine("thruster8", "f64").multistep_se_sweep(X, U, [1], ph, dt=DT, integrator="euler", lag_mode="carry")
    s = se.cpu().numpy()[:, 0]
    assert int(np.argmin(s)) == truth and s[truth] < 1e-20 * np.median(s), (s[truth], np.median(s))


# ------------------------------------------------------------------------------------------------ 5. independence
def test_sweep_is_reproducible_and_candidates_are_independent(B, L, series):
    X, U = series["thruster8"]
    ph = _candidates(B, L, 24, seed=15)
    e = B.Engine("thruster8", "f64")
    se1, _ = e.multistep_se_sweep(X, U, HS, ph, dt=DT)
    se2, _ = e.multistep_se_sweep(X, U, HS, ph, dt=DT)
    assert torch.equal(se1, se2)
    perm = np.random.default_rng(3).permutation(24)
    sep, _ = e.multistep_se_sweep(X, U, HS, ph[perm], dt=DT)
    assert torch.equal(sep, se1[torch.as_tensor(perm, device=se1.device)])
    # the engine's own coefficients play no part
    other = B.default_physical()
    other[L.PH_QUAD:L.PH_QUAD + 6] *= 3.0
    e.set_physical(B.with_minv(other))
    se3, _ = e.multistep_se_sweep(X, U, HS, ph, dt=DT)
    assert torch.equal(se3, se1)
    # one exploding candidate (anti-damping) is flagged in its own health row and changes nothing else
    bad = ph.copy()
    bad[5, L.PH_LIN:L.PH_LIN + 6] = 5000.0
    hc = torch.zeros((24, 2), dtype=torch.int64, device=e.device)
    seb, _ = e.multistep_se_sweep(X, U, HS, bad, dt=DT, health_out=hc)
    h = hc.cpu().numpy()
    assert h[5, 0] > 0 and not np.isfinite(seb[5, 2].item())
    assert np.all(np.delete(h[:, 0], 5) == 0)
    keep = torch.as_tensor(np.delete(np.arange(24), 5), device=se1.device)
    assert torch.equal(seb[keep], se1[keep])
    hc1 = torch.zeros((24, 2), dtype=torch.int64, device=e.device)
    e.multistep_se_sweep(X, U, HS, ph, dt=DT, health_out=hc1)
    assert torch.equal(hc[keep], hc1[keep])


# ------------------------------------------------------------------------------------------------ 6. edges, errors
def test_sweep_edge_cases(B, L, series):
    X, U = series["wrench12"]
    ph = _candidates(B, L, 5, seed=16)
    e = B.Engine("wrench12", "f64")
    se, cnt = e.multistep_se_sweep(X, U, HS, ph[:0], dt=DT)
    assert se.shape == (0, L.MAX_H) and cnt == [3000, 2991, 2901]
    se, cnt = e.multistep_se_sweep(X[:50], U[:50], [50, 60], ph, dt=DT)     # no window: rows <= H
    assert cnt == [0, 0] and torch.count_nonzero(se).item() == 0
    r = e.multistep_rmse_sweep(X[:50], U[:50], [1, 50], ph, dt=DT)
    assert r.shape == (5, 2) and np.all(np.isnan(r[:, 1])) and np.all(np.isfinite(r[:, 0]))
    ref = e.multistep_rmse_sweep(X, U, HS, ph, dt=DT)
    for c in range(5):
        e.set_physical(ph[c])
        assert np.allclose(ref[c], e.multistep_rmse(X, U, HS, dt=DT), rtol=1e-12)
    # split over several launches == one launch
    one, _ = e.multistep_se_sweep(X, U, HS, ph, dt=DT)
    ws1 = L.lib.brov_se_sweep_workspace_bytes(1, 3000, 0)
    split, _ = e.multistep_se_sweep(X, U, HS, ph, dt=DT, workspace_cap=2 * ws1)
    assert torch.equal(one, split)
    with pytest.raises(ValueError):
        e.multistep_se_sweep(X, U, [10, 1], ph, dt=DT)
    with pytest.raises(ValueError):
        e.multistep_se_sweep(X, U, HS, ph, dt=DT, workspace=torch.empty(16, dtype=torch.uint8, device=e.device))
    # unsupported engines
    di = B.Engine("di12_u8", "f64")
    with pytest.raises(B.BrovError, match="Fossen models"):
        di.multistep_se_sweep(X[:, :12], np.zeros((len(X), 8)), HS, ph, dt=DT)
    e.set_wrench_lag1(True)
    with pytest.raises(B.BrovError, match="wrench lag"):
        e.multistep_se_sweep(X, U, HS, ph, dt=DT)


def test_sweep_descriptor_is_validated(B, L):
    """Direct C-ABI callers: workspace, horizons, candidate count and shard geometry are checked before any launch."""
    e = B.Engine("thruster8", "f64")
    rows, P = 400, 3
    X = torch.zeros((rows, 12), device="cuda", dtype=torch.float64)
    U = torch.zeros((rows, 8), device="cuda", dtype=torch.float64)
    kp = torch.as_tensor(B.derive_params(np.tile(B.default_physical(), (P, 1))).T.copy(), device="cuda")
    se = torch.zeros((P, 4), device="cuda", dtype=torch.float64)
    big = torch.empty(L.lib.brov_se_sweep_workspace_bytes(P, rows, 1), device="cuda", dtype=torch.uint8)

    def call(n_windows=390, window0=0, row0=0, carry=0, hs=(10,), n_cand=P, ws_bytes=None):
        d = L.SeSweepDesc()
        d.struct_size = C.sizeof(L.SeSweepDesc)
        d.integrator, d.rows, d.n_windows, d.dt = L.RK4, rows, n_windows, DT
        d.X_dev, d.U_dev, d.se_out_dev = X.data_ptr(), U.data_ptr(), se.data_ptr()
        d.n_horizons = len(hs)
        for i, h in enumerate(hs):
            d.horizons[i] = h
        d.n_candidates, d.kp_soa_dev = n_cand, kp.data_ptr()
        d.workspace_dev = big.data_ptr()
        d.workspace_bytes = big.numel() if ws_bytes is None else ws_bytes
        d.lag_carry, d.window0, d.row0 = carry, window0, row0
        return L.lib.brov_multistep_se_sweep(e._h, C.byref(d), None)

    assert call() == 0
    assert call(ws_bytes=L.lib.brov_se_sweep_workspace_bytes(P, 390, 0) - 1) == -1 and b"workspace" in L.lib.brov_last_error()
    assert call(carry=1, ws_bytes=L.lib.brov_se_sweep_workspace_bytes(P, 390, 0)) == -1   # carry needs the lag rows
    assert call(hs=(10, 5)) == -1 and b"ascending" in L.lib.brov_last_error()
    assert call(hs=(0,)) == -1
    assert call(n_cand=-1) == -1
    assert call(n_cand=1 << 30) == -1 and b"2^31" in L.lib.brov_last_error()
    assert call(n_windows=10, window0=5, row0=0) == -1          # rows before the first window need lag_carry
    assert call(n_windows=380, window0=1000, row0=1000, carry=1) == -1 and b"must start at row" in L.lib.brov_last_error()
    depth = e.carry_steps(DT, "rk4")
    need = (1000 * 10 - depth) // 10
    assert call(n_windows=380 - (1000 - need), window0=1000, row0=need, carry=1) == 0
    assert call(n_windows=395, window0=1000, row0=990, carry=1) == -1 and b"exceed" in L.lib.brov_last_error()
    d = L.SeSweepDesc()
    d.struct_size = 8
    assert L.lib.brov_multistep_se_sweep(e._h, C.byref(d), None) == -1 and b"size mismatch" in L.lib.brov_last_error()
    torch.cuda.synchronize()


def test_sweep_shard_of_a_carried_series_equals_the_whole(B, L, series):
    """window0 / row0: a carried-lag shard of the sweep equals the same shard of the single-vehicle evaluator."""
    X, U = series["thruster8"]
    ph = _candidates(B, L, 3, seed=17)
    e = B.Engine("thruster8", "f64")
    H = 10
    depth = e.carry_steps(DT, "rk4")
    row0 = (1000 * H - depth) // H
    whole = []
    for c in range(3):
        e.set_physical(ph[c])
        s, _ = e.multistep_se(X[row0:1600], U[row0:1600], [H], dt=DT, lag_mode="carry", window0=1000, row0=row0,
                              n_windows=500)
        whole.append(s[0].item())
    kp = torch.as_tensor(B.derive_params(ph).T.copy(), device="cuda")
    Xs, Us = e.tensor(X[row0:1600]), e.tensor(U[row0:1600])
    se = torch.zeros((3, 4), device="cuda", dtype=torch.float64)
    ws = torch.empty(L.lib.brov_se_sweep_workspace_bytes(3, 500, 1), device="cuda", dtype=torch.uint8)
    d = L.SeSweepDesc()
    d.struct_size = C.sizeof(L.SeSweepDesc)
    d.integrator, d.rows, d.n_windows, d.dt = L.RK4, 1600 - row0, 500, DT
    d.X_dev, d.U_dev, d.se_out_dev = Xs.data_ptr(), Us.data_ptr(), se.data_ptr()
    d.n_horizons, d.horizons[0] = 1, H
    d.n_candidates, d.kp_soa_dev = 3, kp.data_ptr()
    d.workspace_dev, d.workspace_bytes = ws.data_ptr(), ws.numel()
    d.lag_carry, d.window0, d.row0 = 1, 1000, row0
    L.check(L.lib.brov_multistep_se_sweep(e._h, C.byref(d), None))
    assert _rel(se[:, 0].cpu().numpy(), np.array(whole)) <= 1e-12


# ------------------------------------------------------------------------------------------------ 7. full size
def test_sweep_full_size_tank_series(B, L):
    """P = 256 on a series as long as the reference's tank recording (45,823 rows), reset and carried lag."""
    X, U = _series(B, "thruster8", 45823, seed=7)
    ph = _candidates(B, L, 256, seed=18)
    e = B.Engine("thruster8", "f64")
    Xt, Ut = e.tensor(X), e.tensor(U)
    pick = [0, 77, 200, 255]
    se, cnt = e.multistep_se_sweep(Xt, Ut, HS, ph, dt=DT)
    assert cnt == [45822, 45813, 45723]
    assert _rel(se.cpu().numpy()[pick, :3], _per_candidate(e, Xt, Ut, HS, ph[pick], "rk4")[:, :3]) <= 1e-12
    for H in HS:
        se, _ = e.multistep_se_sweep(Xt, Ut, [H], ph, dt=DT, lag_mode="carry")
        ref = _per_candidate(e, Xt, Ut, [H], ph[pick], "rk4", lag_mode="carry")[:, 0]
        assert _rel(se.cpu().numpy()[pick, 0], ref) <= 1e-12


def test_evaluator_wrapper_and_sharded_sweep(B, L, series):
    from bluerov2_dynamics_b200 import dist as D
    from bluerov2_dynamics_b200.evaluators import multistep_rmse_endpoint_physics, multistep_rmse_endpoint_physics_sweep
    X, U = series["thruster8"]
    X, U = X[:600], U[:600]
    ph = _candidates(B, L, 6, seed=19)
    got = multistep_rmse_endpoint_physics_sweep(X, U, [1, 10], DT, ph)          # carry mode by default
    assert got.shape == (6, 2)
    e = B.Engine("thruster8", "f64")
    for c in range(6):
        e.set_physical(ph[c])
        ref = multistep_rmse_endpoint_physics(X, U, [1, 10], DT, engine=e)
        assert np.allclose(got[c], ref, rtol=1e-12)
    assert multistep_rmse_endpoint_physics_sweep(X, U, 10, DT, ph, lag_mode="reset").shape == (6,)
    eng = B.Engine("thruster8", "f64")
    full, _ = eng.multistep_se_sweep(X, U, HS, ph, dt=DT)
    sharded = D.sharded_sweep(lambda lo, hi: eng.multistep_se_sweep(X, U, HS, ph[lo:hi], dt=DT)[0], 6, 0, 1)
    assert torch.equal(sharded, full)
