"""The CPU oracles against the UNMODIFIED reference executed live from oracle/_ref/ (byte-compiled by
oracle/build_ref.py from a copy of the reference project, which the repository does not contain; skipped where
oracle/_ref is not built): fresh seeded inputs every run of the suite would be pointless, so the seeds are fixed — what
this adds to the frozen golden files is that the comparison runs against the reference ITSELF wherever it is built."""
import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import fossen_np as O
from oracle import ref_loader as RL
from conftest import normwise

pytestmark = [pytest.mark.skipif(not RL.available(), reason="oracle/_ref not built (oracle/build_ref.py needs a copy of the reference project)"),
              pytest.mark.filterwarnings("ignore")]
DT = 0.02


def test_rk4_rollout_and_hidden_lag_against_live_reference():
    R = RL.load()
    rng = np.random.default_rng(77)
    T, n = 150, 3
    x0 = np.zeros((n, 12))
    x0[:, :3] = rng.uniform(-1, 1, (n, 3))
    x0[:, 3:5] = rng.uniform(-0.2, 0.2, (n, 2))
    x0[:, 5] = rng.uniform(-3, 3, n)
    U = O.smooth_inputs(rng, T, 8, n=n, sigma=0.05)
    want_x, want_lag = [], []
    for i in range(n):
        rov = R.BlueROV2(dt=DT)
        traj = R.simulate_physics(x0[i], U[:, i], DT, rov)          # training/train_tank_brov2_rk4.py:375-396
        want_x.append(traj)
        want_lag.append(np.stack([np.asarray(l._x, float).reshape(3) for l in rov.thruster_lags]))
    want_x, want_lag = np.array(want_x), np.array(want_lag)
    snaps, xT, lagT = O.rollout(O.Model("thruster8", DT), "rk4", x0, U, stride=1)
    assert normwise(np.transpose(snaps, (1, 0, 2)), want_x[:, 1:]) < 1e-12 and normwise(lagT, want_lag) < 1e-12
    if CO.available():
        snaps_c, _, lag_c = CO.rollout("thruster8", "rk4", DT, x0, U, stride=1)
        assert normwise(np.transpose(snaps_c, (1, 0, 2)), want_x[:, 1:]) < 1e-12 and normwise(lag_c, want_lag) < 1e-12


def test_endpoint_rmse_against_live_reference():
    """multistep_rmse_endpoint_physics (training/train_tank_brov2_rk4.py:399-417), the reference's literal semantics:
    ONE model object scores all windows, its lag state carried from window to window."""
    R = RL.load()
    rng = np.random.default_rng(78)
    T = 60
    U = O.smooth_inputs(rng, T, 8, sigma=0.05)
    _, _, _ = None, None, None
    X = np.zeros((T, 12))
    X[:, :3] = np.cumsum(rng.normal(0, 0.01, (T, 3)), axis=0)
    X[:, 5] = np.cumsum(rng.normal(0, 0.01, T))
    X[:, 6:] = rng.normal(0, 0.05, (T, 6))
    m = O.Model("thruster8", DT)
    for H in (1, 5):
        want = R.multistep_rmse_endpoint_physics(X, U, H, DT)
        got = O.multistep_se(m, "rk4", X, U, [H], lag_mode="carry")[H][2]
        assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (H, got, want)


def test_mirror_private_helpers_against_live_reference():
    """_coriolis / _damping / _restoring of the model mirrors (host numpy, attribute surface only) against the
    reference's own methods (fossen/BlueROV2.py:280-355), including after an attribute edit."""
    import bluerov2_dynamics_b200.fossen._base as Bm
    R = RL.load()

    class M(Bm.FossenModelBase):
        pass
    m = M()
    m._init_constants(1000.0, None)
    ref = R.BlueROV2()
    rng = np.random.default_rng(5)
    for obj in (m, ref):
        obj.Xu_dot, obj.Nr_abs, obj.zb = -7.5, -2.0, -0.02
    for _ in range(5):
        nu = rng.normal(size=6)
        assert np.array_equal(m._coriolis(nu), ref._coriolis(nu)) or np.allclose(m._coriolis(nu), ref._coriolis(nu), rtol=1e-15)
        assert np.allclose(m._damping(nu), ref._damping(nu), rtol=1e-15)
        a = rng.uniform(-1, 1, 3)
        assert np.allclose(m._restoring(*a), ref._restoring(*a), rtol=1e-15, atol=1e-18)
