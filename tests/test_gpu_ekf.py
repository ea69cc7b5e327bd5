"""GPU tests of the extended Kalman filter (brov_ekf through Engine.ekf): it agrees with the numpy filter of
oracle/ekf_np.py run on the exact step and Jacobian of Engine.linearize and on independent central differences of the
numpy model, prediction alone reproduces the rollout and the covariance recursion, the filter is statistically
consistent (NEES and NIS), P stays exactly symmetric and positive definite over long runs, operand layouts /
permutation / chunking / repeats leave the bits unchanged, every row of a noise sweep equals its own single-filter
call and the likelihood finds the noise level that generated the data, the health counters and refusals work, and a
covariance trajectory above 2^31 elements is indexed correctly."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy import stats as st

from oracle import ekf_np
from oracle import fossen_np as O

pytestmark = pytest.mark.gpu

DT = 0.02
MODELS = ("thruster8", "wrench12")
CASES = [(m, i, c) for m in MODELS for i in ("rk4", "euler") for c in (False, True)]
IDS = [f"{m}-{i}-{'current' if c else 'still'}" for m, i, c in CASES]
CURRENT = (0.12, -0.07, 0.05)
# measurement noise standard deviations: position, Euler angles, linear velocity, angular velocity
R_STD = np.repeat([0.05, 0.01, 0.02, 0.01], 3)
Q_VAR = np.repeat([1e-8, 1e-8, 1e-6, 1e-6], 3)


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


def _np(t):
    return t.cpu().numpy()


def _normwise(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _scenario(e, n, T, seed, miss=0.3, integ="rk4"):
    """n vehicles from moderate states under smooth inputs: (x0 [n,12], L24 [n,8,3] or None, U [T,n,NU],
    truth [T,n,12], Y [T,n,12] with measurement noise R_STD and a random fraction `miss` of NaNs)"""
    rng = np.random.default_rng(seed)
    x0 = np.zeros((n, 12))
    x0[:, :3] = rng.uniform(-2, 2, (n, 3))
    x0[:, 3:6] = np.stack([rng.uniform(-0.3, 0.3, n), rng.uniform(-0.3, 0.3, n), rng.uniform(-3, 3, n)], axis=1)
    x0[:, 6:] = rng.uniform(-0.2, 0.2, (n, 6))
    thr = e.model == "thruster8"
    L24 = rng.uniform(-0.3, 0.3, (n, 8, 3)) if thr else None
    U = O.smooth_inputs(rng, T, e.nu, n=n, scale=0.5 if thr else 3.0, sigma=0.05)
    r = e.rollout(x0, U, dt=DT, integrator=integ, stride=1, lag0=L24.reshape(n, 24) if thr else None)
    truth = _np(r.traj)
    Y = truth + R_STD * rng.standard_normal(truth.shape)
    Y[rng.random(Y.shape) < miss] = np.nan
    return x0, L24, U, truth, Y


def _p0(n):
    return np.tile(np.diag(np.repeat([0.1, 0.01, 0.01, 0.01], 3)), (n, 1, 1))


def _ekf(e, x0, L24, U, Y, integ="rk4", q=Q_VAR, r=R_STD ** 2, P0=None, **kw):
    n = x0.shape[0]
    return e.ekf(x0, _p0(n) if P0 is None else P0, U, Y, q, r, dt=DT, integrator=integ,
                 lag0=None if L24 is None else L24.reshape(n, 24), **kw)


def _lin_step_jac(e, integ):
    """(step, jac) for ekf_np on Engine.linearize with T = 1: aux is the projected lag [N, 18] (None for wrench12).
    ekf_np calls jac and then step at the same point, so step returns what jac's call computed."""
    thr = e.model == "thruster8"
    last = {}

    def jac(x, aux, u):
        res = e.linearize(x, u, dt=DT, integrator=integ, lag0=aux, lag_repr="projected", want_traj=False)
        z = _np(res.z)
        last["next"] = (z[:, :e.nx], z[:, e.nx:] if thr else None)
        return _np(res.A[0, :, :e.nx, :e.nx])

    def step(x, aux, u):
        return last.pop("next")
    return step, jac


def _check(out, ref, tx, tp, tl):
    assert _normwise(_np(out.x_traj), ref["x_traj"]) <= tx
    assert _normwise(_np(out.P_traj), ref["P_traj"]) <= tp
    assert _normwise(_np(out.loglik), ref["loglik"]) <= tl
    assert _normwise(_np(out.nis), ref["nis"]) <= tl
    assert np.array_equal(_np(out.count), ref["count"])


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_matches_the_oracle_on_the_exact_step_and_jacobian(B, model, integ, cur):
    e = _engine(B, model, cur)
    n, T = 64, 200
    x0, L24, U, _, Y = _scenario(e, n, T, 1, integ=integ)
    out = _ekf(e, x0, L24, U, Y, integ=integ, stride=1, want_cov=True)
    step, jac = _lin_step_jac(e, integ)
    Z0 = _np(e.project_lag(L24.reshape(n, 24))) if L24 is not None else None
    ref = ekf_np.ekf(step, jac, x0, Z0, _p0(n), U, Y, Q_VAR, R_STD ** 2)
    _check(out, ref, 1e-10, 1e-9, 1e-10)
    assert np.array_equal(_np(out.count), np.isfinite(Y).sum(axis=(0, 2)))


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_matches_the_independent_oracle(B, model, integ, cur):
    """Against the numpy model with central-difference Jacobians (h = 1e-5 relative): their truncation error is
    O(h^2 |f'''|) ~ 1e-10 and their rounding error O(eps / h) ~ 1e-11 per entry of A, which the covariance recursion
    carries into P at about 1e-8 relative and, through the gains, into x at about 1e-9; the bars leave a margin of
    100 and 10."""
    e = _engine(B, model, cur)
    n, T = 64, 200
    x0, L24, U, _, Y = _scenario(e, n, T, 2, integ=integ)
    out = _ekf(e, x0, L24, U, Y, integ=integ, stride=1, want_cov=True)
    m = O.Model(model, DT, O.default_params(current=CURRENT if cur else (0.0, 0.0, 0.0)))
    step, jac = ekf_np.fossen_step_jac(m, integ)
    ref = ekf_np.ekf(step, jac, x0, L24, _p0(n), U, Y, Q_VAR, R_STD ** 2)
    _check(out, ref, 1e-8, 1e-6, 1e-8)


@pytest.mark.parametrize("model,integ,cur", CASES, ids=IDS)
def test_prediction_only_is_the_rollout_and_the_covariance_recursion(B, model, integ, cur):
    e = _engine(B, model, cur)
    n, T = 37, 100
    x0, L24, U, truth, Y = _scenario(e, n, T, 3, integ=integ)
    out = _ekf(e, x0, L24, U, np.full_like(Y, np.nan), integ=integ, stride=1, want_cov=True)
    assert _normwise(_np(out.x_traj), truth) <= 1e-12
    lin = e.linearize(x0, U, dt=DT, integrator=integ, lag0=None if L24 is None else L24.reshape(n, 24))
    A = _np(lin.A[:, :, :12, :12])
    P = _p0(n)
    Ps = []
    for k in range(T):
        P = A[k] @ P @ np.swapaxes(A[k], 1, 2) + np.diag(Q_VAR)
        Ps.append(P)
    assert _normwise(_np(out.P_traj), np.array(Ps)) <= 1e-12
    assert torch.equal(out.z, lin.z) and np.all(_np(out.count) == 0) and np.all(_np(out.loglik) == 0)


def _wrap(a):
    return a - 2 * np.pi * np.rint(a / (2 * np.pi))


@pytest.mark.parametrize("model", MODELS)
def test_consistency_nees_and_nis(B, model):
    """2000 seeded realisations x 200 steps: truth with process noise N(0, diag q) added after every engine step and
    measurements with noise N(0, diag r); the mean NEES at several steps and the mean NIS lie in their 99 % chi^2
    intervals."""
    e = _engine(B, model)
    n, T = 2000, 200
    rng = np.random.default_rng(4)
    thr = model == "thruster8"
    x0, _, U, _, _ = _scenario(e, n, T, 5, miss=0.0)
    Z = np.zeros((n, 18)) if thr else None
    P0 = np.diag(np.repeat([0.01, 1e-4, 1e-4, 1e-4], 3))
    xt = x0 + rng.multivariate_normal(np.zeros(12), P0, n)
    X = []
    for k in range(T):
        r = e.rollout(xt, U[k:k + 1], dt=DT, lag0=Z, lag_repr="projected")
        xt = _np(r.xT) + np.sqrt(Q_VAR) * rng.standard_normal((n, 12))
        Z = _np(r.lag) if thr else None
        X.append(xt)
    X = np.array(X)
    Y = X + R_STD * rng.standard_normal(X.shape)
    Y[:, :, :3][rng.random((T, n, 3)) < 0.8] = np.nan                  # position fixes at a fifth of the steps
    out = e.ekf(x0, P0, U, Y, Q_VAR, R_STD ** 2, dt=DT, stride=1, want_cov=True)
    xe, Pe = _np(out.x_traj), _np(out.P_traj)
    lo, hi = st.chi2.ppf([0.005, 0.995], 12 * n) / n
    for k in (9, 49, 99, 199):
        err = X[k] - xe[k]
        err[:, 3:6] = _wrap(err[:, 3:6])
        nees = np.einsum("ni,ni->n", err, np.linalg.solve(Pe[k], err[:, :, None])[:, :, 0])
        assert lo <= nees.mean() <= hi, (k, nees.mean(), lo, hi)
    m = int(_np(out.count).sum())
    lo, hi = st.chi2.ppf([0.005, 0.995], m) / m
    assert lo <= _np(out.nis).sum() / m <= hi


@pytest.mark.parametrize("model", MODELS)
def test_long_run_keeps_p_symmetric_and_positive_definite(B, model):
    e = _engine(B, model)
    n, T = 16, 20000
    rng = np.random.default_rng(6)
    x0, L24, U, truth, _ = _scenario(e, n, T, 7, integ="euler")
    Y = truth + 1e-4 * rng.standard_normal(truth.shape)
    out = _ekf(e, x0, L24, U, Y, integ="euler", q=np.full(12, 1e-14), r=np.full(12, 1e-8), stride=500,
               want_cov=True)
    P = _np(out.P_traj)
    assert np.array_equal(P, np.swapaxes(P, -1, -2))
    np.linalg.cholesky(P)                                # raises unless every snapshot is positive definite
    assert np.all(np.isfinite(_np(out.z)))
    assert _normwise(_np(out.x_traj), truth[499::500]) <= 1e-3


@pytest.mark.parametrize("model", MODELS)
def test_layouts_permutation_chunking_and_repeats_give_the_same_bits(B, model):
    e = _engine(B, model, True)
    n, T = 101, 60                                       # ragged: not a multiple of the filters per block
    x0, L24, U, _, Y = _scenario(e, n, T, 8)
    rng = np.random.default_rng(9)
    qn = Q_VAR * rng.uniform(0.5, 2.0, (n, 12))
    rn = R_STD ** 2 * rng.uniform(0.5, 2.0, (n, 12))
    ref = _ekf(e, x0, L24, U, Y, q=qn, r=rn, stride=7, want_cov=True, health=True)

    def same(a, b):
        return (torch.equal(a.z, b.z) and torch.equal(a.P, b.P) and torch.equal(a.loglik, b.loglik)
                and torch.equal(a.nis, b.nis) and torch.equal(a.count, b.count))
    assert same(ref, _ekf(e, x0, L24, U, Y, q=qn, r=rn, stride=7, want_cov=True))
    # +-inf in Y is not a measurement, exactly as NaN
    assert same(ref, _ekf(e, x0, L24, U, np.where(np.isnan(Y), np.inf, Y), q=qn, r=rn))
    # shared operands against per-filter copies of them
    a = _ekf(e, x0, L24, U[:, 0], Y[:, 0])
    b = _ekf(e, x0, L24, np.repeat(U[:, :1], n, axis=1), np.repeat(Y[:, :1], n, axis=1), q=np.tile(Q_VAR, (n, 1)),
             r=np.tile(R_STD ** 2, (n, 1)))
    assert same(a, b)
    c = _ekf(e, x0, L24, U[0], Y, u_layout="const")
    d = _ekf(e, x0, L24, np.repeat(U[:1], T, axis=0), Y)
    assert same(c, d)
    # the filter order
    perm = rng.permutation(n)
    p = _ekf(e, x0[perm], L24[perm] if L24 is not None else None, U[:, perm], Y[:, perm], q=qn[perm], r=rn[perm],
             stride=7, want_cov=True)
    assert torch.equal(p.z, ref.z[perm]) and torch.equal(p.P, ref.P[perm]) and torch.equal(p.loglik, ref.loglik[perm])
    assert torch.equal(p.P_traj, ref.P_traj[:, perm]) and torch.equal(p.x_traj, ref.x_traj[:, perm])
    # two chunks carrying z, P and the statistics
    h = 25
    c1 = _ekf(e, x0, L24, U[:h], Y[:h], q=qn, r=rn)
    stats = (c1.loglik.clone(), c1.nis.clone(), c1.count.clone())
    c2 = e.ekf(c1.z[:, :12], c1.P, U[h:], Y[h:], qn, rn, dt=DT, lag0=c1.z[:, 12:] if model == "thruster8" else None,
               lag_repr="projected", stats=stats, stats_accumulate=True)
    assert same(c2, ref) and c2.loglik.data_ptr() == stats[0].data_ptr()
    # a yaw measurement offset by 2 pi: y + 2 pi rounds to a coarser grid than y, so the innovations agree to a few
    # ulps of 2 pi, not bit for bit
    Y2 = Y.copy()
    Y2[:, :, 5] += 2 * np.pi
    w = _ekf(e, x0, L24, U, Y2, q=qn, r=rn)
    assert _normwise(_np(w.z[:, :12]), _np(ref.z[:, :12])) <= 1e-12
    assert _normwise(_np(w.P), _np(ref.P)) <= 1e-12 and torch.equal(w.count, ref.count)
    # N = 1, n = 0 and steps = 0
    one = _ekf(e, x0[5:6], L24[5:6] if L24 is not None else None, U[:, 5:6], Y[:, 5:6], q=qn[5:6], r=rn[5:6])
    assert torch.equal(one.z, ref.z[5:6]) and torch.equal(one.P, ref.P[5:6]) and torch.equal(one.loglik, ref.loglik[5:6])
    z0 = _ekf(e, x0[:0], L24[:0] if L24 is not None else None, U[:, :0], Y[:, :0])
    assert z0.z.shape == (0, e.nz) and z0.P.shape == (0, 12, 12)
    s0 = _ekf(e, x0, L24, U[:0], Y[:0], stride=1, want_cov=True)
    assert torch.equal(s0.z[:, :12], e.tensor(x0)) and torch.equal(s0.P, e.tensor(_p0(n)))
    assert torch.all(s0.loglik == 0) and torch.all(s0.count == 0) and s0.x_traj.shape == (0, n, 12)


def test_noise_sweep_rows_equal_single_filters_and_the_likelihood_finds_q(B):
    e = _engine(B, "wrench12")
    T = 2000
    rng = np.random.default_rng(10)
    U = O.smooth_inputs(rng, T, 6, scale=3.0, sigma=0.05)
    q_true = 4.0 * Q_VAR
    x = np.zeros((1, 12))
    X = []
    for k in range(T):
        x = _np(e.rollout(x, U[k:k + 1]).xT) + np.sqrt(q_true) * rng.standard_normal((1, 12))
        X.append(x[0])
    r_std = R_STD / 4                                   # accurate sensors: the innovations see q
    Y = np.array(X) + r_std * rng.standard_normal((T, 12))
    scales = 2.0 ** np.arange(-4, 9)                    # one grid step = a factor of 2; the truth is 2^2
    P0 = np.diag(np.full(12, 1e-4))
    res = e.ekf(np.zeros((len(scales), 12)), P0, U, Y, scales[:, None] * Q_VAR, r_std ** 2, dt=DT)
    best = int(np.argmax(_np(res.loglik)))
    assert abs(np.log2(scales[best]) - 2) <= 1, _np(res.loglik)
    # 64 filters with different q, each equal to its own single-filter call
    q64 = Q_VAR * 2.0 ** rng.uniform(-4, 8, (64, 1))
    sw = e.ekf(np.zeros((64, 12)), P0, U[:300], Y[:300], q64, r_std ** 2, dt=DT)
    for i in range(64):
        one = e.ekf(np.zeros((1, 12)), P0, U[:300], Y[:300], q64[i], r_std ** 2, dt=DT)
        assert torch.equal(one.z[0], sw.z[i]) and torch.equal(one.P[0], sw.P[i])
        assert torch.equal(one.loglik[0], sw.loglik[i]) and torch.equal(one.nis[0], sw.nis[i])


@pytest.mark.parametrize("model", MODELS)
def test_health_counters(B, model):
    e = _engine(B, model)
    n = 50
    x0, L24, U, _, Y = _scenario(e, n, 5, 11)
    assert _ekf(e, x0, L24, U, Y, health=True).health.tolist() == [0, 0]
    x = x0.copy()
    x[[3, 17], 6] = np.nan
    x[[4, 20, 41], 4] = np.pi / 2 - 1e-4                 # |cos theta| = 1e-4 < 1e-3
    Yb = Y.copy()
    Yb[:, [4, 20, 41], 4] = np.nan                       # let the filters stay near the singularity
    r = _ekf(e, x, L24, U, Yb, health=True)
    assert r.health.tolist() == [2, 3]


def test_unsupported_and_invalid_calls(B, L):
    e = _engine(B, "thruster8")
    n = 4
    x0, L24, U, _, Y = _scenario(e, n, 3, 12)
    q, r = Q_VAR, R_STD ** 2
    for eng in (B.Engine("thruster8", "f32"), B.Engine("quat13", "f64")):
        with pytest.raises(B.BrovError, match="-4"):
            eng.ekf(x0 if eng.nx == 12 else np.zeros((n, 13)), np.eye(eng.nx), np.zeros((3, n, eng.nu)),
                    np.zeros((3, n, eng.nx)), np.ones(eng.nx), np.ones(eng.nx))
    di = B.Engine("di12_u8", "f64")
    di.set_di_gains(np.full((8, 3), 0.1), np.full((8, 3), 0.1))
    with pytest.raises(B.BrovError, match="-4"):
        di.ekf(x0, np.eye(12), U, Y, q, r)
    w = B.Engine("wrench12", "f64")
    w.set_wrench_lag1(True, 0.1)
    with pytest.raises(B.BrovError, match="-4"):
        w.ekf(x0, np.eye(12), np.zeros((3, n, 6)), Y, q, r)
    e.set_vehicle_physical(np.tile(B.default_physical(), (n, 1)))
    with pytest.raises(B.BrovError, match="-4"):
        e.ekf(x0, np.eye(12), U, Y, q, r)
    e.set_vehicle_physical(None)
    e.ekf(x0, np.eye(12), U, Y, q, r)                    # fine again once the table is cleared
    for qq, rr in ((-q, r), (q, 0 * r), (q, -r), (q, np.where(np.arange(12) == 3, np.nan, r)),
                   (np.where(np.arange(12) == 0, np.nan, q), r), (np.tile(q, (n, 1)) * [[1], [1], [-1], [1]], r)):
        with pytest.raises(B.BrovError, match="-1"):
            e.ekf(x0, np.eye(12), U, Y, qq, rr)
    with pytest.raises(B.BrovError, match="-1"):
        e.ekf(x0, np.eye(12), U, Y, q, r, dt=-0.02)
    for bad in (dict(U=U[:2]), dict(U=U[..., :6]), dict(Y=Y[..., :11]), dict(q=q[:11]), dict(P0=np.eye(11))):
        kw = dict(U=U, Y=Y, q=q, r=r, P0=np.eye(12))
        kw.update(bad)
        with pytest.raises(ValueError):
            e.ekf(x0, kw["P0"], kw["U"], kw["Y"], kw["q"], kw["r"])
    # the C ABI: NULL operands, a trajectory without a stride, negative strides; n = 0 is a no-op
    t = e.tensor(np.zeros((n, 30)))
    P = e.tensor(np.tile(np.eye(12), (n, 1, 1)))
    d = L.EkfDesc()
    d.struct_size = C.sizeof(L.EkfDesc)
    d.n, d.steps, d.dt = n, 1, DT
    d.z0_dev, d.P0_dev, d.z_out_dev, d.P_out_dev = t.data_ptr(), P.data_ptr(), t.data_ptr(), P.data_ptr()
    assert L.lib.brov_ekf(e._h, C.byref(d), None) == -1                   # u, y, q, r NULL
    d.u_dev = d.y_dev = d.q_dev = d.r_dev = P.data_ptr()
    d.x_traj_dev = t.data_ptr()
    assert L.lib.brov_ekf(e._h, C.byref(d), None) == -1                   # stride 0 with a trajectory
    d.x_traj_dev = None
    d.y_stride_n = -1
    assert L.lib.brov_ekf(e._h, C.byref(d), None) == -1
    d.y_stride_n = 0
    d.n = 0
    assert L.lib.brov_ekf(e._h, C.byref(d), None) == 0
    d.struct_size = 8
    assert L.lib.brov_ekf(e._h, C.byref(d), None) == -1


def test_covariance_trajectory_above_2_31_elements(B):
    e = _engine(B, "wrench12")
    n, T = 65536, 230
    assert T * n * 144 > 2 ** 31
    rng = np.random.default_rng(13)
    x0 = np.zeros((n, 12))
    x0[:, 5] = rng.uniform(-3, 3, n)
    U = torch.as_tensor(O.smooth_inputs(rng, T, 6, scale=3.0, sigma=0.05), device="cuda")
    Y = torch.full((T, 12), float("nan"), dtype=torch.float64, device="cuda")
    Y[::3, 2] = 0.1
    q = Q_VAR * (1 + np.arange(12) / 12)
    r = e.ekf(x0, np.diag(np.full(12, 1e-3)), U, Y, q, R_STD ** 2, dt=DT, stride=1, want_cov=True)
    pick = np.array([0, 1, 2, 12345, 56491, n - 2, n - 1])
    s = e.ekf(x0[pick], np.diag(np.full(12, 1e-3)), U, Y, q, R_STD ** 2, dt=DT, stride=1, want_cov=True)
    assert torch.equal(r.P_traj[:, pick], s.P_traj) and torch.equal(r.x_traj[:, pick], s.x_traj)
    assert torch.equal(r.P[pick], s.P)
    del r
    torch.cuda.empty_cache()
