"""Drop-in versions of the free functions the reference's training scripts define around the models:
`simulate_physics`, `one_step_rmse_physics`, `multistep_rmse_endpoint_physics` (training/train_tank_brov2_rk4.py:375-417
and the Euler twins in train_tank_brov2_full_comparison.py:453-487, train_tank_brov2_koopmanEDMDc.py:222-283,
train_tank_brov2_wrench_comp.py:208-250, train_tank_brov2_wrench_quat.py:249-297).

The reference picks the integrator by which script the function sits in (RK4 in train_tank_brov2_rk4.py, explicit
Euler everywhere else); here it is the `integrator` argument.  One kernel launch replaces the Python loop over
steps (rollout) or the double loop over windows and steps (evaluators)."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

from .engine import PHYS_NAMES, Engine, parameter_indices, with_minv
from .fossen.BlueROV2 import BlueROV2 as _Thruster


def _model_of(rov):
    return rov._MODEL


def simulate_physics(x0: np.ndarray, U_seq: np.ndarray, dt: float, rov, integrator: str = "rk4") -> np.ndarray:
    """Open-loop rollout of one vehicle under the recorded inputs; returns the trajectory [len(U_seq)+1, n_states]
    with row 0 = x0.  For the 8-thruster model the rollout starts from, and leaves behind, `rov`'s lag state — as the
    reference's loop over `rov.dynamics` does."""
    x0 = np.asarray(x0, dtype=float)
    U_seq = np.asarray(U_seq, dtype=float)
    eng = rov.engine("f64")
    H = len(U_seq)
    traj = np.zeros((H + 1, x0.shape[0]))
    traj[0] = x0
    if H == 0:
        return traj
    lag0 = rov._lag_tensor(eng) if isinstance(rov, _Thruster) else None
    res = eng.rollout(x0.reshape(1, -1), U_seq.reshape(H, eng.nu), dt=dt, integrator=integrator, lag0=lag0, stride=1,
                      u_layout="shared")
    traj[1:] = res.traj[:, 0, :].cpu().numpy()
    if lag0 is not None:
        rov._store_lag(res.lag, dt)
    return traj


def _engine_for(X_test, model, dtype, engine):
    if engine is not None:
        return engine
    if model is None:
        model = "quat13" if np.shape(X_test)[1] == 13 else "thruster8"
    return Engine(model, dtype)


def multistep_rmse_endpoint_physics(X_test: np.ndarray, U_test: np.ndarray, H, dt: float, model: str = None,
                                    integrator: str = "rk4", dtype: str = "f64", engine: Engine = None,
                                    lag_mode: str = "carry"):
    """Strict H-step-ahead endpoint RMSE over all sliding windows of a recorded series:
    sqrt(sum_k |sim(X[k], U[k:k+H])[-1] - X[k+H]|^2 / ((T-H) * n_states)), NaN if T <= H.  `H` may be a list.

    lag_mode="carry" (default) is the reference's literal behaviour for the 8-thruster model: ONE model object scores
    all windows in order, so the thruster-lag state leaks from window to window (SURVEY trap T3).
    lag_mode="reset" starts every window from zero lag state, and scores all horizons in a single pass.
    The wrench-input models have no hidden state: both modes coincide."""
    eng = _engine_for(X_test, model, dtype, engine)
    return eng.multistep_rmse(X_test, U_test, H, dt=dt, integrator=integrator, lag_mode=lag_mode)


def multistep_rmse_endpoint_physics_sweep(X_test: np.ndarray, U_test: np.ndarray, H, dt: float, phys_table: np.ndarray,
                                          model: str = None, lag_mode: str = "carry", dtype: str = "f64",
                                          integrator: str = "rk4", engine: Engine = None) -> np.ndarray:
    """`multistep_rmse_endpoint_physics` for P candidate vehicles at once: phys_table [P, NPHYS] holds one physical
    vector per candidate (engine.with_minv rebuilds diag(Minv) after the masses are perturbed).  Returns the RMSE as a
    numpy array [P] for a scalar H, [P, len(H)] for a list; NaN where T <= H.  Same lag modes as the single-vehicle
    function (carry: the thruster lag leaks from window to window; the carried state is shared by all candidates)."""
    eng = _engine_for(X_test, model, dtype, engine)
    out = eng.multistep_rmse_sweep(X_test, U_test, H, phys_table, dt=dt, integrator=integrator, lag_mode=lag_mode)
    return out[:, 0] if np.isscalar(H) else out


@dataclass
class CalibrationResult:
    phys: np.ndarray                 # fitted physical vector [NPHYS] (diag(Minv) rebuilt when rebuild_minv)
    names: list                      # fitted parameters
    theta: np.ndarray                # their fitted values [p]
    rmse: dict                       # horizon -> endpoint RMSE of the fitted vehicle
    gn: np.ndarray                   # final Gauss-Newton matrix of the objective in the parameters [p, p]
    cost: float                      # final objective
    cost0: float                     # objective at phys0
    iterations: int
    converged: bool
    history: list = field(default_factory=list)   # per iteration: cost, lam, step_norm, accepted


def calibrate_physical(X: np.ndarray, U: np.ndarray, dt: float, phys0: np.ndarray, params, horizons=(1, 10, 100),
                       weights=None, model: str = None, integrator: str = "rk4", lag_mode: str = "carry",
                       bounds=None, max_iter: int = 50, tol: float = 1e-10, engine: Engine = None,
                       rebuild_minv: bool = True, lambdas=(0.1, 1.0, 10.0)) -> CalibrationResult:
    """Levenberg-Marquardt fit of physical parameters to a recorded series by the reference's endpoint error:
    minimises  sum_h w_h se_h / (count_h NX)  (the squared endpoint RMSE per horizon, weighted; w_h = 1 by default)
    over the selected parameters (PH_* indices, attribute names or groups, see engine.parameter_indices), starting
    from phys0.  Works in relative units theta_j / theta0_j (1 where theta0_j = 0) so that masses, damping terms and
    currents are on one scale.  Every iteration makes one Engine.multistep_se_grad call (cost, exact gradient, Gauss-
    Newton matrix) and scores the trial steps of all damping values `lambdas` x lam in one multistep_se_sweep call;
    the best trial that lowers the cost is taken, otherwise lam grows tenfold.  bounds: (lo, hi) arrays [p] in
    physical units, enforced by projection.  Stops when the relative cost decrease or the relative step falls below
    tol, or after max_iter iterations.  fp64 engines only.  Raises FloatingPointError where the error or its derivatives
    are not finite (windows through the Euler-angle singularity theta = +-pi/2)."""
    eng = _engine_for(X, model, "f64", engine)
    if eng.dtype != "f64":
        raise ValueError("calibrate_physical needs an fp64 engine")
    hs = sorted(int(h) for h in horizons)
    w = np.ones(len(hs)) if weights is None else np.asarray(weights, float).reshape(len(hs))
    idx = parameter_indices(params)
    ph = np.array(phys0, dtype=np.float64).reshape(-1)
    if rebuild_minv:
        ph = with_minv(ph)
    th0 = ph[idx].copy()
    scale = np.where(th0 != 0.0, np.abs(th0), 1.0)
    lo = hi = None
    if bounds is not None:
        lo, hi = (np.asarray(b, float).reshape(len(idx)) for b in bounds)
    carry = lag_mode == "carry" and eng.model == "thruster8"
    Xt, Ut = eng.tensor(X), eng.tensor(U)

    def vehicle(theta):
        q = ph.copy()
        q[idx] = theta
        return with_minv(q) if rebuild_minv else q

    def project(theta):
        return theta if lo is None else np.clip(theta, lo, hi)

    def trial_costs(table):
        tot = np.zeros(table.shape[0])
        for part in ([[h] for h in hs] if carry else [hs]):
            se, cnt = eng.multistep_se_sweep(Xt, Ut, part, table, dt=dt, integrator=integrator, lag_mode=lag_mode)
            se = se.cpu().numpy()
            for j, h in enumerate(part):
                if cnt[j] > 0:
                    tot += w[hs.index(h)] * se[:, j] / (cnt[j] * eng.nx)
        return np.where(np.isfinite(tot), tot, np.inf)

    health = torch.zeros(2, dtype=torch.int64, device=eng.device)

    def evaluate(theta):
        r = eng.multistep_se_grad(Xt, Ut, hs, vehicle(theta), idx, dt=dt, integrator=integrator, lag_mode=lag_mode,
                                  rebuild_minv=rebuild_minv, health_out=health)
        se, g, G = r.se.cpu().numpy(), r.grad.cpu().numpy(), r.gn.cpu().numpy()
        c = np.array([w[i] / (r.counts[i] * eng.nx) if r.counts[i] > 0 else 0.0 for i in range(len(hs))])
        cost, g, G = float(c @ se), c @ g, 2.0 * np.einsum("h,hij->ij", c, G)
        if not (np.isfinite(cost) and np.all(np.isfinite(g)) and np.all(np.isfinite(G))):
            n_bad, n_sing = (int(v) for v in health.tolist())
            raise FloatingPointError(
                f"the endpoint error or its derivatives are not finite at this vehicle ({n_bad} windows with a "
                f"non-finite error, {n_sing} within 1e-3 of theta = +-pi/2, where the Euler-angle kinematics and their "
                "sensitivities blow up): use a series that stays away from the singularity, or the quaternion model")
        return cost, g, G

    theta = project(th0.copy())
    cost, g, G = evaluate(theta)
    cost0, lam, history, converged, it = cost, 1e-3, [], False, 0
    for it in range(1, max_iter + 1):
        gz, Gz = g * scale, G * np.outer(scale, scale)           # relative units z = theta / scale
        dG = np.maximum(np.diag(Gz), 1e-12 * max(np.max(np.diag(Gz)), 1e-300))
        lams = [lam * f for f in lambdas]
        steps = []
        for lm in lams:
            dz = np.linalg.solve(Gz + lm * np.diag(dG), -gz)
            steps.append(project(theta + dz * scale))
        costs = trial_costs(np.stack([vehicle(t) for t in steps]))
        b = int(np.argmin(costs))
        accepted = bool(costs[b] < cost)
        step_norm = float(np.linalg.norm((steps[b] - theta) / scale))
        history.append(dict(cost=float(costs[b] if accepted else cost), lam=float(lams[b]), step_norm=step_norm,
                            accepted=accepted))
        if not accepted:
            lam *= 10.0
            if lam > 1e12 or step_norm <= tol:
                converged = True
                break
            continue
        decrease = (cost - costs[b]) / max(cost, 1e-300)
        theta = steps[b]
        lam = max(lams[b] / 10.0, 1e-12)
        cost, g, G = evaluate(theta)
        if decrease <= tol or step_norm <= tol:
            converged = True
            break
    fitted = vehicle(theta)
    rmse = {}
    for part in ([[h] for h in hs] if carry else [hs]):
        se, cnt = eng.multistep_se_sweep(Xt, Ut, part, fitted[None], dt=dt, integrator=integrator, lag_mode=lag_mode)
        se = se.cpu().numpy()[0]
        for j, h in enumerate(part):
            rmse[h] = float(np.sqrt(se[j] / (cnt[j] * eng.nx))) if cnt[j] > 0 else float("nan")
    return CalibrationResult(phys=fitted, names=[PHYS_NAMES[i] for i in idx], theta=theta.copy(), rmse=rmse, gn=G,
                             cost=cost, cost0=cost0, iterations=it, converged=converged, history=history)


def one_step_rmse_physics(X_test: np.ndarray, U_test: np.ndarray, dt: float, model: str = None, dtype: str = "f64",
                          engine: Engine = None, lag_mode: str = "carry") -> float:
    """Teacher-forced one-step Euler prediction RMSE, rmse(X[1:], X[:-1] + dt f(X[:-1], U[:-1])); with
    lag_mode="carry" the thruster lag runs on through the rows as in the reference's loop over one model object."""
    eng = _engine_for(X_test, model, dtype, engine)
    return eng.multistep_rmse(X_test, U_test, 1, dt=dt, integrator="euler", lag_mode=lag_mode)


def rmse(y_true: np.ndarray, y_pred: np.ndarray) -> float:
    return float(np.sqrt(np.mean((np.asarray(y_true) - np.asarray(y_pred)) ** 2)))


# ----------------------------------------------------------------------------------------------------------------------
# double-integrator comparison model (training/train_tank_brov2_rk4.py:438-547; Euler twins in
# train_tank_brov2_full_comparison.py:510-598, train_tank_brov2_wrench_comp.py:270-366; quaternion twin in
# train_tank_brov2_wrench_quat.py:301-397)
# ----------------------------------------------------------------------------------------------------------------------
def estimate_di_gains(X_train: np.ndarray, U_train: np.ndarray, dt: float, ridge: float = 1e-3):
    """Ridge least squares of the forward-difference body accelerations on the inputs -> (K_lin, K_ang), each
    [n_inputs, 3].  A 6x6 / 8x8 normal-equation solve: host work, as in the reference (the fit is not on the hot
    path).  Velocities are columns 6:12 of a 12-state series, 7:13 of a 13-state quaternion series."""
    X = np.asarray(X_train, dtype=float)
    U = np.asarray(U_train, dtype=float)
    o = 7 if X.shape[1] == 13 else 6
    acc = (X[1:, o:o + 6] - X[:-1, o:o + 6]) / max(dt, 1e-9)
    G = U[:-1]
    K = np.linalg.solve(G.T @ G + ridge * np.eye(G.shape[1]), G.T @ acc)
    return K[:, :3].copy(), K[:, 3:].copy()


def _di_engine(n_states: int, n_inputs: int, K_lin, K_ang, dtype: str = "f64") -> Engine:
    if n_states == 13:
        if n_inputs != 6:
            raise ValueError("the quaternion double integrator takes 6 wrench inputs")
        model = "diq13_u6"
    elif n_states == 12 and n_inputs in (6, 8):
        model = "di12_u8" if n_inputs == 8 else "di12_u6"
    else:
        raise ValueError(f"no double-integrator model with {n_states} states and {n_inputs} inputs")
    eng = Engine(model, dtype)
    eng.set_di_gains(K_lin, K_ang)
    return eng


def simulate_double_integrator(x0: np.ndarray, U_seq: np.ndarray, dt: float, K_lin: np.ndarray, K_ang: np.ndarray,
                               integrator: str = "rk4") -> np.ndarray:
    """Rollout of the double-integrator model; returns [len(U_seq)+1, n_states] with row 0 = x0.  The reference
    integrates it with RK4 in train_tank_brov2_rk4.py and explicit Euler elsewhere (the quaternion variant: Euler
    only, quaternion normalised before and after every step)."""
    x0 = np.asarray(x0, dtype=float)
    U_seq = np.asarray(U_seq, dtype=float)
    H = len(U_seq)
    traj = np.zeros((H + 1, x0.shape[0]))
    traj[0] = x0
    if H == 0:
        return traj
    eng = _di_engine(x0.shape[0], U_seq.shape[1], K_lin, K_ang)
    res = eng.rollout(x0.reshape(1, -1), U_seq, dt=dt, integrator=integrator, stride=1, u_layout="shared")
    traj[1:] = res.traj[:, 0, :].cpu().numpy()
    return traj


def multistep_rmse_endpoint_di(X_test: np.ndarray, U_test: np.ndarray, H, dt: float, K_lin: np.ndarray,
                               K_ang: np.ndarray, integrator: str = "rk4", dtype: str = "f64"):
    """Endpoint RMSE of the double-integrator model over all sliding windows (NaN if T <= H); `H` may be a list."""
    X_test = np.asarray(X_test, dtype=float)
    eng = _di_engine(X_test.shape[1], np.shape(U_test)[1], K_lin, K_ang, dtype)
    return eng.multistep_rmse(X_test, U_test, H, dt=dt, integrator=integrator)
