"""Calibration by gradient: fit all 18 hydrodynamic coefficients of a BlueROV2 to a tank-length recording.

A series as long as the reference's tank recording (45,823 rows at 50 Hz) is simulated with a "true" vehicle whose 6
added masses, 6 linear and 6 quadratic damping terms each differ from the defaults by up to 30 %, plus 1e-3
measurement noise.  evaluators.calibrate_physical fits all 18 from the defaults by Levenberg-Marquardt on the
reference's endpoint error at H = 1 / 10 / 100 (carried thruster lag): every iteration is one exact gradient +
Gauss-Newton call (Engine.multistep_se_grad) and one sweep call that scores the trial steps.  For comparison, the
best of a 300-candidate random sweep (examples/parameter_sweep.py's approach, all 18 coefficients drawn) is shown.

    python examples/calibrate.py [--rows 45823] [--candidates 300]
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bluerov2_dynamics_b200 as B                      # noqa: E402
from bluerov2_dynamics_b200 import _lib as L            # noqa: E402
from bluerov2_dynamics_b200.evaluators import calibrate_physical   # noqa: E402

DT, HS = 0.02, [1, 10, 100]
PARAMS = ["added", "lin", "quad"]


def perturbed(rng, n):
    """n physical vectors with the 18 coefficients scaled by U(0.7, 1.3); diag(Minv) rebuilt"""
    ph = np.tile(B.default_physical(), (n, 1))
    for col in (L.PH_ADDED, L.PH_LIN, L.PH_QUAD):
        ph[:, col:col + 6] *= rng.uniform(0.7, 1.3, (n, 6))
    return B.with_minv(ph)


def run(rows=45823, candidates=300, verbose=True):
    rng = np.random.default_rng(1)
    truth = perturbed(rng, 1)[0]
    sim = B.Engine("thruster8", "f64")
    sim.set_physical(truth)
    # the reference's smooth random command signal u <- clip(0.98 u + 0.02 N(0,1), -1, 1), at half scale: the vehicle
    # stays away from theta = +-pi/2, where the Euler-angle kinematics (and the sensitivities) blow up
    U = np.zeros((rows, 8))
    s = np.zeros(8)
    for k in range(rows):
        s = np.clip(0.98 * s + 0.02 * rng.standard_normal(8), -1.0, 1.0)
        U[k] = 0.5 * s
    x0 = np.zeros((1, 12))
    r = sim.rollout(x0, U[:-1], dt=DT, integrator="rk4", stride=1, u_layout="shared")
    X = np.concatenate([x0, r.traj[:, 0, :].cpu().numpy()])
    X += rng.normal(0, 1e-3, X.shape)                                                 # measurement noise

    e = B.Engine("thruster8", "f64")
    Xt, Ut = e.tensor(X), e.tensor(U)
    calibrate_physical(Xt[:2000], Ut[:2000], DT, B.default_physical(), PARAMS, engine=e, max_iter=1)   # warm-up
    t0 = time.perf_counter()
    res = calibrate_physical(Xt, Ut, DT, B.default_physical(), PARAMS, horizons=HS, engine=e)
    t_fit = time.perf_counter() - t0
    t0 = time.perf_counter()
    table = perturbed(rng, candidates)
    sweep = e.multistep_rmse_sweep(Xt, Ut, HS, table, dt=DT, lag_mode="carry")
    t_sweep = time.perf_counter() - t0
    best = int(np.argmin(sweep[:, 1]))
    at_truth = e.multistep_rmse_sweep(Xt, Ut, HS, truth[None], dt=DT, lag_mode="carry")[0]
    idx = B.parameter_indices(PARAMS)
    scale = np.where(truth[idx] != 0.0, np.abs(truth[idx]), 1.0)
    out = dict(rows=rows, iterations=res.iterations, converged=res.converged, cost0=res.cost0, cost=res.cost,
               fit_s=t_fit, sweep_s=t_sweep, rmse_fit=[res.rmse[h] for h in HS], rmse_truth=list(at_truth),
               rmse_best_sweep=list(sweep[best]), rel_err=dict(zip(res.names, ((res.theta - truth[idx]) / scale).tolist())))
    if verbose:
        print(f"{rows} rows, 18 coefficients fitted from the defaults: {res.iterations} iterations "
              f"({'converged' if res.converged else 'not converged'}), cost {res.cost0:.4e} -> {res.cost:.4e}, "
              f"{t_fit:.2f} s")
        print("coefficient      truth        fitted      default     error (relative to |truth|)")
        d0 = B.default_physical()
        for j, i in enumerate(idx):
            print(f"  {res.names[j]:<8} {truth[i]:12.5g} {res.theta[j]:12.5g} {d0[i]:12.5g}   {out['rel_err'][res.names[j]]:+.2e}")
        print("endpoint RMSE        H=1         H=10        H=100")
        for name, v in (("fit", out["rmse_fit"]), ("truth", out["rmse_truth"]),
                        (f"best of {candidates}", out["rmse_best_sweep"])):
            print(f"  {name:<16} " + "  ".join(f"{x:.5e}" for x in v))
        print(f"sweep of {candidates} random candidates: {t_sweep:.2f} s")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=45823)
    ap.add_argument("--candidates", type=int, default=300)
    a = ap.parse_args()
    run(a.rows, a.candidates)


if __name__ == "__main__":
    main()
