"""Calibration by sweep: which vehicle produced this tank recording?

A series as long as the reference's tank recording (45,823 rows at 50 Hz) is simulated with a "true" BlueROV2 whose
linear / quadratic damping and added masses differ from the defaults, plus measurement noise.  A few hundred candidate
vehicles around the defaults (the truth among them) are scored by the reference's endpoint RMSE at H = 1 / 10 / 100 in
one Engine.multistep_rmse_sweep call per lag mode, and the time is compared with the serial loop
`set_physical + multistep_rmse` per candidate that a user would otherwise write.

    python examples/parameter_sweep.py [--candidates 300] [--rows 45823] [--lag-mode carry|reset]
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bluerov2_dynamics_b200 as B                      # noqa: E402
from bluerov2_dynamics_b200 import _lib as L            # noqa: E402

DT, HS = 0.02, [1, 10, 100]


def scaled(scales):
    """physical table of vehicles whose added mass, linear and quadratic damping are the defaults times `scales`
    [P, 3]; diag(Minv) rebuilt from the new masses as the reference's __init__ does"""
    ph = np.tile(B.default_physical(), (len(scales), 1))
    ph[:, L.PH_ADDED:L.PH_ADDED + 6] *= scales[:, 0:1]
    ph[:, L.PH_LIN:L.PH_LIN + 6] *= scales[:, 1:2]
    ph[:, L.PH_QUAD:L.PH_QUAD + 6] *= scales[:, 2:3]
    return B.with_minv(ph)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--candidates", type=int, default=300)
    ap.add_argument("--rows", type=int, default=45823)
    ap.add_argument("--lag-mode", default="carry", choices=["carry", "reset"])
    a = ap.parse_args()
    rng = np.random.default_rng(1)

    true_scales = np.array([[1.15, 0.85, 1.2]])
    truth = scaled(true_scales)[0]
    sim = B.Engine("thruster8", "f64")
    sim.set_physical(truth)
    U = np.clip(np.cumsum(rng.normal(0, 0.02, (a.rows, 8)), axis=0) * 0.3, -0.6, 0.6)   # smooth thruster commands
    x0 = np.zeros((1, 12))
    r = sim.rollout(x0, U[:-1], dt=DT, integrator="rk4", stride=1, u_layout="shared")
    X = np.concatenate([x0, r.traj[:, 0, :].cpu().numpy()])
    X += rng.normal(0, 1e-3, X.shape)                                                     # measurement noise

    scales = np.concatenate([rng.uniform(0.7, 1.3, (a.candidates - 1, 3)), true_scales])
    scales = scales[rng.permutation(len(scales))]
    ph = scaled(scales)
    e = B.Engine("thruster8", "f64")
    Xt, Ut = e.tensor(X), e.tensor(U)
    e.multistep_rmse_sweep(Xt, Ut, HS, ph[:2], dt=DT, lag_mode=a.lag_mode)                # warm-up
    t0 = time.perf_counter()
    rmse = e.multistep_rmse_sweep(Xt, Ut, HS, ph, dt=DT, lag_mode=a.lag_mode)             # [P, 3], synchronises
    t_sweep = time.perf_counter() - t0

    n_serial = min(len(ph), 32)
    t0 = time.perf_counter()
    for c in range(n_serial):
        e.set_physical(ph[c])
        e.multistep_rmse(Xt, Ut, HS, dt=DT, lag_mode=a.lag_mode)
    t_serial = (time.perf_counter() - t0) * len(ph) / n_serial

    print(f"{len(ph)} candidates x {a.rows} rows, H = {HS}, lag_mode = {a.lag_mode}")
    order = np.argsort(rmse[:, 1])
    print("best candidates by RMSE at H = 10 (scales of added mass, linear damping, quadratic damping):")
    for i in order[:5]:
        tag = "  <- truth" if np.allclose(scales[i], true_scales[0]) else ""
        print(f"  {scales[i].round(3)}  rmse H=1 {rmse[i, 0]:.3e}  H=10 {rmse[i, 1]:.3e}  H=100 {rmse[i, 2]:.3e}{tag}")
    print(f"sweep {t_sweep * 1e3:.1f} ms; serial loop of set_physical + multistep_rmse {t_serial * 1e3:.1f} ms "
          f"(timed over {n_serial} candidates, scaled); speed-up {t_serial / t_sweep:.1f}x")


if __name__ == "__main__":
    main()
