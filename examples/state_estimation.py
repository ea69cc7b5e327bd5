"""State estimation with extended Kalman filters on the thruster model, and noise tuning by likelihood in one launch.

1. A "real" vehicle: the default coefficients with the linear and quadratic damping 15 % larger.  It runs under the
   reference's smooth random thruster commands (datasets.smooth_random_inputs) with generate_sim_dataset's Euler step
   and its sensor noise (0.5 mm, 1 mrad, 0.5 mm/s, 1 mrad/s standard deviations).  A BlueROV2-like sensor suite
   measures depth, attitude and the gyro rates at every step and the DVL body velocities u, v, w at every 10th step;
   nothing measures x and y.
2. Tuning: 64 filters on the DEFAULT model (so the model is wrong by the damping change), each with the process noise
   q = s * q0 for its own scale s on a log grid, in one Engine.ekf launch with shared inputs and measurements and
   per-filter q.  The scale with the highest log-likelihood is chosen.
3. Prints the RMSE against the truth per state group for the raw measurements, the filter at the chosen q and the
   filter at the smallest q (velocities also at the DVL steps alone), the x / y drift, and the time of the tuning
   launch.

    python examples/state_estimation.py [--steps 6000] [--filters 64]
"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bluerov2_dynamics_b200 as B                      # noqa: E402
from bluerov2_dynamics_b200 import _lib as L            # noqa: E402
from bluerov2_dynamics_b200.datasets import smooth_random_inputs  # noqa: E402

DT = 0.05
NOISE = np.repeat([0.0005, 0.001, 0.0005, 0.001], 3)     # generate_sim_dataset's per-group standard deviations
Q0 = np.repeat([1e-6, 1e-6, 1e-4, 1e-4], 3) * DT         # process-noise shape: mostly on the velocities and rates
GROUPS = {"depth z": [2], "attitude": [3, 4, 5], "velocity u v w": [6, 7, 8], "rates p q r": [9, 10, 11]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=6000)
    ap.add_argument("--filters", type=int, default=64)
    a = ap.parse_args()
    T, nf = a.steps, a.filters

    # 1. the real vehicle and its sensors
    real = B.Engine("thruster8", "f64")
    ph = B.default_physical()
    ph[L.PH_LIN:L.PH_LIN + 6] *= 1.15
    ph[L.PH_QUAD:L.PH_QUAD + 6] *= 1.15
    real.set_physical(ph)
    U, draws = smooth_random_inputs(T, seed=42)
    truth = real.rollout(np.zeros((1, 12)), U, dt=DT, integrator="euler", stride=1).traj[:, 0].cpu().numpy()
    meas = truth + draws * NOISE
    Y = meas.copy()
    Y[:, :2] = np.nan                                    # no position fix
    Y[np.arange(T) % 10 != 9, 6:9] = np.nan              # DVL at a tenth of the rate

    # 2. 64 candidate process-noise levels, one launch
    e = B.Engine("thruster8", "f64")
    scales = np.logspace(-4, 4, nf)
    q = scales[:, None] * Q0
    r = NOISE ** 2
    P0 = np.diag(np.full(12, 1e-4))
    x0 = np.zeros((nf, 12))
    Ut, Yt = e.tensor(U), e.tensor(Y)
    e.ekf(x0, P0, Ut, Yt, q, r, dt=DT, integrator="euler", stride=1)        # warm-up (module load)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    res = e.ekf(x0, P0, Ut, Yt, q, r, dt=DT, integrator="euler", stride=1)
    t1.record()
    torch.cuda.synchronize()
    ll = res.loglik.cpu().numpy()
    best = int(np.argmax(ll))
    xs = res.x_traj.cpu().numpy()                        # [T, nf, 12]
    print(f"{nf} filters x {T} steps, one Engine.ekf launch: {t0.elapsed_time(t1):.2f} ms; "
          f"{int(res.count[0])} scalar updates per filter")
    print(f"log-likelihood peaks at q = {scales[best]:.3g} q0 (grid {scales[0]:.0e} .. {scales[-1]:.0e}); "
          f"loglik {ll[best]:.1f} against {ll[0]:.1f} at the smallest q")

    # 3. errors against the truth
    def rmse(est, cols, ref=truth):                      # over the steps where est has a value
        d = est[:, cols] - ref[:, cols]
        if cols == [3, 4, 5]:
            d = d - 2 * np.pi * np.rint(d / (2 * np.pi))
        return float(np.sqrt(np.nanmean(d * d)))
    print(f"{'RMSE':<16}{'raw sensor':>14}{'filter, best q':>16}{'filter, min q':>16}")
    for name, cols in GROUPS.items():
        raw = rmse(Y, cols)
        print(f"{name:<16}{raw:>14.3e}{rmse(xs[:, best], cols):>16.3e}{rmse(xs[:, 0], cols):>16.3e}")
    dvl = np.arange(T) % 10 == 9
    vel = [6, 7, 8]
    print(f"{'  at DVL steps':<16}{rmse(Y[dvl], vel, truth[dvl]):>14.3e}{rmse(xs[dvl, best], vel, truth[dvl]):>16.3e}"
          f"{rmse(xs[dvl, 0], vel, truth[dvl]):>16.3e}")
    drift = np.hypot(*(xs[-1, best, :2] - truth[-1, :2]))
    print(f"x, y (not measured): RMSE {rmse(xs[:, best], [0, 1]):.3e} m at the best q, {rmse(xs[:, 0], [0, 1]):.3e} m "
          f"at the smallest; horizontal drift after {T * DT:.0f} s: {drift:.3f} m over a "
          f"{np.hypot(*(truth[-1, :2] - truth[0, :2])):.2f} m track")


if __name__ == "__main__":
    main()
