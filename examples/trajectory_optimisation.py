"""Trajectory optimisation by shooting, with exact gradients from the adjoint rollout (Engine.rollout_diff).

4096 thruster-model vehicles (fp64, RK4, dt = 0.02 s) start from the hover trim of station_keeping_lqr.py at 1 m depth,
perturbed by up to +-1 m in position, +-0.2 rad in roll and pitch and +-pi/2 in yaw.  Each vehicle optimises its own
200-step (4 s) thrust plan u = 0.9 tanh(W) to come to rest at the trim pose.  The loss is a weighted terminal pose and
velocity error (angles wrapped to one turn) plus a small effort term.  One Adam optimiser runs over every vehicle's plan
at once; every gradient is one forward rollout and one adjoint launch.

Prints the initial and final losses, the fraction of vehicles that end within 5 cm and 3 degrees of the goal and at rest,
the seconds per gradient, and one vehicle's gradient against central differences at the initial plan.

    python examples/trajectory_optimisation.py [--vehicles 4096] [--iters 300]
"""
import argparse
import math
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bluerov2_dynamics_b200 as B                      # noqa: E402
from station_keeping_lqr import trim                    # noqa: E402

DT = 0.02
STEPS = 200
NX, NZ, NU = 12, 30, 8
W_POS, W_ANG, W_VEL, W_EFF = 10.0, 10.0, 1.0, 1e-3


def loss_fn(xT, U, goal):
    """per-vehicle loss [N]: terminal pose (wrapped angles) and velocity error, plus the mean squared input"""
    dp = xT[:, :3] - goal[:3]
    da = torch.atan2(torch.sin(xT[:, 3:6] - goal[3:6]), torch.cos(xT[:, 3:6] - goal[3:6]))
    return (W_POS * (dp ** 2).sum(1) + W_ANG * (da ** 2).sum(1) + W_VEL * (xT[:, 6:] ** 2).sum(1)
            + W_EFF * (U ** 2).mean(dim=(0, 2)))


def run(vehicles=4096, iters=300, lr=0.05, seed=0, verbose=True):
    e = B.Engine("thruster8", "f64")
    zs, us, _, _ = trim(e)
    rng = np.random.default_rng(seed)
    n = vehicles
    x0 = np.repeat(zs[None, :NX], n, axis=0)
    x0[:, :3] += rng.uniform(-1.0, 1.0, (n, 3))
    x0[:, 3:5] += rng.uniform(-0.2, 0.2, (n, 2))
    x0[:, 5] += rng.uniform(-math.pi / 2, math.pi / 2, n)
    x0 = e.tensor(x0)
    lag0 = e.tensor(np.repeat(zs[None, NX:], n, axis=0))
    goal = e.tensor(zs[:NX])
    W = torch.atanh(e.tensor(np.clip(us / 0.9, -0.99, 0.99)))[None, None].expand(STEPS, n, NU).clone()
    W.requires_grad_(True)

    def total_loss(Wv):
        U = 0.9 * torch.tanh(Wv)
        _, xT, _ = e.rollout_diff(x0, U, lag0=lag0, dt=DT, integrator="rk4", stride=0)
        return loss_fn(xT, U, goal)

    # one vehicle's gradient against central differences of the rollout at the initial plan
    lv = total_loss(W)
    g = torch.autograd.grad(lv.sum(), W)[0]
    d = torch.zeros_like(W)
    d[:, 0] = e.tensor(rng.standard_normal((STEPS, NU)))
    h = 1e-6
    with torch.no_grad():
        fd = float((total_loss(W + h * d)[0] - total_loss(W - h * d)[0]) / (2 * h))
    ad = float((g * d).sum())
    fd_rel = abs(ad - fd) / max(abs(fd), 1e-300)

    opt = torch.optim.Adam([W], lr=lr)
    loss0 = float(lv.detach().mean())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        opt.zero_grad(set_to_none=True)
        lv = total_loss(W)
        lv.sum().backward()
        opt.step()
    torch.cuda.synchronize()
    elapsed = time.perf_counter() - t0
    with torch.no_grad():
        U = 0.9 * torch.tanh(W)
        r = e.rollout(x0, U, dt=DT, lag0=lag0, lag_repr="projected")
        lv = loss_fn(r.xT, U, goal)
        pos_err = (r.xT[:, :3] - goal[:3]).norm(dim=1)
        ang_err = torch.atan2(torch.sin(r.xT[:, 3:6] - goal[3:6]), torch.cos(r.xT[:, 3:6] - goal[3:6])).abs().amax(1)
        speed = r.xT[:, 6:].abs().amax(1)
        ok = (pos_err < 0.05) & (ang_err < math.radians(3.0)) & (speed < 0.05)
    out = dict(vehicles=n, steps=STEPS, iters=iters, loss_initial_mean=loss0, loss_final_mean=float(lv.mean()),
               loss_final_median=float(lv.median()), within_5cm_3deg_at_rest=float(ok.double().mean()),
               median_position_error_m=float(pos_err.median()), median_angle_error_deg=math.degrees(float(ang_err.median())),
               seconds_per_gradient=elapsed / iters, seconds_total=elapsed,
               gradient_check=dict(adjoint=ad, central_difference=fd, relative_error=fd_rel))
    if verbose:
        print(f"{n} vehicles x {STEPS} steps (thruster8 fp64 RK4, dt {DT}), Adam lr {lr}, {iters} iterations")
        print(f"gradient check (vehicle 0, random direction): adjoint {ad:.12e}  central difference {fd:.12e}  "
              f"relative error {fd_rel:.2e}")
        print(f"mean loss: initial {loss0:.4e}  final {out['loss_final_mean']:.4e}  (final median {out['loss_final_median']:.4e})")
        print(f"within 5 cm / 3 deg of the goal and at rest (|nu| < 0.05): {100 * out['within_5cm_3deg_at_rest']:.1f} %  "
              f"(median errors {out['median_position_error_m'] * 100:.2f} cm, {out['median_angle_error_deg']:.2f} deg)")
        print(f"{out['seconds_per_gradient'] * 1e3:.2f} ms per gradient (forward rollout + adjoint + Adam step), "
              f"{elapsed:.2f} s in total")
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--vehicles", type=int, default=4096)
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--lr", type=float, default=0.05)
    a = ap.parse_args()
    run(a.vehicles, a.iters, a.lr)
