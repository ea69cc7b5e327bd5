"""Station keeping by LQR on the exact step Jacobians of the thruster model.

1. Hover trim at 1 m depth.  The vehicle is about 1 N heavy (W = 132.57 N, B = 131.588 N), so the vertical thrusters
   must hold it.  (z*, u*) solves Phi(z, u) = z for the one-step map of the 30-state thruster model (12 rigid-body
   states + the 18 allocation-projected lag states), found by minimum-norm Newton steps on [A - I | B] with A, B from
   Engine.linearize.
2. Discrete LQR on the linearisation at the trim (scipy.linalg.solve_discrete_are).
3. Closed-loop Monte-Carlo: 4096 vehicles start from the trim perturbed by up to +-0.5 m in position, +-0.3 rad in
   roll / pitch / yaw and +-0.2 m/s (rad/s) in the body rates, and run under u = clip(u* - K (z - z*), -1, 1) with the
   feedback evaluated inside the kernel (Engine.closed_loop, chunks of 100 steps, z after every step for the band).
4. Robustness: the same LQR on 4096 vehicles whose added masses and linear / quadratic damping are each off by up to
   +-20 % (a per-vehicle coefficient table, Engine.set_vehicle_physical).
5. Prints the trim residual, the fraction of vehicles that settle and their settling times.

    python examples/station_keeping_lqr.py [--vehicles 4096] [--seconds 30]
"""
import argparse
import os
import sys
import time

import numpy as np
import scipy.linalg
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bluerov2_dynamics_b200 as B                      # noqa: E402

DT = 0.02
DEPTH = 1.0
NX, NZ, NU = 12, 30, 8


def trim(e, iters=20, tol=1e-13):
    """Minimum-norm Newton on r(z, u) = Phi(z, u) - z from the vehicle at rest at DEPTH with zero input."""
    z = np.zeros(NZ)
    z[2] = DEPTH
    u = np.zeros(NU)
    res = np.inf
    for it in range(iters):
        r = e.linearize(z[None, :NX], u[None], dt=DT, lag0=z[None, NX:], lag_repr="projected", want_traj=False)
        F = r.z[0].cpu().numpy() - z
        res = np.linalg.norm(F)
        if res < tol:
            break
        M = np.concatenate([r.A[0, 0].cpu().numpy() - np.eye(NZ), r.B[0, 0].cpu().numpy()], axis=1)
        step = np.linalg.lstsq(M, -F, rcond=None)[0]
        z += step[:NZ]
        u += step[NZ:]
    return z, u, res, it


def lag_steady(u, steps=2000):
    """per-thruster lag state [8, 3] under the held input u: the engine advances it to its fixed point"""
    e = B.Engine("thruster8", "f64")
    r = e.rollout(np.zeros((1, NX)), (np.asarray(u)[None], steps), dt=DT, u_layout="const")
    return r.lag[0].reshape(8, 3)


def settle(e, x, lag24, zs, us, K, steps, chunk=100):
    """closed loop from (x, per-thruster lag) under u = clip(u* - K (z - z*), -1, 1) in chunks of `chunk` steps;
    returns (settling times [s] of the vehicles that settle, settled mask)"""
    n = x.shape[0]
    inside = torch.zeros((steps, n), dtype=torch.bool, device=e.device)
    lag, repr_ = lag24, "thruster"
    zs_t = torch.as_tensor(zs, device=e.device)
    for k0 in range(0, steps, chunk):
        m = min(chunk, steps - k0)
        r = e.closed_loop(x, K, zs, us, steps=m, dt=DT, lag0=lag, lag_repr=repr_, stride=1)
        x, lag, repr_ = r.z[:, :NX], r.z[:, NX:], "projected"
        err = (r.z_traj[:, :, :NX] - zs_t[:NX]).abs()
        err[:, :, 3:6] = torch.remainder(err[:, :, 3:6] + np.pi, 2 * np.pi) - np.pi      # angle error on (-pi, pi]
        err = err.abs()
        inside[k0:k0 + m] = (err[..., :3].amax(2) < 0.02) & (err[..., 3:6].amax(2) < 0.02) & (err[..., 6:].amax(2) < 0.02)
    # settled: inside the band from some step to the end; settling time = first such step
    stay = torch.flip(torch.cumprod(torch.flip(inside, [0]).to(torch.int32), 0), [0]).bool()
    settled = stay[-1]
    first = torch.where(stay.any(0), stay.to(torch.int8).argmax(0), steps)
    return (first[settled].double() + 1).cpu().numpy() * DT, settled


def run(vehicles=4096, seconds=30.0, seed=0, verbose=True):
    e = B.Engine("thruster8", "f64")
    t0 = time.perf_counter()
    zs, us, res, iters = trim(e)
    r = e.linearize(zs[None, :NX], us[None], dt=DT, lag0=zs[None, NX:], lag_repr="projected", want_traj=False)
    A, Bm = r.A[0, 0].cpu().numpy(), r.B[0, 0].cpu().numpy()
    resid = float(np.linalg.norm(r.z[0].cpu().numpy() - zs))
    # weights: pose and body rates; the lag states are stable and left almost free
    Q = np.diag([10, 10, 10, 5, 5, 5] + [1] * 6 + [1e-6] * 18)
    R = 0.5 * np.eye(NU)
    P = scipy.linalg.solve_discrete_are(A, Bm, Q, R)
    K = np.linalg.solve(R + Bm.T @ P @ Bm, Bm.T @ P @ A)
    rho = float(np.max(np.abs(np.linalg.eigvals(A - Bm @ K))))

    rng = np.random.default_rng(seed)
    n = vehicles
    x = np.tile(zs[:NX], (n, 1))
    x[:, 0:3] += rng.uniform(-0.5, 0.5, (n, 3))
    x[:, 3:6] += rng.uniform(-0.3, 0.3, (n, 3))
    x[:, 6:12] += rng.uniform(-0.2, 0.2, (n, 6))
    steps = int(round(seconds / DT))
    lag = lag_steady(us).reshape(1, 24).repeat(n, 1)
    ts, settled = settle(e, x, lag, zs, us, K, steps)
    # robustness: every vehicle's added masses and damping off by up to +-20 %
    table = np.tile(e.phys, (n, 1))
    for grp in ("added", "lin", "quad"):
        idx = B.engine.PARAM_GROUPS[grp]
        table[:, idx] *= rng.uniform(0.8, 1.2, (n, len(idx)))
    table = B.with_minv(table)
    e.set_vehicle_physical(table)
    ts_pv, settled_pv = settle(e, x, lag, zs, us, K, steps)
    e.set_vehicle_physical(None)
    wall = time.perf_counter() - t0
    out = dict(trim_residual=resid, newton_iters=iters + 1, newton_residual=float(res), u_trim=us.tolist(),
               closed_loop_spectral_radius=rho, vehicles=n, seconds=seconds,
               settled_fraction=float(settled.float().mean()),
               settling_time_s={"median": float(np.median(ts)), "p95": float(np.percentile(ts, 95)),
                                "max": float(ts.max())} if ts.size else None,
               perturbed_settled_fraction=float(settled_pv.float().mean()),
               perturbed_settling_time_median_s=float(np.median(ts_pv)) if ts_pv.size else None,
               wall_s=wall)
    if verbose:
        print(f"trim at {DEPTH} m depth: {out['newton_iters']} Newton steps, residual |Phi(z*,u*) - z*| = {resid:.3e}")
        print("  u* =", np.array2string(us, precision=4))
        print(f"LQR: closed-loop spectral radius {rho:.6f}")
        print(f"closed loop, {n} vehicles, {seconds:g} s: {100 * out['settled_fraction']:.2f} % settle "
              "(|pos| < 2 cm, |angle| < 0.02 rad, |rates| < 0.02 until the end)")
        if ts.size:
            s = out["settling_time_s"]
            print(f"  settling time median {s['median']:.2f} s, p95 {s['p95']:.2f} s, max {s['max']:.2f} s")
        print(f"same LQR, {n} vehicles with added masses and damping each off by up to +-20 %: "
              f"{100 * out['perturbed_settled_fraction']:.2f} % settle"
              + (f", median {out['perturbed_settling_time_median_s']:.2f} s" if ts_pv.size else ""))
        print(f"  wall time {wall:.2f} s")
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--vehicles", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=30.0)
    a = ap.parse_args()
    run(a.vehicles, a.seconds)
