"""Robust gain tuning: one feedback gain fitted to a fleet of perturbed vehicles through the closed-loop adjoint.

1. The hover trim and LQR gain K0 of examples/station_keeping_lqr.py (same Q, R).
2. A training fleet of thruster8 vehicles whose added masses and linear and quadratic damping are each off by up to
   +-30 % (a per-vehicle coefficient table), started from the station-keeping example's perturbed initial states.
3. One shared gain K = K0 + dK (const_shared layout) fitted with Adam through Engine.closed_loop_diff: the loss is the
   mean closed-loop cost sum_k dz'Q dz + (u - u*)'R (u - u*) over 10 s; every gradient is one closed_loop call and one
   closed_loop_vjp call, the clamp and the feedback differentiated through.
4. For K0 and the tuned K: the mean cost on the training fleet and on a held-out fleet drawn with another seed, and the
   held-out settle fraction and median settling time over 30 s; the time per gradient.
5. One gK entry against a central difference of closed_loop's cost.

    python examples/robust_gain_tuning.py [--vehicles 8192] [--iters 100]
"""
import argparse
import os
import sys
import time

import numpy as np
import scipy.linalg
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bluerov2_dynamics_b200 as B                      # noqa: E402
from station_keeping_lqr import DT, NU, NX, lag_steady, settle, trim   # noqa: E402

Q = np.diag([10, 10, 10, 5, 5, 5] + [1] * 6 + [1e-6] * 18)
R = 0.5 * np.eye(NU)


def fleet(e, zs, us, n, seed):
    """initial states (as station_keeping_lqr), per-thruster lag at the trim, a +-30 % coefficient table"""
    rng = np.random.default_rng(seed)
    x = np.tile(zs[:NX], (n, 1))
    x[:, 0:3] += rng.uniform(-0.5, 0.5, (n, 3))
    x[:, 3:6] += rng.uniform(-0.3, 0.3, (n, 3))
    x[:, 6:12] += rng.uniform(-0.2, 0.2, (n, 6))
    table = np.tile(e.phys, (n, 1))
    for grp in ("added", "lin", "quad"):
        idx = B.engine.PARAM_GROUPS[grp]
        table[:, idx] *= rng.uniform(0.7, 1.3, (n, len(idx)))
    x = torch.as_tensor(x, device=e.device)
    lag = e.project_lag(lag_steady(us).reshape(1, 24).repeat(n, 1))
    return x, lag, B.with_minv(table)


def mean_cost(e, x, lag, table, K, zs, us, steps):
    e.set_vehicle_physical(table)
    try:
        return float(e.closed_loop(x, K, zs, us, steps=steps, dt=DT, lag0=lag, lag_repr="projected",
                                   cost_q=np.diag(Q), cost_r=np.diag(R)).cost.mean())
    finally:
        e.set_vehicle_physical(None)


def run(vehicles=8192, iters=100, seconds=10.0, eval_seconds=30.0, lr=2e-3, verbose=True):
    e = B.Engine("thruster8", "f64")
    zs, us, _, _ = trim(e)
    r = e.linearize(zs[None, :NX], us[None], dt=DT, lag0=zs[None, NX:], lag_repr="projected", want_traj=False)
    A, Bm = r.A[0, 0].cpu().numpy(), r.B[0, 0].cpu().numpy()
    P = scipy.linalg.solve_discrete_are(A, Bm, Q, R)
    K0 = np.linalg.solve(R + Bm.T @ P @ Bm, Bm.T @ P @ A)
    steps = int(round(seconds / DT))
    x, lag, table = fleet(e, zs, us, vehicles, 0)
    xh, lagh, tableh = fleet(e, zs, us, vehicles, 1)
    zs_t, us_t = torch.as_tensor(zs, device=e.device), torch.as_tensor(us, device=e.device)
    K0_t = torch.as_tensor(K0, device=e.device)
    dK = torch.zeros_like(K0_t, requires_grad=True)
    opt = torch.optim.Adam([dK], lr=lr)
    e.set_vehicle_physical(table)
    hist = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    try:
        for it in range(iters):
            opt.zero_grad()
            _, _, cost = e.closed_loop_diff(x, K0_t + dK, zs_t, us_t, lag0=lag, steps=steps, dt=DT,
                                            cost_q=np.diag(Q), cost_r=np.diag(R))
            loss = cost.mean()
            loss.backward()
            opt.step()
            hist.append(float(loss.detach()))
        torch.cuda.synchronize()
    finally:
        e.set_vehicle_physical(None)
    t_grad = (time.perf_counter() - t0) / iters
    K1 = (K0_t + dK.detach()).cpu().numpy()

    # one gK entry against a central difference of closed_loop's mean cost (256 training vehicles)
    m = 256
    e.set_vehicle_physical(table[:m])
    try:
        g = e.closed_loop_vjp(x[:m], K1, zs, us, gcost=torch.full((m,), 1.0 / m, device=e.device, dtype=torch.float64),
                              steps=steps, dt=DT, lag0=lag[:m], lag_repr="projected", cost_q=np.diag(Q),
                              cost_r=np.diag(R), want=("K",)).gK.cpu().numpy()
    finally:
        e.set_vehicle_physical(None)
    ri, rj = np.unravel_index(np.argmax(np.abs(g)), g.shape)
    h = 1e-6

    def f(s):
        Kp = K1.copy()
        Kp[ri, rj] += s
        return mean_cost(e, x[:m], lag[:m], table[:m], Kp, zs, us, steps)

    fd = (f(h) - f(-h)) / (2 * h)
    out = dict(vehicles=vehicles, iters=iters, seconds=seconds, lr=lr, ms_per_gradient=1e3 * t_grad,
               loss_first=hist[0], loss_last=hist[-1],
               train_cost={"K0": mean_cost(e, x, lag, table, K0, zs, us, steps),
                           "tuned": mean_cost(e, x, lag, table, K1, zs, us, steps)},
               heldout_cost={"K0": mean_cost(e, xh, lagh, tableh, K0, zs, us, steps),
                             "tuned": mean_cost(e, xh, lagh, tableh, K1, zs, us, steps)},
               gK_check={"entry": [int(ri), int(rj)], "adjoint": float(g[ri, rj]), "central_difference": float(fd),
                         "rel_err": float(abs(g[ri, rj] - fd) / abs(fd))})
    ev = int(round(eval_seconds / DT))
    lag24 = lag_steady(us).reshape(1, 24).repeat(vehicles, 1)
    e.set_vehicle_physical(tableh)
    try:
        for name, K in (("K0", K0), ("tuned", K1)):
            ts, settled = settle(e, xh, lag24, zs, us, K, ev)
            out[f"heldout_settle_{name}"] = {"fraction": float(settled.float().mean()),
                                             "median_s": float(np.median(ts)) if ts.size else None}
    finally:
        e.set_vehicle_physical(None)
    if verbose:
        print(f"{vehicles} thruster8 vehicles, added mass and damping each off by up to +-30 %, {seconds:g} s horizon")
        print(f"Adam, {iters} iterations: mean cost {hist[0]:.4f} -> {hist[-1]:.4f}, {out['ms_per_gradient']:.2f} ms "
              "per gradient (closed_loop + closed_loop_vjp)")
        for k in ("K0", "tuned"):
            s = out[f"heldout_settle_{k}"]
            print(f"  {k:5s}: mean cost train {out['train_cost'][k]:.4f}, held-out {out['heldout_cost'][k]:.4f}; "
                  f"held-out over {eval_seconds:g} s: {100 * s['fraction']:.2f} % settle, median "
                  + (f"{s['median_s']:.2f} s" if s["median_s"] is not None else "-"))
        c = out["gK_check"]
        print(f"gK[{ri}, {rj}] = {c['adjoint']:.9e}, central difference {c['central_difference']:.9e}, "
              f"relative error {c['rel_err']:.1e}")
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--vehicles", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=100)
    a = ap.parse_args()
    run(a.vehicles, a.iters)
