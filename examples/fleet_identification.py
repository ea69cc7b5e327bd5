"""Fleet identification by multiple shooting, with exact coefficient gradients from the adjoint rollout
(Engine.rollout_diff(kp=...), derive_params_torch).

256 thruster-model vehicles (fp64, RK4, dt = 0.02 s) each have their own "true" 6 added masses, 6 linear and 6
quadratic damping terms, drawn within +-30 % of the defaults as in examples/calibrate.py.  Each vehicle has its own
simulated 20 s recording under smooth random thrust commands, with 1e-3 noise on every recorded state, cut into 50-step
segments.  Every segment starts from the recorded state (and the recorded thruster lag) and is scored on its full
trajectory.  All vehicles are fitted in one batched optimisation: one Adam optimiser over every vehicle's 18 log-scale
factors of the defaults, the segments of a vehicle sharing its coefficient table column; every gradient is one forward
rollout and one adjoint launch over all 256 x 20 segments.

Prints the loss before and after for the fleet (and how many vehicles reduced theirs), the median and 95th-percentile
relative coefficient error per group, and one vehicle's gradient against central differences.

    python examples/fleet_identification.py [--vehicles 256] [--iters 300]
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bluerov2_dynamics_b200 as B                      # noqa: E402
from bluerov2_dynamics_b200 import _lib as L           # noqa: E402

DT = 0.02
SEG = 50
SECONDS = 20.0
NOISE = 1e-3
GROUPS = {"added": L.PH_ADDED, "lin": L.PH_LIN, "quad": L.PH_QUAD}
IDX = [i for c in GROUPS.values() for i in range(c, c + 6)]


def record(e, ph_true, rng):
    """per-vehicle recordings: X [T+1, n, 12] (noisy), lag [S, n, 18] at segment starts, U [T, n, 8]"""
    n = ph_true.shape[0]
    T = int(round(SECONDS / DT))
    ar = np.zeros((n, 8))
    U = np.empty((T, n, 8))
    for k in range(T):                                   # smooth thrust commands, AR(1)
        ar = np.clip(0.98 * ar + 0.04 * rng.standard_normal((n, 8)), -1, 1)
        U[k] = 0.5 * ar
    x = np.zeros((n, 12))
    x[:, 2] = 1.0 + rng.uniform(-0.5, 0.5, n)
    x[:, 5] = rng.uniform(-3, 3, n)
    e.set_vehicle_physical(ph_true)
    Xs, lags = [x], []
    lag = torch.zeros((n, 18), dtype=torch.float64, device=e.device)
    for s in range(T // SEG):
        lags.append(lag)
        r = e.rollout(Xs[-1], U[s * SEG:(s + 1) * SEG], dt=DT, stride=1, lag0=lag, lag_repr="projected", want_lag=True)
        Xs.extend(list(r.traj.cpu().numpy()))
        lag = r.lag
    e.set_vehicle_physical(None)
    X = np.stack(Xs) + NOISE * rng.standard_normal((T + 1, n, 12))
    return X, torch.stack(lags), U


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vehicles", type=int, default=256)
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--lr", type=float, default=0.02)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    rng = np.random.default_rng(a.seed)
    e = B.Engine("thruster8", "f64")
    dev = e.device
    n = a.vehicles
    ph0 = B.default_physical()
    ph_true = np.tile(ph0, (n, 1))
    ph_true[:, IDX] *= rng.uniform(0.7, 1.3, (n, len(IDX)))
    ph_true = B.with_minv(ph_true)
    X, lags, U = record(e, ph_true, rng)
    S = (X.shape[0] - 1) // SEG
    # segment j = s * n + i: vehicle i, steps s*SEG .. (s+1)*SEG
    x0 = torch.from_numpy(X[0:S * SEG:SEG].reshape(S * n, 12)).to(dev)
    lag0 = lags.reshape(S * n, 18)
    Useg = torch.from_numpy(U.reshape(S, SEG, n, 8).transpose(1, 0, 2, 3).reshape(SEG, S * n, 8).copy()).to(dev)
    Xseg = torch.from_numpy(X[1:].reshape(S, SEG, n, 12).transpose(1, 0, 2, 3).reshape(SEG, S * n, 12).copy()).to(dev)
    owner = torch.arange(n, device=dev).repeat(S)
    base = torch.from_numpy(ph0).to(dev)
    idx = torch.tensor(IDX, device=dev)

    def phys_of(logf):
        ph = base.repeat(n, 1)
        return ph.index_copy(1, idx, ph[:, idx] * torch.exp(logf))

    def vehicle_loss(logf):
        kp = B.derive_params_torch(phys_of(logf))[owner]                    # [S n, NKP]: one column per vehicle
        traj, _, _ = e.rollout_diff(x0, Useg, lag0=lag0, dt=DT, stride=1, kp=kp)
        seg = ((traj - Xseg) ** 2).mean(dim=(0, 2))                          # [S n]
        return torch.zeros(n, dtype=torch.float64, device=dev).index_add(0, owner, seg) / S

    logf = torch.zeros((n, len(IDX)), dtype=torch.float64, device=dev, requires_grad=True)
    with torch.no_grad():
        l0 = vehicle_loss(logf)
    # one vehicle's gradient against central differences at the start
    lv = vehicle_loss(logf)
    g = torch.autograd.grad(lv[0], logf)[0][0].cpu().numpy()
    fd = np.zeros(len(IDX))
    h = 1e-6
    with torch.no_grad():
        for j in range(len(IDX)):
            v = []
            for sgn in (1, -1):
                p = logf.detach().clone()
                p[0, j] += sgn * h
                v.append(float(vehicle_loss(p)[0]))
            fd[j] = (v[0] - v[1]) / (2 * h)
    gerr = float(np.abs(g - fd).max() / np.abs(fd).max())
    opt = torch.optim.Adam([logf], lr=a.lr)
    torch.cuda.synchronize()
    t0 = time.time()
    for _ in range(a.iters):
        opt.zero_grad()
        vehicle_loss(logf).sum().backward()
        opt.step()
    torch.cuda.synchronize()
    t1 = time.time()
    with torch.no_grad():
        l1 = vehicle_loss(logf)
        fit = phys_of(logf).cpu().numpy()
    print(f"fleet identification: {n} thruster8 vehicles, {S} segments of {SEG} steps each ({SECONDS:g} s at dt = {DT}),"
          f" noise {NOISE:g}, {a.iters} Adam iterations in {t1 - t0:.1f} s ({1e3 * (t1 - t0) / a.iters:.1f} ms per gradient)")
    print(f"mean segment loss per vehicle: {float(l0.mean()):.4e} -> {float(l1.mean()):.4e};"
          f" {int((l1 < l0).sum())} of {n} vehicles reduced their loss;"
          f" noise floor (the loss at the true coefficients is about the noise variance) {NOISE ** 2:.1e}")
    for name, c in GROUPS.items():
        # the default linear damping has zero entries (Y_v, K_p, N_r): a scale factor keeps them at zero, so the
        # relative error is taken over the nonzero coefficients
        nz = ph0[c:c + 6] != 0.0
        true = ph_true[:, c:c + 6][:, nz]
        rel = np.abs(fit[:, c:c + 6][:, nz] - true) / np.abs(true)
        start = np.abs(ph0[c:c + 6][nz] - true) / np.abs(true)
        print(f"  {name:5s} relative coefficient error over its {int(nz.sum())} nonzero coefficients: median"
              f" {np.median(rel):.3e}, 95th percentile {np.percentile(rel, 95):.3e} (at the defaults: median"
              f" {np.median(start):.3e})")
    print(f"vehicle 0 gradient against central differences (h = {h:g} in the log factors): normwise relative"
          f" error {gerr:.2e}")


if __name__ == "__main__":
    main()
