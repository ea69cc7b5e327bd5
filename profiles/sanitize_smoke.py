"""Small-size pass over every kernel of libbrov.so, meant to run under compute-sanitizer on a B200:

    python profiles/sanitize_smoke.py                      (plain: ragged-size pass over every kernel)
    compute-sanitizer --tool memcheck  python profiles/sanitize_smoke.py
    compute-sanitizer --tool racecheck python profiles/sanitize_smoke.py

Sizes are ragged on purpose (partial warps / blocks, odd snapshot counts, unaligned quaternion rows)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bluerov2_dynamics_b200 as B  # noqa: E402
from bluerov2_dynamics_b200 import pinc as P  # noqa: E402
from bluerov2_dynamics_b200.Koopman.koopmanEDMDc import KoopmanEDMDc  # noqa: E402

rng = np.random.default_rng(0)
dt = 0.02
for dtype in ("f64", "f32"):
    for model, nx, nu in (("thruster8", 12, 8), ("wrench12", 12, 6), ("quat13", 13, 6), ("di12_u8", 12, 8),
                          ("di12_u6", 12, 6), ("diq13_u6", 13, 6)):
        e = B.Engine(model, dtype)
        if e.is_di:
            e.set_di_gains(rng.normal(0, 0.1, (nu, 3)), rng.normal(0, 0.1, (nu, 3)))
        n, T = 333, 23
        x0 = rng.uniform(-0.5, 0.5, (n, nx))
        if nx == 13:
            x0[:, 3:7] /= np.linalg.norm(x0[:, 3:7], axis=1, keepdims=True)
        U = rng.uniform(-0.5, 0.5, (T, n, nu))
        for integ in ("rk4", "euler"):
            r = e.rollout(x0, U, dt=dt, integrator=integ, stride=5)
            r2 = e.rollout(x0, U[:, 0], dt=dt, integrator=integ, stride=0, u_layout="shared")
            e.rollout(x0, U, dt=dt, integrator=integ, stride=3, time_slices=3)
            assert torch.isfinite(r.xT).all() and torch.isfinite(r2.xT).all()
        if not e.is_di:   # round-2 paths: generated commands, projected lag carry, health counters, materialised stream
            gen = B.InputGenerator(seed=7, sigma=0.05, scale=None if nu == 8 else [8, 8, 8, 0.3, 0.3, 0.3], vehicle0=11)
            mc = torch.empty(n, device="cuda", dtype=e.tdtype)
            r1 = e.rollout(x0, gen=gen, steps=T, dt=dt, stride=4, health=True, min_abs_cos=mc,
                           lag_repr="projected" if model == "thruster8" else "thruster")
            r2 = e.rollout(r1.xT, gen=gen, steps=60, step0=T, dt=dt, lag0=r1.lag, gen_state=r1.gen_state, health=True,
                           min_abs_cos=mc, min_abs_cos_accumulate=True, time_slices=2,
                           lag_repr="projected" if model == "thruster8" else "thruster")
            assert torch.isfinite(r2.xT).all() and int(r2.health[0]) == 0
            e.generate_inputs(gen, steps=T, first=5, n_sel=17)
            e.rollout_host(np.ascontiguousarray(x0.astype(e.ndtype)), gen=gen, steps=41, dt=dt, chunk_steps=16, health=np.zeros(2, np.uint64))
            if model == "thruster8":   # per-thruster lag epilogue: shorter and longer than the filter memory
                e.rollout(x0, gen=gen, steps=5, dt=dt, lag0=np.full((n, 24), 0.01))
                e.rollout(x0, gen=gen, steps=70, dt=dt, lag0=np.full((n, 24), 0.01))
                e.rollout(x0, np.tile(U, (4, 1, 1)), dt=dt, lag0=np.full((n, 24), 0.01))
            if dtype == "f64":   # step Jacobians: ragged last block of the shared-memory J tile, both integrators
                for integ in ("rk4", "euler"):
                    rl = e.linearize(x0[:101], U[:5, :101], dt=dt, integrator=integ, health=True)
                    assert torch.isfinite(rl.A).all() and int(rl.health[0]) == 0
            # closed loop: ragged n (partial last warp of the snapshot tiles), per-vehicle time-varying gains, cost
            nz = e.nz
            Kc = rng.normal(0, 0.05, (T, 101, nu, nz))
            rc = e.closed_loop(x0[:101], Kc, np.zeros(nz), np.zeros(nu), dt=dt, stride=2, want_u=True,
                               cost_q=1.0, cost_r=1.0, health=True, u_min=-1.0, u_max=1.0)
            assert torch.isfinite(rc.z).all() and int(rc.health[0]) == 0
            if dtype == "f64" and model != "quat13":
                # extended Kalman filters: partial last block, NaN measurement masks, per-filter q and r, P snapshots
                Ye = x0[:101] + 0.01 * rng.standard_normal((T, 101, nx))
                Ye[rng.random(Ye.shape) < 0.5] = np.nan
                for integ in ("rk4", "euler"):
                    re_ = e.ekf(x0[:101], np.eye(nx) * 0.01, U[:, :101], Ye, rng.uniform(1e-6, 1e-4, (101, nx)),
                                rng.uniform(1e-4, 1e-3, (101, nx)), dt=dt, integrator=integ, stride=4, want_cov=True,
                                health=True)
                    assert torch.isfinite(re_.P).all() and int(re_.health[0]) == 0
        e.rhs(x0, U[0])
        e.step(x0, U[0], dt=dt, integrator="euler")
        if model != "thruster8":
            e.rhs_host(x0.astype(e.ndtype), U[0].astype(e.ndtype), dt=dt)
        X = r.traj[:, 0, :].contiguous()
        e.multistep_rmse(np.tile(X.cpu().numpy(), (8, 1)), np.tile(U[:X.shape[0], 0], (8, 1)), [1, 3, 7], dt=dt)
        if model == "thruster8":
            e.thruster_wrench(U[0], lag=torch.zeros((n, 24), device="cuda", dtype=e.tdtype), dt=dt)
            e.thruster_wrench_series(U[:, 0], lag0=np.full(24, 0.01), dt=dt)
            e.thruster_wrench_host(U[0].astype(e.ndtype), lag=np.zeros((n, 24), e.ndtype), dt=dt)
            e.rhs_host(x0.astype(e.ndtype), U[0].astype(e.ndtype), lag=np.zeros((n, 24), e.ndtype), dt=dt)
            e.multistep_rmse(np.tile(X.cpu().numpy(), (60, 1)), np.tile(U[:X.shape[0], 0], (60, 1)), 5, dt=dt,
                             lag_mode="carry")
            xh, uh = x0.astype(e.ndtype), U.astype(e.ndtype)
            e.rollout_host(np.ascontiguousarray(xh), np.ascontiguousarray(uh), dt=dt, stride=4, chunk_steps=8)
        if model in ("wrench12", "quat13"):
            ph = np.tile(B.default_physical(), (n, 1)) * rng.uniform(0.9, 1.1, (n, 1))
            e.set_vehicle_physical(ph)
            e.rollout(x0, U, dt=dt, stride=2)
            e.set_vehicle_physical(None)
            e.set_wrench_lag1(True, 0.1)
            e.rollout(x0, U, dt=dt, stride=0)
    x9 = torch.randn((1001, 9), device="cuda", dtype=torch.float32 if dtype == "f32" else torch.float64)
    B.reduced9_rhs(x9, torch.randn((1001, 4), device="cuda", dtype=x9.dtype))

# Koopman
n, r, k, T = 12, 8, 37, 300
K = KoopmanEDMDc(state_dim=n, input_dim=r, n_rbfs=k, gamma=0.5)
K.centers_ = rng.uniform(-1, 1, (k, n))
K.A_ = 0.9 * np.linalg.qr(rng.standard_normal((n + k, n + k)))[0]
K.B_ = 0.1 * rng.standard_normal((n + k, r))
Xk, Uk = np.cumsum(0.05 * rng.standard_normal((T, n)), axis=0), rng.uniform(-1, 1, (T, r))
for H in (1, 7, 150):
    assert np.isfinite(K.multistep_rmse(Xk, Uk, H))
K.multistep_rmse_multi(Xk, Uk, [1, 7, 150, 2, 33])
K.simulate(Xk[0], Uk[:77])
K.simulate_batch(Xk[:5], Uk[:33])
K._lift(Xk[:19])

# PINc (reference checkpoint from the golden file)
cg = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors_cmp.npz"))
g = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))
M = P.PincModel({kk[len("pinc_sd_"):]: cg[kk] for kk in cg.files if kk.startswith("pinc_sd_")})
M(cg["pinc_dataset_zin"][:77])
M.rollout(np.tile(g["rmse_X12"][:3], (150, 1))[:401], np.tile(g["rmse_U8"][:17, None, :], (1, 401, 1)), dt, stride=4)
P.multistep_rmse_endpoint_pinc(g["rmse_X12"], g["rmse_U8"], [1, 10, 100], dt, M, lag_mode="reset")
P.multistep_rmse_endpoint_pinc(g["rmse_X12"], g["rmse_U8"], 10, dt, M)
# tensor-core evaluator: more windows than one CTA's two tiles, ragged last tile, both lag modes
Xl, Ul = np.tile(g["rmse_X12"], (6, 1)), np.tile(g["rmse_U8"], (6, 1))
P.multistep_rmse_endpoint_pinc(Xl, Ul, [1, 10, 100], dt, M, lag_mode="reset")
P.multistep_rmse_endpoint_pinc(Xl, Ul, 10, dt, M)
M(np.tile(cg["pinc_dataset_zin"], (8, 1))[:700])
torch.cuda.synchronize()
print("sanitize_smoke OK")
