"""Coefficient gradients of batched rollouts (brov_rollout_vjp_coef) against the adjoint without them, against central
differences and against the forward-mode gradient of multistep_se_grad, on a GPU.

    python profiles/adjoint_coef_timing.py [--out DIR] [--quick]

  N = 65,536 x T = 1000, fp64 RK4, per-vehicle U, cotangents on x every 10 steps plus a terminal one, every model:
      Engine.rollout_vjp(coef=True) next to rollout_vjp(coef=False) and Engine.rollout on the same inputs (target:
      coef <= 1.5x the plain adjoint), and, thruster8, with a per-vehicle table of N rows (target <= 1.1x the shared
      call).  Central differences in all 34 coefficients cost 69 rollouts: 69 x the rollout time of the same call,
      against the 5x target.
  N = 16,384 x T = 50, thruster8 RK4, single-window loss |x_50 - X_50|^2 from 16,384 starting rows of one series:
      rollout_vjp(coef=True) against Engine.multistep_se_grad at p = 18 (added, lin, quad) and p = 36 (every physical
      parameter, rebuild_minv=False).
Every timing is the median of several CUDA-event-timed calls after a warm-up call of the same shape; the 65,536-vehicle
inputs are larger than the L2 cache.  Registers and stack of every adjoint_coef_kernel instantiation come from
compiling csrc/brov_adj.cu with -Xptxas -v into a temporary directory.  Writes DIR/adjoint_coef_timing.json (default:
the current directory) with the card's name, power limit and maximum SM clock read in the same run."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from adjoint_timing import DT, problem, timed  # noqa: E402


def ptxas_report():
    from bluerov2_dynamics_b200.build import CSRC, NVCC_FLAGS, _nvcc
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, "brov_adj.cu"), "-o", os.path.join(d, "a.o")],
                           capture_output=True, text=True, check=True)
    out, name = {}, None
    models = {"0": "thruster8", "1": "wrench12", "2": "quat13"}
    integs = {"0": "rk4", "1": "euler"}
    for line in r.stderr.splitlines():
        m = re.search(r"adjoint_coef_kernelILi(\d)ELi(\d)ELb(\d)E", line)
        if "Compiling entry" in line:
            name = f"{models[m.group(1)]}-{integs[m.group(2)]}-{'table' if m.group(3) == '1' else 'shared'}" if m else None
            if name:
                out[name] = {}
        elif name and "stack frame" in line:
            out[name]["stack_bytes"] = int(re.search(r"(\d+) bytes stack frame", line).group(1))
            out[name]["spill_store_bytes"] = int(re.search(r"(\d+) bytes spill stores", line).group(1))
        elif name and "Used" in line and "registers" in line:
            out[name]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
    return out


def main():
    import numpy as np
    import torch
    import bluerov2_dynamics_b200 as B
    from bluerov2_dynamics_b200 import _lib as L
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".")
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": info[torch.cuda.current_device()] if info else torch.cuda.get_device_name(),
           "ptxas": ptxas_report()}
    reps = 3 if a.quick else 5

    n, T, stride = (8192, 200, 10) if a.quick else (65536, 1000, 10)
    res["big"] = {}
    for model in ("thruster8", "wrench12", "quat13"):
        e = B.Engine(model, "f64")
        x0, U = problem(e, n, T, 1)
        g = torch.Generator(device=e.device).manual_seed(2)
        gtraj = torch.randn((T // stride, n, e.nx), generator=g, device=e.device, dtype=torch.float64)
        gzT = torch.randn((n, e.nz), generator=g, device=e.device, dtype=torch.float64)

        def vjp(coef):
            return lambda: e.rollout_vjp(x0, U, gtraj=gtraj, gzT=gzT, stride=stride, dt=DT, coef=coef)

        t_c, all_c = timed(vjp(True), reps)
        t_v, all_v = timed(vjp(False), reps)
        t_r, _ = timed(lambda: e.rollout(x0, U, dt=DT, stride=stride, lag_repr="projected"), reps)
        r = dict(n=n, steps=T, stride=stride, coef_ms=t_c, vjp_ms=t_v, rollout_ms=t_r, coef_ms_all=all_c,
                 vjp_ms_all=all_v, coef_over_vjp=t_c / t_v, target_coef_over_vjp=1.5,
                 central_differences_ms=69 * t_r, central_differences_over_coef=69 * t_r / t_c,
                 target_central_differences_over_coef=5.0)
        if model == "thruster8":
            rng = np.random.default_rng(5)
            ph = np.tile(B.default_physical(), (n, 1))
            ph[:, L.PH_ADDED:L.PH_QUAD + 6] *= rng.uniform(0.7, 1.3, (n, 18))
            e.set_vehicle_physical(B.with_minv(ph))
            t_t, all_t = timed(vjp(True), reps)
            e.set_vehicle_physical(None)
            r.update(table_ms=t_t, table_ms_all=all_t, table_over_shared=t_t / t_c, target_table_over_shared=1.1)
        res["big"][model] = r
        print(model, json.dumps(r), flush=True)
        del x0, U, gtraj, gzT
        torch.cuda.empty_cache()

    # ---- 16,384 x 50: against forward mode on the same single-window loss
    n, H = (4096, 50) if a.quick else (16384, 50)
    e = B.Engine("thruster8", "f64")
    x0, Us = problem(e, 1, n + H, 7)
    X = e.rollout(x0, Us, dt=DT, stride=1).traj[:, 0]                      # [n + H, NX] recorded series
    X = torch.cat([x0, X[:-1]], 0).contiguous()                             # row k: the state before step k
    X = X + 1e-3 * torch.randn_like(X)
    Uw = torch.stack([Us[k:k + H, 0] for k in range(n)], 1).contiguous()    # [H, n, NU]: window k's inputs
    ph = e.phys
    kp = torch.from_numpy(B.derive_params(B.with_minv(ph))).to(e.device)
    starts, ends = X[:n], X[H:H + n]
    with e._coefficients(kp):
        xH = e.rollout(starts, Uw, dt=DT).xT
    gzT = torch.zeros((n, e.nz), dtype=torch.float64, device=e.device)
    gzT[:, :e.nx] = 2.0 * (xH - ends)

    def adj():
        with e._coefficients(kp):
            return e.rollout_vjp(starts, Uw, gzT=gzT, dt=DT, coef=True)

    t_a, _ = timed(adj, reps)
    Xs, Ust = X[:n + H].contiguous(), Us[:n + H, 0].contiguous()
    p36 = [i for i in range(L.NPHYS) if i != L.PH_TLAG1]
    fwd = {}
    for p, params, rb in ((18, ["added", "lin", "quad"], True), (36, p36, False)):
        t_f, _ = timed(lambda: e.multistep_se_grad(Xs, Ust, [H], ph, params, dt=DT, rebuild_minv=rb), reps)
        ref = e.multistep_se_grad(Xs, Ust, [H], ph, params, dt=DT, rebuild_minv=rb).grad[0].cpu().numpy()
        kpr = torch.from_numpy(B.derive_params(B.with_minv(ph) if rb else ph)).to(e.device)
        with e._coefficients(kpr):
            gk = e.rollout_vjp(starts, Uw, gzT=gzT, dt=DT, coef=True).gkp.sum(0).cpu().numpy()
        got = B.coefficient_directions(ph, params, rebuild_minv=rb) @ gk
        fwd[f"p{p}"] = dict(se_grad_ms=t_f, se_grad_over_adjoint=t_f / t_a,
                            normwise_diff=float(np.abs(got - ref).max() / np.abs(ref).max()))
    res["forward_mode"] = dict(model="thruster8", integrator="rk4", windows=n, horizon=H, adjoint_coef_ms=t_a, **fwd)
    print(json.dumps(res["forward_mode"]), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "adjoint_coef_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
