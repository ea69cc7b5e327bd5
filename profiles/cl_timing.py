"""Closed-loop rollouts (brov_closed_loop) against the open-loop rollout, on a GPU.

    python profiles/cl_timing.py [--out DIR]

Measured, all RK4, start states about the hover trim of examples/station_keeping_lqr.py (thruster8) or near rest
(wrench models), the LQR gain of that example (thruster8) or a small constant gain:
  headline      thruster8 fp64, 65,536 vehicles x 1000 steps, one K for every vehicle and step: vehicle-steps/s and
                the ratio to Engine.rollout of the same size in the same run (shared input series [T, 8], and per-vehicle
                inputs [T, N, 8]);
  cost / traj   the same with the cost on, and with z and u stored every 10 steps;
  models        wrench12 / quat13 fp64 at 65,536 vehicles, thruster8 fp32 at 1,048,576 vehicles, each with its rollout;
  tnc_gains     a per-vehicle time-varying K [T, N, 8, 30] (fp64, 65,536 x 100): operand bytes / s against 7.7 TB/s;
  table         a per-vehicle coefficient table (thruster8 fp64, 65,536 x 1000) against the rollout with the same table;
  example       the example's closed loop (4096 vehicles x 1500 steps, stride 1, band test): Engine.closed_loop in
                chunks of 100 against the Engine.step loop it replaced (project_lag, cat, wrap, matmul, clamp in torch).
Registers and stack of every closed_loop_kernel instantiation come from compiling csrc/brov_cl.cu with -Xptxas -v into
a temporary directory.  Writes DIR/cl_timing.json with the card's name, power limit and maximum SM clock read in the
same run."""
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
DT = 0.02


def ptxas_report():
    from bluerov2_dynamics_b200.build import CSRC, NVCC_FLAGS, _nvcc
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, "brov_cl.cu"), "-o", os.path.join(d, "c.o")],
                           capture_output=True, text=True, check=True)
    out, name = {}, None
    dt = {"d": "f64", "f": "f32"}
    models = {"0": "thruster8", "1": "wrench12", "2": "quat13"}
    integs = {"0": "rk4", "1": "euler"}
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '_ZN4brov18closed_loop_kernelI([df])Li(\d)ELi(\d)ELb(\d)ELb(\d)E", line)
        if m:
            t, mo, i, pv, cu = m.groups()
            name = f"{dt[t]}_{models[mo]}_{integs[i]}{'_table' if pv == '1' else ''}{'_current' if cu == '1' else ''}"
            out[name] = {}
        elif name and "bytes stack frame" in line:
            v = [int(x) for x in re.findall(r"(\d+) bytes", line)]
            out[name].update(stack=v[0], spill_stores=v[1], spill_loads=v[2])
        elif name and "Used" in line and "registers" in line:
            out[name]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
    return out


def main():
    import numpy as np
    import torch
    import bluerov2_dynamics_b200 as B
    import station_keeping_lqr as ex
    args = sys.argv[1:]
    outdir = args[args.index("--out") + 1] if "--out" in args else os.getcwd()
    os.makedirs(outdir, exist_ok=True)
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    regs = ptxas_report()
    rng = np.random.default_rng(0)

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for _ in range(reps):
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return min(ts)

    res = {"device": info, "ptxas": regs}
    # hover trim and LQR of the example
    e = B.Engine("thruster8", "f64")
    zs, us, _, _ = ex.trim(e)
    r = e.linearize(zs[None, :12], us[None], dt=DT, lag0=zs[None, 12:], lag_repr="projected", want_traj=False)
    import scipy.linalg
    A, Bm = r.A[0, 0].cpu().numpy(), r.B[0, 0].cpu().numpy()
    Q = np.diag([10, 10, 10, 5, 5, 5] + [1] * 6 + [1e-6] * 18)
    R = 0.5 * np.eye(8)
    P = scipy.linalg.solve_discrete_are(A, Bm, Q, R)
    K = np.linalg.solve(R + Bm.T @ P @ Bm, Bm.T @ P @ A)

    def start(eng, n, zref):
        z = np.tile(zref, (n, 1))
        z[:, 0:3] += rng.uniform(-0.5, 0.5, (n, 3))
        if eng.nx == 12:
            z[:, 3:6] += rng.uniform(-0.3, 0.3, (n, 3))
        z[:, eng.nx - 6:eng.nx] += rng.uniform(-0.2, 0.2, (n, 6))
        return z

    def pair(eng, n, T, Kx, zref, uref, label, **kw):
        z0 = start(eng, n, zref)
        nx = eng.nx
        thr = eng.model == "thruster8"
        x0, l0 = eng.tensor(z0[:, :nx]), (eng.tensor(z0[:, nx:]) if thr else None)
        Kt, zt, ut = eng.tensor(Kx), eng.tensor(zref), eng.tensor(uref)
        cl = timed(lambda: eng.closed_loop(x0, Kt, zt, ut, steps=T, dt=DT, lag0=l0, lag_repr="projected", **kw))
        Us = eng.tensor(np.clip(uref + 0.05 * rng.standard_normal((T, eng.nu)), -1, 1))
        ro = timed(lambda: eng.rollout(x0, Us, dt=DT, lag0=l0, lag_repr="projected"))
        out = {"n": n, "steps": T, "closed_loop_ms": cl, "vehicle_steps_per_s": n * T / cl * 1e3,
               "rollout_shared_u_ms": ro, "ratio_to_rollout_shared_u": ro / cl}
        if n * T * eng.nu * (8 if eng.dtype == "f64" else 4) <= 8e9:
            Ut = eng.tensor(np.zeros((1, 1, eng.nu))).expand(T, n, eng.nu).contiguous()
            rt = timed(lambda: eng.rollout(x0, Ut, dt=DT, lag0=l0, lag_repr="projected"))
            out.update(rollout_tnc_u_ms=rt, ratio_to_rollout_tnc_u=rt / cl)
            del Ut
        print(label, json.dumps(out), flush=True)
        return out

    n, T = 65536, 1000
    res["headline_thruster8_f64"] = pair(e, n, T, K, zs, us, "headline")
    res["cost_on"] = pair(e, n, T, K, zs, us, "cost", cost_q=np.diag(Q), cost_r=np.diag(R))
    res["traj_stride10"] = pair(e, n, T, K, zs, us, "traj", stride=10, want_u=True)
    for model in ("wrench12", "quat13"):
        w = B.Engine(model, "f64")
        nz = w.nz
        zr = np.zeros(nz)
        zr[2] = 1.0
        if nz == 13:
            zr[3] = 1.0
        Kw = 0.5 * np.concatenate([np.eye(6), np.zeros((6, nz - 12)), np.eye(6)], axis=1)
        res[f"{model}_f64"] = pair(w, n, T, Kw, zr, np.zeros(6), model, u_min=-20.0, u_max=20.0)
    e32 = B.Engine("thruster8", "f32")
    res["thruster8_f32_1M"] = pair(e32, 1 << 20, T, K, zs, us, "f32")
    del e32

    # per-vehicle time-varying gains
    Tk = 100
    z0 = start(e, n, zs)
    x0, l0 = e.tensor(z0[:, :12]), e.tensor(z0[:, 12:])
    Kt = e.tensor(K).expand(Tk, n, 8, 30).contiguous()
    zt, ut = e.tensor(zs), e.tensor(us)
    ms = timed(lambda: e.closed_loop(x0, Kt, zt, ut, dt=DT, lag0=l0, lag_repr="projected"))
    byt = Kt.numel() * 8
    res["tnc_gains"] = {"n": n, "steps": Tk, "ms": ms, "gain_bytes": byt, "bytes_per_s": byt / ms * 1e3,
                        "share_of_7p7_TBps": byt / ms * 1e3 / 7.7e12, "vehicle_steps_per_s": n * Tk / ms * 1e3}
    print("tnc", json.dumps(res["tnc_gains"]), flush=True)
    del Kt
    torch.cuda.empty_cache()

    # per-vehicle coefficient table
    table = np.tile(e.phys, (n, 1))
    for grp in ("added", "lin", "quad"):
        idx = B.engine.PARAM_GROUPS[grp]
        table[:, idx] *= rng.uniform(0.8, 1.2, (n, len(idx)))
    e.set_vehicle_physical(B.with_minv(table))
    res["table"] = pair(e, n, T, K, zs, us, "table")
    e.set_vehicle_physical(None)

    # the example's closed loop: Engine.closed_loop in chunks against the Engine.step loop
    nv, steps = 4096, 1500
    x = start(e, nv, zs)[:, :12]
    lag = ex.lag_steady(us).reshape(1, 24).repeat(nv, 1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ts, settled = ex.settle(e, x, lag, zs, us, K, steps)
    torch.cuda.synchronize()
    t_cl = time.perf_counter() - t0
    t0 = time.perf_counter()
    ts_s, settled_s = step_loop(e, x, lag.clone(), zs, us, K, steps)
    torch.cuda.synchronize()
    t_step = time.perf_counter() - t0
    res["example"] = {"vehicles": nv, "steps": steps, "closed_loop_s": t_cl, "step_loop_s": t_step,
                      "speedup": t_step / t_cl, "settled_closed_loop": int(settled.sum()),
                      "settled_step_loop": int(settled_s.sum()),
                      "median_settling_s_closed_loop": float(np.median(ts)),
                      "median_settling_s_step_loop": float(np.median(ts_s))}
    print("example", json.dumps(res["example"]), flush=True)
    with open(os.path.join(outdir, "cl_timing.json"), "w") as f:
        json.dump(res, f, indent=1)


def step_loop(e, x, lag, zs, us, K, steps):
    """the example's closed loop before Engine.closed_loop: one Engine.step per integrator step, feedback in torch"""
    import numpy as np
    import torch
    dev = e.device
    xt = torch.as_tensor(x, device=dev)
    zs_t, us_t, Kt = (torch.as_tensor(v, device=dev) for v in (zs, us, K))
    n = xt.shape[0]
    inside = torch.zeros((steps, n), dtype=torch.bool, device=dev)
    for k in range(steps):
        dz = torch.cat([xt, e.project_lag(lag)], dim=1) - zs_t
        dz[:, 5] = torch.remainder(dz[:, 5] + np.pi, 2 * np.pi) - np.pi
        u = torch.clamp(us_t - dz @ Kt.T, -1.0, 1.0)
        xt = e.step(xt, u, lag=lag, dt=DT).xT
        err = torch.cat([xt[:, :3] - zs_t[:3], dz[:, 3:6], xt[:, 6:12]], dim=1).abs()
        inside[k] = (err[:, :3].amax(1) < 0.02) & (err[:, 3:6].amax(1) < 0.02) & (err[:, 6:].amax(1) < 0.02)
    stay = torch.flip(torch.cumprod(torch.flip(inside, [0]).to(torch.int32), 0), [0]).bool()
    settled = stay[-1]
    first = torch.where(stay.any(0), stay.to(torch.int8).argmax(0), steps)
    return (first[settled].double() + 1).cpu().numpy() * DT, settled


if __name__ == "__main__":
    main()
