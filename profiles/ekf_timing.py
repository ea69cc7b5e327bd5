"""Extended Kalman filters (brov_ekf) against Engine.linearize and against the composed torch loop, on a GPU.

    python profiles/ekf_timing.py [--out DIR] [--quick]

For thruster8 and wrench12 (fp64, RK4):
  N = 16,384 x T = 50, every component measured: one Engine.ekf call next to one Engine.linearize call of the same
      shape; rate = N * T * NX / ekf_ms and N * T * NC / lin_ms, in thread-steps per second (one thread per filter
      and column in both kernels), and their ratio;
  N = 65,536 x T = 1000: every component measured, and the BlueROV2 sensor pattern (depth, attitude and gyro every
      step, DVL u, v, w every 10th step, no x, y).
The composed loop — per step one Engine.linearize call with T = 1 and the covariance algebra and scalar updates as
torch operations on the device, the filter of oracle/ekf_np.py path (b) — is timed at N = 4096 x T = 1000 after its
final state, covariance and log-likelihood have been checked against the kernel's.  Per-filter inputs and
measurements are larger than the L2 cache at the big sizes.  Registers and stack of every ekf_kernel instantiation
come from compiling csrc/brov_lin.cu with -Xptxas -v into a temporary directory.  Writes DIR/ekf_timing.json
(default: the current directory) with the card's name, power limit and maximum SM clock read in the same run."""
import json
import math
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DT = 0.02
R_STD = [0.05] * 3 + [0.01] * 3 + [0.02] * 3 + [0.01] * 3
Q_VAR = [1e-8] * 6 + [1e-6] * 6


def ptxas_report():
    from bluerov2_dynamics_b200.build import CSRC, NVCC_FLAGS, _nvcc
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, "brov_lin.cu"), "-o", os.path.join(d, "l.o")],
                           capture_output=True, text=True, check=True)
    out, name = {}, None
    models = {"0": "thruster8", "1": "wrench12"}
    integs = {"0": "rk4", "1": "euler"}
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '_ZN4brov(\d+)(\w+?)_kernelILi(\d)ELi(\d)E", line)
        if m:
            name = f"{models[m.group(3)]}_{integs[m.group(4)]}" if m.group(2) == "ekf" else None
            if name:
                out[name] = {}
        elif name and "bytes stack frame" in line:
            v = [int(x) for x in re.findall(r"(\d+) bytes", line)]
            out[name].update(stack=v[0], spill_stores=v[1], spill_loads=v[2])
        elif name and "Used" in line and "registers" in line:
            out[name]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
            out[name]["smem"] = int(re.search(r"(\d+) bytes smem", line).group(1))
    return out


def composed_ekf(e, x0, Z0, P0, U, Y, q, r):
    """the filter of brov_ekf as a Python loop: Engine.linearize (T = 1) per step, torch for the rest"""
    import torch
    nx = e.nx
    x, Z, P = x0.clone(), Z0, P0.clone()
    n = x.shape[0]
    ll = torch.zeros(n, dtype=torch.float64, device=x.device)
    nis = torch.zeros_like(ll)
    cnt = torch.zeros(n, dtype=torch.int64, device=x.device)
    Q = torch.diag(q)
    eye = torch.eye(nx, dtype=torch.float64, device=x.device)
    two_pi = 2 * math.pi
    for k in range(Y.shape[0]):
        res = e.linearize(x, U[k], dt=DT, lag0=Z, lag_repr="projected", want_traj=False)
        A = res.A[0, :, :nx, :nx]
        x = res.z[:, :nx].clone()
        Z = res.z[:, nx:] if Z is not None else None
        P = A @ P @ A.transpose(1, 2) + Q
        P = torch.triu(P) + torch.triu(P, 1).transpose(1, 2)
        for j in range(nx):
            y = Y[k, :, j]
            m = torch.isfinite(y)
            nu = torch.where(m, y - x[:, j], 0.0)
            if 3 <= j < 6:
                nu = nu - two_pi * torch.round(nu / two_pi)
            s = P[:, j, j] + r[j]
            g = P[:, :, j] / s[:, None]
            x = x + torch.where(m[:, None], g * nu[:, None], 0.0)
            Kf = eye - g[:, :, None] * eye[j][None, None, :]
            Pn = Kf @ P @ Kf.transpose(1, 2) + r[j] * g[:, :, None] * g[:, None, :]
            Pn = torch.triu(Pn) + torch.triu(Pn, 1).transpose(1, 2)
            P = torch.where(m[:, None, None], Pn, P)
            e2 = nu * nu / s
            ll = ll - torch.where(m, 0.5 * (e2 + torch.log(s) + math.log(two_pi)), 0.0)
            nis = nis + torch.where(m, e2, 0.0)
            cnt = cnt + m.to(torch.int64)
    return x, P, ll, nis, cnt


def main():
    import numpy as np
    import torch
    import bluerov2_dynamics_b200 as B
    args = sys.argv[1:]
    outdir = args[args.index("--out") + 1] if "--out" in args else os.getcwd()
    quick = "--quick" in args
    os.makedirs(outdir, exist_ok=True)
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    regs = ptxas_report()
    print(json.dumps(regs), flush=True)
    rng = np.random.default_rng(0)

    def timed(fn, min_s=0.5):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        one = a.elapsed_time(b)
        reps = max(1, min(20, int(min_s * 1e3 / max(one, 1e-3))))
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def problem(e, n, T, pattern):
        x0 = np.zeros((n, 12))
        x0[:, :3] = rng.uniform(-1, 1, (n, 3))
        x0[:, 3:6] = rng.uniform(-0.3, 0.3, (n, 3))
        x0[:, 6:] = rng.uniform(-0.2, 0.2, (n, 6))
        thr = e.model == "thruster8"
        U = torch.as_tensor(rng.uniform(-0.5, 0.5, (T, n, e.nu)) * (1.0 if thr else 5.0), device="cuda")
        Y = torch.as_tensor(np.repeat(x0[None], T, axis=0), device="cuda")
        Y += torch.randn_like(Y) * torch.as_tensor(R_STD, device="cuda", dtype=torch.float64)
        if pattern == "bluerov2":
            Y[:, :, :2] = float("nan")
            Y[(torch.arange(T, device="cuda") % 10 != 9)[:, None].expand(T, n), 6:9] = float("nan")
        Z0 = e.tensor(rng.uniform(-0.5, 0.5, (n, 18))) if thr else None
        return e.tensor(x0), Z0, U, Y

    q = np.array(Q_VAR)
    rv = np.array(R_STD) ** 2
    P0 = np.diag(np.full(12, 1e-2))
    cases = []
    for model in ("thruster8", "wrench12"):
        e = B.Engine(model, "f64")
        nc = e.nz + e.nu
        sizes = [(16384, 50, "all")] + ([] if quick else [(65536, 1000, "all"), (65536, 1000, "bluerov2")])
        for n, T, pattern in sizes:
            x0, Z0, U, Y = problem(e, n, T, pattern)
            kw = dict(dt=DT, lag0=Z0, lag_repr="projected")
            t_ekf = timed(lambda: e.ekf(x0, P0, U, Y, q, rv, **kw))
            row = dict(model=model, integrator="rk4", N=n, T=T, measured=pattern, ekf_ms=t_ekf,
                       ekf_thread_steps_per_s=n * T * 12 / (t_ekf * 1e-3), filter_steps_per_s=n * T / (t_ekf * 1e-3),
                       scalar_updates=int(torch.isfinite(Y).sum()))
            if T == 50:
                t_lin = timed(lambda: e.linearize(x0, U, dt=DT, lag0=Z0, lag_repr="projected", want_traj=False))
                row.update(lin_ms=t_lin, NC=nc, lin_thread_steps_per_s=n * T * nc / (t_lin * 1e-3))
                row["rate_over_linearize"] = row["ekf_thread_steps_per_s"] / row["lin_thread_steps_per_s"]
            with_traj = timed(lambda: e.ekf(x0, P0, U, Y, q, rv, stride=10, **kw)) if T == 1000 else None
            if with_traj is not None:
                row["ekf_ms_x_traj_stride10"] = with_traj
            cases.append(row)
            print(json.dumps(row), flush=True)
            del U, Y
            torch.cuda.empty_cache()

    # the composed torch loop of oracle path (b), checked against the kernel first
    comp = []
    for model in ("thruster8", "wrench12"):
        e = B.Engine(model, "f64")
        n, T = 4096, (100 if quick else 1000)
        x0, Z0, U, Y = problem(e, n, T, "bluerov2")
        qt, rt, P0t = e.tensor(q), e.tensor(rv), e.tensor(np.tile(P0, (n, 1, 1)))
        k = e.ekf(x0, P0t, U, Y, q, rv, dt=DT, lag0=Z0, lag_repr="projected")
        c = composed_ekf(e, x0, Z0, P0t, U, Y, qt, rt)
        torch.cuda.synchronize()

        def nw(a, b):
            return float((a - b).abs().max() / b.abs().max())
        agree = dict(x=nw(c[0], k.z[:, :12]), P=nw(c[1], k.P), loglik=nw(c[2], k.loglik),
                     count_equal=bool(torch.equal(c[4], k.count)))
        t_k = timed(lambda: e.ekf(x0, P0t, U, Y, q, rv, dt=DT, lag0=Z0, lag_repr="projected"))
        t_c = timed(lambda: composed_ekf(e, x0, Z0, P0t, U, Y, qt, rt), min_s=0.0)
        row = dict(model=model, N=n, T=T, measured="bluerov2", ekf_ms=t_k, composed_ms=t_c, speedup=t_c / t_k,
                   composed_vs_kernel=agree)
        comp.append(row)
        print(json.dumps(row), flush=True)
    res = dict(gpu=info, ptxas=regs, cases=cases, composed=comp)
    with open(os.path.join(outdir, "ekf_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("# gpu:", info)


if __name__ == "__main__":
    main()
