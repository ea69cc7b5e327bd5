"""Step Jacobians (brov_linearize) against central differences of the rollout, on a GPU.

    python profiles/lin_timing.py [--out DIR] [--quick]

For thruster8, wrench12 and quat13 (fp64, RK4) at N in {1, 64, 4096, 16384} vehicles and T in {1, 50} steps:
  lin_ms   one Engine.linearize call (J [T, N, NZ, NC], primal trajectory and final state);
  cd_ms    the same Jacobians by central differences: the nominal trajectory (one Engine.rollout with stride 1; for the
           thruster model T one-step calls, since the projected lag of every step is needed), the N*T*2*NC perturbed
           copies assembled on the device, one batched Engine.rollout(steps=1, lag_repr="projected") over all of
           them, and the differences; cd_rollout_ms is the nominal trajectory and the batched rollout alone;
  rate     N * NC * T / lin_ms, in thread-steps per second (one thread per vehicle and column).
se_grad_kernel's rate is measured in the same run for comparison (thruster8 RK4, a 45,823-row series, 18 directions,
H = 1/10/100: windows x 18 x 100 thread-steps).  Registers and stack of every linearize_kernel instantiation come from
compiling csrc/brov_lin.cu with -Xptxas -v into a temporary directory.  Writes DIR/lin_timing.json (default: the
current directory) with the card's name, power limit and maximum SM clock read in the same run.  States and inputs are
random in the tank's range: the cost does not depend on the values."""
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DT = 0.02


def ptxas_report():
    from bluerov2_dynamics_b200.build import CSRC, NVCC_FLAGS, _nvcc
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, "brov_lin.cu"), "-o", os.path.join(d, "l.o")],
                           capture_output=True, text=True, check=True)
    out, name = {}, None
    models = {"0": "thruster8", "1": "wrench12", "2": "quat13"}
    integs = {"0": "rk4", "1": "euler"}
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '_ZN4brov16linearize_kernelILi(\d)ELi(\d)E", line)
        if m:
            name = f"{models[m.group(1)]}_{integs[m.group(2)]}"
            out[name] = {}
        elif name and "bytes stack frame" in line:
            v = [int(x) for x in re.findall(r"(\d+) bytes", line)]
            out[name].update(stack=v[0], spill_stores=v[1], spill_loads=v[2])
        elif name and "Used" in line and "registers" in line:
            out[name]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
            out[name]["smem"] = int(re.search(r"(\d+) bytes smem", line).group(1))
    return out


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

    def timed(fn, min_s=0.3):
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

    # se_grad_kernel reference rate
    e = B.Engine("thruster8", "f64")
    rows = 45823
    X = 0.3 * np.tanh(np.cumsum(rng.normal(0, 0.01, (rows, 12)), axis=0))
    U = np.clip(np.cumsum(rng.normal(0, 0.02, (rows, 8)), axis=0) * 0.2, -1, 1)
    Xt, Ut = e.tensor(X), e.tensor(U)
    ph = B.with_minv(B.default_physical())
    t_grad = timed(lambda: e.multistep_se_grad(Xt, Ut, [1, 10, 100], ph, ["added", "lin", "quad"], dt=DT))
    grad = dict(rows=rows, p=18, H=[1, 10, 100], ms=t_grad, thread_steps_per_s=(rows - 1) * 18 * 100 / (t_grad * 1e-3))
    print(json.dumps(grad), flush=True)
    del Xt, Ut

    cases = []
    for model in ("thruster8", "wrench12", "quat13"):
        e = B.Engine(model, "f64")
        nx, nu, nz = e.nx, e.nu, e.nz
        nc = nz + nu
        thr = model == "thruster8"
        for n in ((1, 4096) if quick else (1, 64, 4096, 16384)):
            for T in (1, 50):
                x0 = np.zeros((n, nx))
                x0[:, :3] = rng.uniform(-1, 1, (n, 3))
                if nx == 13:
                    x0[:, 3] = 1.0
                    x0[:, 7:] = rng.uniform(-0.2, 0.2, (n, 6))
                else:
                    x0[:, 3:6] = rng.uniform(-0.3, 0.3, (n, 3))
                    x0[:, 6:] = rng.uniform(-0.2, 0.2, (n, 6))
                x0t = e.tensor(x0)
                lag0 = e.tensor(rng.uniform(-0.5, 0.5, (n, 18))) if thr else None
                Ut = e.tensor(rng.uniform(-0.5, 0.5, (T, n, nu)) * (1.0 if thr else 5.0))
                t_lin = timed(lambda: e.linearize(x0t, Ut, dt=DT, lag0=lag0, lag_repr="projected"))
                h = 1e-6

                def nominal():
                    if not thr:
                        return e.rollout(x0t, Ut, dt=DT, stride=1).traj
                    # the rollout's trajectory holds x only: the projected lag of every step takes one-step calls
                    zs, x, lg = [], x0t, lag0
                    for k in range(T):
                        r = e.rollout(x, Ut[k:k + 1], dt=DT, lag0=lg, lag_repr="projected")
                        x, lg = r.xT, r.lag
                        zs.append(torch.cat([x, lg], dim=1))
                    return torch.stack(zs)

                def perturbed(zs):
                    z_in = torch.cat([torch.cat([x0t] + ([lag0] if thr else []), dim=1)[None], zs[:-1]])   # [T, n, nz]
                    w = torch.cat([z_in, Ut], dim=2)                                                     # [T, n, nc]
                    W = w[:, :, None, None, :].expand(T, n, nc, 2, nc).clone()
                    idx = torch.arange(nc, device=W.device)
                    W[:, :, idx, 0, idx] += h
                    W[:, :, idx, 1, idx] -= h
                    return W.reshape(-1, nc)

                def batched(W):
                    r = e.rollout(W[:, :nx], W[:, nz:][None], dt=DT, lag0=W[:, nx:nz] if thr else None,
                                  lag_repr="projected")
                    return torch.cat([r.xT, r.lag], dim=1) if thr else r.xT

                def cd():
                    W = perturbed(nominal())
                    out = batched(W).reshape(T, n, nc, 2, nz)
                    return ((out[:, :, :, 0] - out[:, :, :, 1]) / (2 * h)).transpose(2, 3)

                t_cd = timed(cd)
                W = perturbed(nominal())
                t_cd_roll = timed(nominal) + timed(lambda: batched(W))
                del W
                rate = n * nc * T / (t_lin * 1e-3)
                r = dict(model=model, integrator="rk4", N=n, T=T, NC=nc, lin_ms=t_lin, cd_ms=t_cd,
                         cd_rollout_ms=t_cd_roll, cd_copies=n * T * 2 * nc, cd_over_lin=t_cd / t_lin,
                         thread_steps_per_s=rate, rate_over_se_grad=rate / grad["thread_steps_per_s"],
                         jac_GB_per_s=T * n * nz * nc * 8 / (t_lin * 1e-3) / 1e9)
                cases.append(r)
                print(json.dumps(r), flush=True)
                torch.cuda.empty_cache()
    res = dict(gpu=info, ptxas=regs, se_grad=grad, cases=cases)
    with open(os.path.join(outdir, "lin_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("# gpu:", info)


if __name__ == "__main__":
    main()
