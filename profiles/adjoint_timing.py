"""Reverse-mode rollout gradients (brov_rollout_vjp) against Engine.rollout and against the composed route through
Engine.linearize, on a GPU.

    python profiles/adjoint_timing.py [--out DIR] [--quick]

  thruster8 fp64 RK4, N = 65,536 x T = 1000, per-vehicle U, cotangents on x every 10 steps plus a terminal one: one
      Engine.rollout_vjp call next to one Engine.rollout call with the same inputs and a trajectory every 10 steps,
      their ratio against the 6x target, and the workspace traffic (N * T * NZ doubles written and read once).  The
      composed route cannot run here: J alone would be N * T * NZ * NC doubles (598 GB).
  N = 16,384 x T = 50, all three models, RK4: one rollout_vjp call against Engine.linearize followed by the chain
      lambda_k = A_k^T lambda_{k+1} + c_k, gu_k = B_k^T lambda_{k+1} in torch (2T launches), with the gradients of both
      compared, against the 5x target.
Every timing is the median of several CUDA-event-timed calls after a warm-up call of the same shape; the inputs are
larger than the L2 cache.  Registers and stack of every adjoint_kernel instantiation come from compiling
csrc/brov_adj.cu with -Xptxas -v into a temporary directory.  Writes DIR/adjoint_timing.json (default: the current
directory) with the card's name, power limit and maximum SM clock read in the same run."""
import argparse
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
        r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, "brov_adj.cu"), "-o", os.path.join(d, "a.o")],
                           capture_output=True, text=True, check=True)
    out, name = {}, None
    models = {"0": "thruster8", "1": "wrench12", "2": "quat13"}
    integs = {"0": "rk4", "1": "euler"}
    for line in r.stderr.splitlines():
        m = re.search(r"adjoint_kernelILi(\d)ELi(\d)E", line)
        if m and "Compiling entry" in line:
            name = f"{models[m.group(1)]}-{integs[m.group(2)]}"
            out[name] = {}
        elif name and "stack frame" in line:
            out[name]["stack_bytes"] = int(re.search(r"(\d+) bytes stack frame", line).group(1))
            out[name]["spill_store_bytes"] = int(re.search(r"(\d+) bytes spill stores", line).group(1))
        elif name and "Used" in line and "registers" in line:
            out[name]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
            sm = re.search(r"(\d+) bytes smem", line)
            out[name]["smem_bytes"] = int(sm.group(1)) if sm else 0
    return out


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts


def problem(e, n, T, seed):
    import torch
    g = torch.Generator(device=e.device).manual_seed(seed)
    x0 = torch.zeros((n, e.nx), dtype=torch.float64, device=e.device)
    x0[:, :3] = torch.rand((n, 3), generator=g, device=e.device, dtype=torch.float64) * 2 - 1
    if e.nx == 13:
        x0[:, 3] = 1.0
        x0[:, 7:] = (torch.rand((n, 6), generator=g, device=e.device, dtype=torch.float64) - 0.5) * 0.4
    else:
        x0[:, 3:6] = (torch.rand((n, 3), generator=g, device=e.device, dtype=torch.float64) - 0.5) * 0.6
        x0[:, 6:] = (torch.rand((n, 6), generator=g, device=e.device, dtype=torch.float64) - 0.5) * 0.4
    scale = 0.5 if e.model == "thruster8" else 3.0
    U = (torch.rand((T, n, e.nu), generator=g, device=e.device, dtype=torch.float64) - 0.5) * 2 * scale
    return x0, U


def main():
    import torch
    import bluerov2_dynamics_b200 as B
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".")
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": info[torch.cuda.current_device()] if info else torch.cuda.get_device_name(),
           "ptxas": ptxas_report()}
    reps = 3 if a.quick else 5

    # ---- 65,536 x 1000 thruster8 RK4
    n, T, stride = (8192, 200, 10) if a.quick else (65536, 1000, 10)
    e = B.Engine("thruster8", "f64")
    x0, U = problem(e, n, T, 1)
    g = torch.Generator(device=e.device).manual_seed(2)
    gtraj = torch.randn((T // stride, n, 12), generator=g, device=e.device, dtype=torch.float64)
    gzT = torch.randn((n, 30), generator=g, device=e.device, dtype=torch.float64)
    t_vjp, all_vjp = timed(lambda: e.rollout_vjp(x0, U, gtraj=gtraj, gzT=gzT, stride=stride, dt=DT), reps)
    t_ro, all_ro = timed(lambda: e.rollout(x0, U, dt=DT, stride=stride, lag_repr="projected"), reps)
    ws = n * T * 30 * 8
    ratio = t_vjp / t_ro
    res["big"] = dict(model="thruster8", integrator="rk4", n=n, steps=T, stride=stride, vjp_ms=t_vjp, rollout_ms=t_ro,
                      vjp_ms_all=all_vjp, rollout_ms_all=all_ro, ratio=ratio, target_ratio=6.0,
                      target="met" if ratio <= 6.0 else "missed",
                      workspace_written_GB=ws / 1e9, workspace_read_GB=ws / 1e9,
                      workspace_traffic_GBps=2 * ws / 1e9 / (t_vjp / 1e3),
                      composed_route_jacobian_GB=n * T * 30 * 38 * 8 / 1e9)
    print(json.dumps(res["big"]), flush=True)
    del x0, U, gtraj, gzT
    torch.cuda.empty_cache()

    # ---- 16,384 x 50, all models: adjoint against linearize + torch chain
    n, T, stride = (4096, 50, 10) if a.quick else (16384, 50, 10)
    res["small"] = {}
    for model in ("thruster8", "wrench12", "quat13"):
        e = B.Engine(model, "f64")
        x0, U = problem(e, n, T, 3)
        g = torch.Generator(device=e.device).manual_seed(4)
        gtraj = torch.randn((T // stride, n, e.nx), generator=g, device=e.device, dtype=torch.float64)
        gzT = torch.randn((n, e.nz), generator=g, device=e.device, dtype=torch.float64)

        def composed():
            lin = e.linearize(x0, U, dt=DT, want_traj=False)
            lam = gzT.clone()
            gU = torch.empty((T, n, e.nu), dtype=torch.float64, device=e.device)
            for k in range(T - 1, -1, -1):
                if (k + 1) % stride == 0:
                    lam[:, :e.nx] += gtraj[(k + 1) // stride - 1]
                gU[k] = torch.einsum("nzu,nz->nu", lin.B[k], lam)
                lam = torch.einsum("nzy,nz->ny", lin.A[k], lam)
            return lam, gU

        def vjp():
            return e.rollout_vjp(x0, U, gtraj=gtraj, gzT=gzT, stride=stride, dt=DT, lag_repr="projected")

        t_v, _ = timed(vjp, reps)
        t_c, _ = timed(composed, reps)
        r = vjp()
        lam, gU = composed()
        gz0 = torch.cat([r.gx0, r.glag0], 1) if model == "thruster8" else r.gx0
        err = float((gz0 - lam).abs().max() / lam.abs().max())
        err_u = float((r.gU - gU).abs().max() / gU.abs().max())
        sp = t_c / t_v
        res["small"][model] = dict(n=n, steps=T, stride=stride, vjp_ms=t_v, linearize_chain_ms=t_c, speedup=sp,
                                   target_speedup=5.0, target="met" if sp >= 5.0 else "missed",
                                   jacobian_GB_of_composed=n * T * e.nz * (e.nz + e.nu) * 8 / 1e9,
                                   normwise_diff_gz0=err, normwise_diff_gU=err_u)
        print(model, json.dumps(res["small"][model]), flush=True)
        del x0, U, gtraj, gzT, r, lam, gU
        torch.cuda.empty_cache()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "adjoint_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
