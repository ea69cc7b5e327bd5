"""Reverse-mode gradients of closed-loop rollouts (brov_closed_loop_vjp) against the open-loop adjoint and against
central differences of the closed loop, on a GPU.

    python profiles/cl_vjp_timing.py [--out DIR] [--quick]

  N = 65,536 x T = 1000, fp64 RK4, every model: Engine.closed_loop_vjp with one const_shared K, the cost cotangent
      g_c only and the gain gradient requested, next to Engine.rollout_vjp on the same size (per-vehicle U, cotangents
      every 10 steps plus a terminal one) in the same run (target for thruster8: <= 1.5x).
  thruster8, N = 8192 x T = 1000, a tnc gain [T][N][8][30]: the same call with and without the gain gradient, and the
      device time of the reduction kernel alone (torch.profiler, a separate pass); the bytes it must move (z_k and gv
      read once, gK written) over that time are its achieved HBM bandwidth.
  thruster8, N = 4096 x T = 500, const_shared K: the gain gradient against central differences in the 240 gains, run as
      one batched Engine.closed_loop call of 481 N vehicles with the const K layout (target >= 10x).
Every timing is the median of several CUDA-event-timed calls after a warm-up call of the same shape; the inputs of the
large calls are larger than the L2 cache.  Registers and stack of every closed_loop_adjoint_kernel instantiation come
from compiling csrc/brov_adj.cu with -Xptxas -v into a temporary directory.  Writes DIR/cl_vjp_timing.json (default:
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
        m = re.search(r"closed_loop_adjoint_kernelILi(\d)ELi(\d)ELb(\d)E", line)
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


def feedback(e, n, T, seed):
    """a hover-like closed loop: references at z0's neighbourhood, a small gain, moderate feedforward"""
    import torch
    g = torch.Generator(device=e.device).manual_seed(seed)
    x0, _ = problem(e, n, 1, seed)
    zr = torch.zeros(e.nz, dtype=torch.float64, device=e.device)
    if e.nx == 13:
        zr[3] = 1.0
    scale = 0.3 if e.model == "thruster8" else 5.0
    K = (torch.rand((e.nu, e.nz), generator=g, device=e.device, dtype=torch.float64) - 0.5) * scale
    ur = torch.zeros(e.nu, dtype=torch.float64, device=e.device)
    return x0, K, zr, ur


def main():
    import numpy as np
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
    qw = np.ones(30)
    rw = np.ones(8)

    n, T, stride = (8192, 200, 10) if a.quick else (65536, 1000, 10)
    res["big"] = {}
    for model in ("thruster8", "wrench12", "quat13"):
        e = B.Engine(model, "f64")
        lim = dict(u_min=-1.0, u_max=1.0) if model == "thruster8" else dict(u_min=-50.0, u_max=50.0)
        x0, K, zr, ur = feedback(e, n, T, 1)
        gc = torch.full((n,), 1.0 / n, dtype=torch.float64, device=e.device)

        def clvjp():
            return e.closed_loop_vjp(x0, K, zr, ur, gcost=gc, steps=T, dt=DT, want=("K",), cost_q=qw[:e.nz],
                                     cost_r=rw[:e.nu], **lim)

        t_c, all_c = timed(clvjp, reps)
        _, U = problem(e, n, T, 2)
        g = torch.Generator(device=e.device).manual_seed(3)
        gtraj = torch.randn((T // stride, n, e.nx), generator=g, device=e.device, dtype=torch.float64)
        gzT = torch.randn((n, e.nz), generator=g, device=e.device, dtype=torch.float64)
        t_v, all_v = timed(lambda: e.rollout_vjp(x0, U, gtraj=gtraj, gzT=gzT, stride=stride, dt=DT), reps)
        r = dict(n=n, steps=T, closed_loop_vjp_ms=t_c, rollout_vjp_ms=t_v, closed_loop_vjp_ms_all=all_c,
                 rollout_vjp_ms_all=all_v, ratio=t_c / t_v, target_ratio=1.5 if model == "thruster8" else None)
        res["big"][model] = r
        print(model, json.dumps(r), flush=True)
        del x0, U, gtraj, gzT
        torch.cuda.empty_cache()

    # ---- tnc gain gradient: the reduction's bandwidth
    n, T = (2048, 200) if a.quick else (8192, 1000)
    e = B.Engine("thruster8", "f64")
    x0, K1, zr, ur = feedback(e, n, T, 4)
    Kt = K1.expand(T, n, 8, 30).contiguous()
    gzT = torch.randn((n, e.nz), device=e.device, dtype=torch.float64)

    def tnc(want):
        return lambda: e.closed_loop_vjp(x0, Kt, zr, ur, gzT=gzT, dt=DT, want=want, k_layout="tnc")

    t_with, _ = timed(tnc(("K",)), reps)
    t_without, _ = timed(tnc(()), reps)
    # the reduction kernel on its own: its device time from torch.profiler, in a separate pass after the timed calls
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            tnc(("K",))()
        torch.cuda.synchronize()
    red = [ev for ev in prof.key_averages() if "cl_red_steps_kernel" in ev.key]
    red_us = sum(getattr(ev, "device_time_total", 0) or ev.cuda_time_total for ev in red)
    red_ms = red_us / 1e3 / reps
    nbytes = n * T * 8 * (30 + 8 + 240)           # z_k and gv read once, gK written once
    res["tnc_gK"] = dict(n=n, steps=T, with_gK_ms=t_with, without_gK_ms=t_without, reduction_kernel_ms=red_ms,
                         reduction_kernel_launches=sum(ev.count for ev in red) // reps, reduction_bytes=nbytes,
                         reduction_TBps=nbytes / (red_ms * 1e-3) / 1e12,
                         bytes_note="z_k [T][30][N] and gv [T][8][N] counted once and gK [T][N][8][30] written once; "
                                    "each gv element is read by the 30 row threads of its vehicle, from cache after the "
                                    "first; the difference with_gK_ms - without_gK_ms also contains the sweep's gv stores")
    print(json.dumps(res["tnc_gK"]), flush=True)
    del Kt
    torch.cuda.empty_cache()

    # ---- central differences in the 240 gains as one batched closed_loop call
    n, T = (512, 100) if a.quick else (4096, 500)
    x0, K, zr, ur = feedback(e, n, T, 5)
    lim = dict(u_min=-1.0, u_max=1.0)
    gc = torch.full((n,), 1.0 / n, dtype=torch.float64, device=e.device)
    t_a, _ = timed(lambda: e.closed_loop_vjp(x0, K, zr, ur, gcost=gc, steps=T, dt=DT, want=("K",), cost_q=qw,
                                             cost_r=rw, **lim), reps)
    nb = 481 * n
    h = 1e-6
    dirs = torch.zeros((481, 8, 30), dtype=torch.float64, device=e.device)
    dirs[1:241].view(240, 240)[torch.arange(240), torch.arange(240)] = h
    dirs[241:].view(240, 240)[torch.arange(240), torch.arange(240)] = -h
    Kb = (K[None] + dirs)[:, None].expand(481, n, 8, 30).reshape(nb, 8, 30).contiguous()
    xb = x0.repeat(481, 1)
    t_cd, _ = timed(lambda: e.closed_loop(xb, Kb, zr, ur, steps=T, dt=DT, k_layout="const", cost_q=qw, cost_r=rw, **lim),
                    reps)
    res["central_differences"] = dict(model="thruster8", n=n, steps=T, adjoint_ms=t_a, batched_closed_loop_vehicles=nb,
                                      central_differences_ms=t_cd, ratio=t_cd / t_a, target_ratio=10.0)
    print(json.dumps(res["central_differences"]), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "cl_vjp_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
