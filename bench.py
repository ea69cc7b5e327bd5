#!/usr/bin/env python3
"""bench.py — RK4 vehicle-steps/s of the batched BlueROV2 Fossen rollout (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA engine
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference itself on the host CPU cores
    python bench.py ... --dump-outputs DIR                           # also save the headline leg's results as .npy

One "step" = one pass of the hot path over one batch of synthetic input: ONE rollout call that advances every vehicle
of the ensemble by 1000 RK4 steps (configs[1]; 100 for configs[2], whose snapshots are written every 10 steps).  The
default K = 20 is twice the 10,000-step rollout of BASELINE configs[1].

Primary line (`value`, `roofline`, `e2e`): configs[1] — 65,536 vehicles per GPU, fp64, 8-thruster model with the
3rd-order lag, dt = 0.02, the reference's smooth random thrust commands.  The commands are the engine's counter-based
stream (Philox4x32-10 keyed on seed / vehicle / step, training/train_sim_brov2_koopmanEDMDc.py:161-164 as the
recursion), so three ways of feeding them exist and all are timed on the SAME numbers:
  value             inputs resident in HBM as a time-major array (10 distinct 1000-step chunks = 10,000 distinct steps,
                    41.9 GB, each chunk far larger than L2 and read once per launch), streamed by the kernel;
  roofline.generated  inputs generated inside the kernel (no input array at all);
  e2e               host buffers through brov_rollout_host: every call copies its chunk of inputs host->device from
                    pinned memory and the final state back (PCIe-bound); e2e.generated: ONE call runs the whole
                    10,000-step job of configs[1] with generated inputs, only x0 / lag / generator state cross PCIe.
`roofline` nests the other BASELINE configs so that the driver's record keeps them: fp32 (configs[2], 1,048,576
vehicles, stride-10 writeback), monte_carlo (configs[3]), rmse (configs[4], NCCL all-reduce for N > 1, both lag
semantics), default_api (per-thruster lag states returned, the drop-in default).  N > 1: the ensemble is sharded by
vehicle, each rank runs its own shard (weak scaling, no data-path collective).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
# version banner there on every rank), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a saved
# copy of the original stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


METRIC = "rk4_vehicle_steps_per_s"
UNIT = "vehicle-steps/s"
DT = 0.02
SEED = 1
FLOP_PER_STEP = {"thruster8": 1756.0, "wrench12": 676.0, "quat13": 805.0}   # SURVEY 8(d), algorithmic
NOMINAL_TFLOPS = {"f64": 37.2, "f32": 74.4}       # 148 SMs x 64 (128) FMA lanes x 2 x 1.965 GHz (SURVEY 8d)
# executed-instruction evidence from the committed ncu captures (profiles/README.md): share of cycles the FP pipe is busy
PIPE_ACTIVE = {"rollout_f64": {"value": 0.715, "capture": "profiles/r02af_rollout_raw.csv (sm__pipe_fp64_cycles_active, % of peak sustained active; 0.694 of elapsed)"},
               "rollout_f32": {"value": 0.72, "capture": "profiles/r01j_rollout_f32_raw.csv"}}
CFG2 = dict(name="cfg2", model="thruster8", dtype="f64", n_per_gpu=65536, stride=0, chunk=1000, ring=10)
CFG3 = dict(name="cfg3", model="thruster8", dtype="f32", n_per_gpu=1 << 20, stride=10, chunk=100, ring=8)


def cfg_x0(n: int, rank: int) -> np.ndarray:
    """Initial states of SURVEY 8(d) cfg2: positions in a tank-sized box, small roll / pitch, any yaw, at rest.  Host
    numpy so that the GPU arm and the reference arm start the same vehicles from the same states."""
    rng = np.random.default_rng(1000 + rank)
    x = np.zeros((n, 12))
    x[:, 0:2] = rng.uniform(-2, 2, (n, 2))
    x[:, 2] = rng.uniform(0, 3, n)
    x[:, 3:5] = rng.uniform(-0.2, 0.2, (n, 2))
    x[:, 5] = rng.uniform(-np.pi, np.pi, n)
    return x


# ------------------------------------------------------------------------------------------------------------------
# CPU legs: the reference itself (oracle/_ref, byte-compiled from /root/reference) or, where that is absent, the numpy
# port — the only place bench.py may execute oracle/
# ------------------------------------------------------------------------------------------------------------------
def _cpu_worker(job):
    """One host core: its vehicles one at a time through the reference's own simulate_physics
    (training/train_tank_brov2_rk4.py:375-396) with a fresh BlueROV2 per vehicle."""
    os.environ["OMP_NUM_THREADS"] = "1"
    x0, U, use_ref = job
    t0 = time.perf_counter()
    if use_ref:
        import warnings
        warnings.filterwarnings("ignore")
        from oracle import ref_loader
        R = ref_loader.load()
        for i in range(x0.shape[0]):
            R.simulate_physics(x0[i], U[:, i], DT, R.BlueROV2(dt=DT))
    else:
        from oracle import fossen_np as O
        m = O.Model("thruster8", DT)
        for i in range(x0.shape[0]):
            O.rollout(m, "rk4", x0[i:i + 1], U[:, i])
    return time.perf_counter() - t0


def reference_inputs(n_vehicles: int, steps: int):
    """x0 and the command signal of the FIRST n_vehicles vehicles of rank 0's configs[1] ensemble — the very numbers the
    GPU arm integrates — for `steps` steps.  The signal comes out of the engine's generator when a GPU and libbrov are
    there (bit-identical), else out of its numpy restatement (same Philox stream, transcendental rounding differs)."""
    x0 = cfg_x0(CFG2["n_per_gpu"], 0)[:n_vehicles]
    try:
        import torch
        import bluerov2_dynamics_b200 as B
        assert torch.cuda.is_available()
        e = B.Engine("thruster8", "f64", device=0)
        U = e.generate_inputs(B.InputGenerator(seed=SEED), steps=steps, n_sel=n_vehicles)[0].cpu().numpy()
        how = "engine generator (bit-identical to the GPU arm's inputs)"
        del e
    except Exception:
        from oracle import inputgen_np as G
        U = G.command_signal(SEED, np.arange(n_vehicles), 0, steps)[0]
        how = "numpy restatement of the generator (same stream, ~1e-6 apart)"
    return x0, np.ascontiguousarray(U), how


def cpu_reference_rate(cores: int, steps_per_vehicle: int, x0=None, U=None):
    """Aggregate RK4 vehicle-steps/s of `cores` processes, each rolling ONE vehicle for steps_per_vehicle steps."""
    import multiprocessing as mp
    from oracle import ref_loader
    use_ref = ref_loader.available()
    if use_ref:
        import warnings
        warnings.filterwarnings("ignore")
        ref_loader.load()      # in the parent, so that the forked workers time the rollouts, not the imports
    how = None
    if x0 is None:
        x0, U, how = reference_inputs(cores, steps_per_vehicle)
    jobs = [(x0[i:i + 1], U[:, i:i + 1], use_ref) for i in range(cores)]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    return cores * steps_per_vehicle / wall, wall, ("reference" if use_ref else "port"), how


def cpu_c_oracle_rate(n: int = 8192, steps: int = 400):
    """The plain-C oracle (oracle/brov_oracle.c: scalar float64, reference operation structure, OpenMP over vehicles)
    on all host cores: the strongest CPU baseline — compiled code instead of the reference's Python."""
    from oracle import c_oracle as CO
    if not CO.available():
        return None, 0
    rng = np.random.default_rng(2)
    x = np.zeros((n, 12))
    x[:, 2] = 1.0
    U = rng.uniform(-0.4, 0.4, (steps, n, 8))
    CO.rollout("thruster8", "rk4", DT, x[:64], U[:10, :64])
    t0 = time.perf_counter()
    CO.rollout("thruster8", "rk4", DT, x, U)
    return n * steps / (time.perf_counter() - t0), CO.threads()


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline_block(cores: int, cpu_steps: int) -> dict:
    rate, wall, kind, how = cpu_reference_rate(cores, cpu_steps)
    what = ("the UNMODIFIED reference (oracle/_ref: fossen.BlueROV2 + training/train_tank_brov2_rk4.simulate_physics)"
            if kind == "reference" else "numpy port of the reference (oracle/fossen_np.py), one vehicle per Python call")
    cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": f"{cores} processes x 1 vehicle x {cpu_steps} RK4 steps: the first {cores} vehicles of rank 0's configs[1] "
                     f"ensemble, same x0 and commands ({how}); {what}; wall {wall:.1f} s",
           "same_config": f"same model, dt, x0 and command stream as the GPU arm; a subset of {cores} vehicles x {cpu_steps} steps"}
    c_rate, c_thr = cpu_c_oracle_rate()
    if c_rate is not None:
        cpu["c_port_value"] = c_rate
        cpu["c_port_threads"] = c_thr
        cpu["c_port_sample"] = "oracle/brov_oracle.c (scalar float64 C restatement, OpenMP over vehicles): 8192 vehicles x 400 RK4 steps"
    return cpu


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, windows):
        """windows: list of (t0, t1) perf_counter intervals that were timed."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if windows and not any(a - 0.05 <= t <= b + 0.15 for a, b in windows):
                continue
            f = [s.strip() for s in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def dump_outputs(path: str, arrays: dict) -> None:
    """Writes the headline leg's final results as <path>/<name>.npy in float64 (rank 0's shard: 65,536 vehicles,
    xT [N,12] and the allocation-projected lag [N,18], 15.7 MB).  x0 and the command stream are seeded, so two builds
    run with the same arguments can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.double().cpu().numpy())


def timed(torch, dist, world, dev, fn, warmup, steps, windows):
    """W untimed calls, then K timed ones between CUDA events on the launching stream, barrier + synchronize on both
    sides, max over ranks."""
    for k in range(warmup):
        fn(k)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for k in range(steps):
        fn(warmup + k)
    e1.record()
    torch.cuda.synchronize()
    windows.append((t0, time.perf_counter()))
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    return ms


def run_rollout_legs(torch, dist, B, cfg, steps, warmup, rank, local, world, windows, default_api=False):
    """Streamed-input leg (inputs resident in HBM as `ring` distinct chunks of the generated signal), generated-input leg
    and — fp64 only — the default-API leg (per-thruster lag states returned) on one ensemble."""
    eng = B.Engine(cfg["model"], cfg["dtype"], device=local)
    n, stride, chunk, ring = cfg["n_per_gpu"], cfg["stride"], cfg["chunk"], cfg["ring"]
    gen = B.InputGenerator(seed=SEED, vehicle0=rank * n)
    x0 = eng.tensor(cfg_x0(n, rank))
    ring = min(ring, max(2, warmup + steps))
    # the command signal of steps [0, ring*chunk) materialised by the engine's own generator: the streamed leg reads
    # the numbers the generated leg computes
    U, gs = [], None
    for r in range(ring):
        u, gs = eng.generate_inputs(gen, steps=chunk, step0=r * chunk, n_sel=n, state_in=gs)
        U.append(u)
    out = {"n": n, "eng": eng, "x0": x0, "U": U, "gen": gen, "chunk": chunk}

    def fresh():
        x = x0.clone()
        lag = torch.zeros((n, 18), device=eng.device, dtype=eng.tdtype)   # allocation-projected lag carried between chunks
        return x, lag

    traj = [torch.empty((chunk // stride, n, 12), device=eng.device, dtype=eng.tdtype) for _ in range(2)] if stride else None
    # --- streamed
    x, lag = fresh()
    ms = timed(torch, dist, world, eng.device,
               lambda k: eng.rollout(x, U[k % ring], dt=DT, integrator="rk4", lag0=lag, stride=stride, step0=k * chunk,
                                     xT_out=x, lag_out=lag, traj_out=traj[k % 2] if stride else None, lag_repr="projected"),
               warmup, steps, windows)
    out["streamed"] = dict(ms_total=ms, ms_per_step=ms / steps, finite=bool(torch.isfinite(x).all().item()))
    out["outputs"] = {"xT": x, "lag": lag}     # what the last timed call returned (it writes in place)
    # --- generated in the kernel: every step of every launch is a distinct step of the stream
    x, lag = fresh()
    gst = torch.zeros((n, 8), device=eng.device, dtype=eng.tdtype)
    hc = []

    def one_gen(k):
        r = eng.rollout(x, gen=gen, steps=chunk, step0=k * chunk, dt=DT, integrator="rk4", lag0=lag, stride=stride,
                        xT_out=x, lag_out=lag, traj_out=traj[k % 2] if stride else None, lag_repr="projected", gen_state=gst,
                        gen_state_out=gst, health=True)
        hc.append(r.health)
    ms = timed(torch, dist, world, eng.device, one_gen, warmup, steps, windows)
    out["generated"] = dict(ms_total=ms, ms_per_step=ms / steps, finite=bool(torch.isfinite(x).all().item()),
                            health=[int(v) for v in hc[-1].tolist()], distinct_steps=(warmup + steps) * chunk)
    # --- the drop-in default: per-thruster lag states [N,8,3] in and out (lag epilogue after the kernel)
    if default_api:
        x = x0.clone()
        lag24 = torch.zeros((n, 24), device=eng.device, dtype=eng.tdtype)
        ms = timed(torch, dist, world, eng.device,
                   lambda k: eng.rollout(x, U[k % ring], dt=DT, integrator="rk4", lag0=lag24, step0=k * chunk, xT_out=x,
                                         lag_out=lag24),
                   warmup, steps, windows)
        out["default_api"] = dict(ms_total=ms, ms_per_step=ms / steps)
    sz = 8 if cfg["dtype"] == "f64" else 4
    out["bytes_per_launch"] = n * chunk * 8 * sz + (n * 12 * sz * (chunk // stride) if stride else 0) + 2 * n * 30 * sz
    out["bytes_per_launch_generated"] = (n * 12 * sz * (chunk // stride) if stride else 0) + 2 * n * 38 * sz
    return out


def run_e2e_legs(torch, dist, B, cfg, leg, steps, warmup, world, windows):
    """The same workload through the host-buffer API (brov_rollout_host).  Host-streamed: per call the chunk's inputs +
    x0 + lag go host->device from pinned memory and the final state + lag come back.  Generated: only x0 / lag /
    generator state cross PCIe."""
    eng, n, gen = leg["eng"], leg["n"], leg["gen"]
    chunk = 250   # 1.07 GB of inputs per call from pinned memory (keeps 8 ranks' pinned pools small)
    ring = 2
    Uh = [B.pinned_empty((chunk, n, 8), eng.ndtype) for _ in range(ring)]
    for r in range(ring):
        Uh[r][...] = leg["U"][0][r * chunk:(r + 1) * chunk].cpu().numpy()
    xh = B.pinned_empty((n, 12), eng.ndtype)
    lagh = B.pinned_empty((n, 18), eng.ndtype)
    gsh = B.pinned_empty((n, 8), eng.ndtype)

    def reset():
        xh[...] = leg["x0"].cpu().numpy()
        lagh[...] = 0
        gsh[...] = 0

    def wall(fn, k_steps):
        for k in range(max(1, min(warmup, 3))):
            fn(k)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for k in range(k_steps):
            fn(k)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        windows.append((t0, t1))
        sec = t1 - t0
        if world > 1:
            t = torch.tensor([sec], device=eng.device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return sec

    reset()
    sec = wall(lambda k: eng.rollout_host(xh, Uh[k % ring], dt=DT, integrator="rk4", lag0=lagh, out_xT=xh, out_lag=lagh,
                                          chunk_steps=25, lag_repr="projected"), steps)
    h2d = Uh[0].nbytes + xh.nbytes + lagh.nbytes
    d2h = xh.nbytes + lagh.nbytes
    e2e = dict(value=float(n) * world * chunk * steps / sec, unit=UNIT, h2d_bytes_per_step=int(h2d),
               d2h_bytes_per_step=int(d2h), steps=steps, ms_per_step=1e3 * sec / steps, h2d_gbs=h2d * steps / sec / 1e9,
               rk4_steps_per_call=chunk,
               api="Engine.rollout_host -> brov_rollout_host (C ABI), pinned host buffers, 250 RK4 steps per call in 10 "
                   "sub-chunks double-buffered on a copy stream")
    reset()
    # ONE call = the whole job of configs[1]: 10,000 RK4 steps of every vehicle (one launch, the library's default for
    # generated commands); x0 / lag / generator state go up once per call and come back once
    gchunk = 10 * leg["chunk"]
    health = np.zeros(2, np.uint64)
    sec = wall(lambda k: eng.rollout_host(xh, gen=gen, steps=gchunk, dt=DT, integrator="rk4", lag0=lagh, out_xT=xh,
                                          out_lag=lagh, lag_repr="projected", gen_state=gsh, out_gen_state=gsh, health=health),
               steps)
    h2d = xh.nbytes + lagh.nbytes + gsh.nbytes
    e2e["generated"] = dict(value=float(n) * world * gchunk * steps / sec, unit=UNIT, h2d_bytes_per_step=int(h2d),
                            d2h_bytes_per_step=int(h2d + 16), steps=steps, ms_per_step=1e3 * sec / steps,
                            rk4_steps_per_call=gchunk, health=[int(v) for v in health],
                            api="the same call with gen=InputGenerator(seed): commands generated in the kernel, host "
                                "buffers hold x0 / lag / generator state and the results")
    return e2e


def tank_series(torch, dev, T):
    """configs[4]: a synthetic tank-shaped 50 Hz series: smooth bounded motion in a tank-sized box plus sensor-like noise."""
    g = torch.Generator(device=dev).manual_seed(4)
    U = (torch.rand((T, 8), device=dev, dtype=torch.float64, generator=g) * 0.8 - 0.4)
    t = torch.arange(T, device=dev, dtype=torch.float64) * DT
    X = torch.zeros((T, 12), device=dev, dtype=torch.float64)
    X[:, 0] = 2.0 * torch.sin(0.05 * t); X[:, 1] = 2.0 * torch.cos(0.04 * t); X[:, 2] = 1.5 + torch.sin(0.03 * t)
    X[:, 5] = 0.5 * torch.sin(0.02 * t)
    X[:, 6] = 0.1 * torch.cos(0.05 * t); X[:, 7] = -0.08 * torch.sin(0.04 * t); X[:, 8] = 0.03 * torch.cos(0.03 * t)
    X += 1e-3 * torch.randn((T, 12), device=dev, dtype=torch.float64, generator=g)
    return X, U


def run_rmse_leg(torch, dist, B, local, rank, world, windows, fp64_peak, T=1_000_100, horizons=(1, 10, 100)):
    """configs[4]: multi-horizon endpoint RMSE over ~1M sliding windows of one series; windows sharded over ranks (halo
    rows replicated), kernels + NCCL all-reduce captured in one CUDA graph per evaluator.  `reset`: every window from
    zero lag, all horizons in one pass.  `carry`: the drop-in default — the reference's literal semantics, lag state
    handed from window to window — one pass per horizon."""
    from bluerov2_dynamics_b200 import dist as D
    eng = B.Engine("thruster8", "f64", device=local)
    X, U = tank_series(torch, eng.device, T)
    hs = list(horizons)
    out = {"workload": f"configs[4]: T={T} rows, H={hs}, RK4, 8-thruster fp64, windows sharded over {world} GPU(s)"
                       + (", NCCL all-reduce of the SE vector inside the captured graph" if world > 1 else ""),
           "windows": D.global_counts(T, hs)}

    def time_ev(evs, reps=5):
        for _ in range(2):
            for ev in evs:
                ev.run()
        ms = timed(torch, dist, world, eng.device, lambda k: [ev.run() for ev in evs], 1, reps, windows) / reps
        return ms

    ev = D.ShardedEvaluator(eng, X, U, hs, DT, "rk4", rank, world, lag_mode="reset")
    ms = time_ev([ev])
    hm = hs[-1]
    vsteps = float(max(T - hm, 0) * hm + hm * (hm - 1) // 2)        # all horizons are read off ONE rollout per window
    r, hc = ev.rmse()
    tf = vsteps / world / (ms * 1e-3) * FLOP_PER_STEP["thruster8"] / 1e12
    out["reset"] = {"ms": ms, "vehicle_steps_per_s": vsteps / (ms * 1e-3), "rmse": r, "health": hc,
                    "graph": ev.graph is not None, "frac": tf / fp64_peak, "achieved_tflops_per_gpu": tf}
    evc = D.ShardedEvaluator(eng, X, U, hs, DT, "rk4", rank, world, lag_mode="carry")
    ms_c = time_ev([evc])
    vsteps_c = float(sum((T - h) * h for h in hs))
    out["carry"] = {"ms": ms_c, "vehicle_steps_per_s": vsteps_c / (ms_c * 1e-3), "rmse": evc.rmse()[0],
                    "graph": evc.graph is not None,
                    "note": "one pass per horizon (111 instead of 100 steps per window), the three passes concurrent on forked "
                            "streams inside one graph; each thread scores several consecutive windows and replays the "
                            "~49-step lag history once per group", "cost_over_reset": ms_c / ms}
    out["kernel"] = "brov::se_kernel<double, THRUSTER8, RK4> + se_finish_kernel" + (" + ncclAllReduce (graph)" if world > 1 else "")
    return out


def run_reduced9_leg(torch, B, local, peaks, peak_src, windows, rows=1 << 24, traffic=None):
    """bluerov_compute (fossen/bluerov_torch.py:20-67) batched over `rows` states: 13 scalars in, 9 out per row —
    38 FLOP per 88 B in fp32, HBM-bound.  Two input/output sets (1.48 GB each, far larger than L2) used alternately."""
    dev = torch.device("cuda", local)
    g = torch.Generator(device=dev).manual_seed(9)
    X = [torch.randn((rows, 9), device=dev, dtype=torch.float32, generator=g) for _ in range(2)]
    U = [torch.randn((rows, 4), device=dev, dtype=torch.float32, generator=g) for _ in range(2)]
    O = [torch.empty((rows, 9), device=dev, dtype=torch.float32) for _ in range(2)]
    for k in range(3):
        B.reduced9_rhs(X[k % 2], U[k % 2], out=O[k % 2])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    t0 = time.perf_counter()
    e0.record()
    for k in range(n):
        B.reduced9_rhs(X[k % 2], U[k % 2], out=O[k % 2])
    e1.record()
    torch.cuda.synchronize()
    windows.append((t0, time.perf_counter()))
    ms = e0.elapsed_time(e1) / n
    nbytes = rows * (9 + 4 + 9) * 4
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"workload": f"bluerov_compute RHS, {rows} rows fp32, 88 B algorithmic per row", "ms": ms,
            "evals_per_s": rows / (ms * 1e-3), "launches": n,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm_gbs"], "traffic": (traffic or {}).get("bytes"),
                         "traffic_source": (traffic or {}).get("capture"), "kernel": "brov::reduced9_kernel<float>",
                         "bytes_per_launch": nbytes, "peak_source": peak_src}}


def run_compare_leg(torch, B, local, windows, fp32_peak, fp64_peak, T=1_000_100, horizons=(1, 10, 100), cpu=True):
    """The reference's model-comparison table (training/train_tank_brov2_full_comparison.py:977-1009: endpoint RMSE at
    H = 1/10/100 of the Fossen, Koopman, double-integrator and PINc models) on one synthetic 50 Hz series of T rows:
    device time of each evaluator, and the oracle timed on a bounded prefix of the same series on the host cores."""
    from bluerov2_dynamics_b200.Koopman.koopmanEDMDc import KoopmanEDMDc
    from bluerov2_dynamics_b200 import pinc as P
    dev = torch.device("cuda", local)
    X, U = tank_series(torch, dev, T)
    g = torch.Generator(device=dev).manual_seed(5)
    hs = list(horizons)
    rng = np.random.default_rng(12)
    out = {"workload": f"comparison table: endpoint RMSE at H={hs} over all windows of a {T}-row synthetic series",
           "models": {}}

    def tm(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(reps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        windows.append((t0, time.perf_counter()))
        return e0.elapsed_time(e1) / reps, r

    nwin = [T - h for h in hs]
    steps_all = float(sum((T - h) * h for h in hs))
    e = B.Engine("di12_u8", "f64", device=local)
    K_lin, K_ang = rng.normal(0, 0.05, (8, 3)), rng.normal(0, 0.05, (8, 3))
    e.set_di_gains(K_lin, K_ang)
    ms, _ = tm(lambda: e.multistep_se(X, U, hs, dt=DT, integrator="rk4")[0])
    out["models"]["double_integrator_rk4_f64"] = {"ms": ms, "windows": nwin, "kernel": "brov::se_kernel<double, DI12_U8, RK4>"}
    k = 500
    Kc = X[torch.randint(0, T, (k,), device=dev, generator=g)].cpu().numpy()
    A = 0.98 * np.linalg.qr(rng.standard_normal((12 + k, 12 + k)))[0]
    Bm = 0.02 * rng.standard_normal((12 + k, 8))
    KM = KoopmanEDMDc(state_dim=12, input_dim=8, n_rbfs=k, gamma=3.0)
    KM.centers_, KM.A_, KM.B_ = Kc, A, Bm
    h_k = KM._handle()
    from bluerov2_dynamics_b200 import _lib as L
    arr_h = (__import__("ctypes").c_int * len(hs))(*hs)
    se_k = torch.zeros(len(hs), device=dev, dtype=torch.float64)

    def koop_all():   # all horizons from ONE lift pass (brov_koopman_multistep_se_multi)
        L.check(L.lib.brov_koopman_multistep_se_multi(h_k, X.data_ptr(), U.data_ptr(), T, len(hs), arr_h, se_k.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream))
        return se_k
    ms, _ = tm(koop_all)
    flop_k = (T - hs[0]) * k * 26.0 + sum((T - h) * (2.0 * 12 * (12 + k) + 2.0 * 12 * 8 * h) for h in hs)
    out["models"]["koopman_d512_f64"] = {
        "ms": ms, "windows": nwin, "kernel": "koop_liftw_kernel<12, 3> + koop_fir_se_kernel<12, 8>",
        "algorithmic_tflops": flop_k / (ms * 1e-3) / 1e12, "frac_fp64_pipe": flop_k / (ms * 1e-3) / 1e12 / fp64_peak,
        "note": "decoder-row formulation: 2 n (d + r H) + lift flop per window instead of the reference's 2 d^2 H"}
    cg = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors_cmp.npz"))
    PM = P.PincModel({kk[len("pinc_sd_"):]: cg[kk] for kk in cg.files if kk.startswith("pinc_sd_")}, device=local)
    ms, _ = tm(lambda: PM.multistep_se(X, U, hs, DT, "reset")[0], reps=2)
    hm = hs[-1]
    steps_p = float((T - hm) * hm + hm * (hm - 1) // 2)
    flop_p = steps_p * 2.0 * (14 * 64 + 3 * 64 * 64 + 64 * 9)
    out["models"]["pinc_f32"] = {"ms": ms, "windows": nwin, "kernel": "pinc_se_tc_kernel (tcgen05.mma kind::tf32 + kind::f16, split operands, 3 tiles per SM)", "network_steps": steps_p,
                                 "algorithmic_tflops": flop_p / (ms * 1e-3) / 1e12,
                                 "vs_fp32_vector_peak": flop_p / (ms * 1e-3) / 1e12 / fp32_peak,
                                 "bound": "epilogue (2 MUFU per activation + issue slots), not the tensor pipe",
                                 "pipes": {"tensor_active": 0.23, "xu_active": 0.43, "issue_active": 0.46,
                                           "capture": "profiles/r02v_pinc_tc_raw.csv"},
                                 "note": "the dense layers run on the tensor cores (3 split products per layer: 2 x kind::tf32 "
                                         "+ 1 x kind::f16, fp32 accumulation in TMEM), so the algorithmic rate exceeds the "
                                         "FP32 vector peak the CUDA-core kernel (79 ms) was bound by"}
    if cpu:
        from oracle import compare_np as CN
        Tc = 2100
        Xc, Uc = X[:Tc].cpu().numpy(), U[:Tc].cpu().numpy()
        t0 = time.perf_counter(); CN.di_multistep_se("di12", "rk4", Xc, Uc, hs, DT, K_lin, K_ang); t_di = time.perf_counter() - t0
        t0 = time.perf_counter()
        for h in hs:
            CN.koop_multistep_se(Xc, Uc, h, Kc, 3.0, A, Bm)
        t_k = time.perf_counter() - t0
        layers = CN.pinc_weights(cg)
        t0 = time.perf_counter(); CN.pinc_multistep_se(Xc, Uc, hs, DT, layers, "reset"); t_p = time.perf_counter() - t0
        scale = steps_all / float(sum((Tc - h) * h for h in hs))
        out["cpu_oracle"] = {"rows": Tc, "kind": "port", "double_integrator_s": t_di, "koopman_s": t_k, "pinc_s": t_p,
                             "extrapolated_s": {"double_integrator": t_di * scale, "koopman": t_k * scale, "pinc": t_p * scale}}
    return out


def run_monte_carlo_leg(torch, B, local, fp32_peak, windows, n=1 << 20, steps=5, chunk=100):
    """BASELINE configs[3]: Monte-Carlo sweep — per-vehicle added-mass / damping coefficients (table [36][N], held in
    registers for the launch) with wrench input and the first-order wrench lag, fp32, 100 RK4 steps per launch."""
    e = B.Engine("wrench12", "f32", device=local)
    rng = np.random.default_rng(3)
    ph = np.tile(B.default_physical(), (n, 1))
    ph[:, 9:27] *= rng.uniform(0.7, 1.3, (n, 18))
    ph[:, 27:30] = 1.0 / (ph[:, 0:1] - ph[:, 9:12])
    ph[:, 30:33] = 1.0 / (ph[:, 6:9] - ph[:, 12:15])
    ph[:, 36] = rng.uniform(0.05, 0.3, n)
    e.set_wrench_lag1(True)
    e.set_vehicle_physical(ph)
    gen = B.InputGenerator(seed=33, scale=[40, 40, 40, 5, 5, 5.0])
    U = [e.generate_inputs(gen, steps=chunk, step0=r * chunk, n_sel=n)[0] for r in range(2)]
    x = torch.zeros((n, 12), device=e.device, dtype=torch.float32)
    lag = torch.zeros((n, 6), device=e.device, dtype=torch.float32)

    def one(k):
        e.rollout(x, U[k % 2], dt=DT, integrator="rk4", lag0=lag, xT_out=x, lag_out=lag, step0=k * chunk)
    for k in range(3):
        one(k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for k in range(steps):
        one(3 + k)
    e1.record()
    torch.cuda.synchronize()
    windows.append((t0, time.perf_counter()))
    ms = e0.elapsed_time(e1) / steps
    rate = n * chunk / (ms * 1e-3)
    flop = FLOP_PER_STEP["wrench12"] + 4 * 12.0     # + first-order lag: 12 flop per RHS evaluation (SURVEY 8d)
    return {"workload": f"configs[3]: {n} vehicles, per-vehicle coefficients + first-order wrench lag, wrench-input "
                        "12-state model, fp32, 100 RK4 steps per launch", "ms": ms, "value": rate, "unit": UNIT,
            "finite": bool(torch.isfinite(x).all().item()), "achieved_tflops": rate * flop / 1e12,
            "frac": rate * flop / 1e12 / fp32_peak, "flop_per_vehicle_step": flop,
            "kernel": "brov::rollout_kernel<float, WRENCH12, RK4, lag1, per-vehicle>"}


def main_ours(args):
    import torch
    import torch.distributed as dist
    import bluerov2_dynamics_b200 as B
    from bluerov2_dynamics_b200 import dist as D

    rank, world, local = D.init_from_env()
    if world != args.gpus and rank == 0:
        print(f"[bench] note: WORLD_SIZE={world} but --gpus {args.gpus}; using {world}", file=sys.stderr)
    torch.cuda.set_device(local)
    cores = host_cores()

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_baseline_block(cores, args.cpu_steps)      # before the timed GPU regions; forked workers never touch CUDA
    if world > 1:
        dist.barrier()

    sampler = ClockSampler(local) if rank == 0 else None
    windows = []
    peaks, peak_src = measured_peaks()
    fp64_peak, _ = B.fma_peak("f64", local, 2048)     # in-run FP pipe peaks (MEASURED_PEAKS.json has HBM and bf16 GEMM only)
    fp32_peak, _ = B.fma_peak("f32", local, 8192)

    leg2 = run_rollout_legs(torch, dist, B, CFG2, args.steps, args.warmup, rank, local, world, windows, default_api=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, leg2["outputs"])
    e2e = run_e2e_legs(torch, dist, B, CFG2, leg2, min(args.steps, args.e2e_steps), args.warmup, world, windows)
    for k in ("U", "x0", "eng", "gen", "outputs"):
        leg2.pop(k)
    torch.cuda.empty_cache()
    leg3 = run_rollout_legs(torch, dist, B, CFG3, args.steps, args.warmup, rank, local, world, windows)
    for k in ("U", "x0", "eng", "gen", "outputs"):
        leg3.pop(k)
    torch.cuda.empty_cache()
    rmse = run_rmse_leg(torch, dist, B, local, rank, world, windows, fp64_peak) if not args.no_rmse else None
    mc = run_monte_carlo_leg(torch, B, local, fp32_peak, windows) if rank == 0 and not args.no_compare else None
    compare = (run_compare_leg(torch, B, local, windows, fp32_peak, fp64_peak, cpu=not args.no_cpu_baseline)
               if rank == 0 and not args.no_compare else None)
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except OSError:
        traffic = {}
    red9 = run_reduced9_leg(torch, B, local, peaks, peak_src, windows, traffic=traffic.get("reduced9_f32")) if rank == 0 else None

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    clocks = sampler.stop(windows)

    def rate(leg, which, cfg):
        return leg["n"] * world * cfg["chunk"] * args.steps / (leg[which]["ms_total"] * 1e-3)

    def roof(leg, cfg, peak, which="streamed"):
        per_gpu = rate(leg, which, cfg) / world
        tf = FLOP_PER_STEP[cfg["model"]] * per_gpu / 1e12
        nb = leg["bytes_per_launch" if which == "streamed" else "bytes_per_launch_generated"]
        gbs = nb / (leg[which]["ms_per_step"] * 1e-3) / 1e9
        return {"value": rate(leg, which, cfg), "ms_per_step": leg[which]["ms_per_step"], "achieved": tf, "frac": tf / peak,
                "frac_nominal": tf / NOMINAL_TFLOPS[cfg["dtype"]],
                "hbm": {"achieved": gbs, "frac": gbs / peaks["hbm_gbs"], "bytes_per_launch": nb}}

    v2 = rate(leg2, "streamed", CFG2)
    r2 = roof(leg2, CFG2, fp64_peak)
    tr = traffic.get("rollout_f64", {})
    roofline = {
        "bound": "fp64_pipe", "achieved": r2["achieved"], "peak": fp64_peak, "unit": "TFLOP/s", "frac": r2["frac"],
        "traffic": tr.get("bytes"), "traffic_source": tr.get("capture"),
        "kernel": "brov::rollout_kernel<double, THRUSTER8, RK4>", "flop_per_vehicle_step": FLOP_PER_STEP["thruster8"],
        "peak_source": "in-run FMA-chain microbenchmark (brov_fma_peak), 2 flop per FMA; MEASURED_PEAKS.json has no FP64 vector peak",
        "peak_nominal": NOMINAL_TFLOPS["f64"], "frac_nominal": r2["frac_nominal"],
        "pipe_active": PIPE_ACTIVE["rollout_f64"],
        "note": "frac = ALGORITHMIC flop (SURVEY 8d: 1756 per RK4 vehicle-step) / time / peak; the kernel executes fewer FP64 "
                "instructions than that (projected lag, angle-addition trig), so frac is not pipe utilisation: pipe_active is",
        "kernel_ms": leg2["streamed"]["ms_per_step"], "hbm": dict(r2["hbm"], peak=peaks["hbm_gbs"], unit="GB/s", peak_source=peak_src),
        "generated": dict(roof(leg2, CFG2, fp64_peak, "generated"), health=leg2["generated"]["health"],
                          distinct_steps=leg2["generated"]["distinct_steps"],
                          note="commands generated in the kernel (Philox4x32-10 + Box-Muller, interleaved with the RK4 stages)"),
        "default_api": {"value": rate(leg2, "default_api", CFG2), "ms_per_step": leg2["default_api"]["ms_per_step"],
                        "vs_value": rate(leg2, "default_api", CFG2) / v2,
                        "note": "Engine.rollout defaults (per-thruster lag states in and out): same kernel + lag epilogue"},
        "fp32": dict(roof(leg3, CFG3, fp32_peak), dtype="f32", peak=fp32_peak, peak_nominal=NOMINAL_TFLOPS["f32"],
                     pipe_active=PIPE_ACTIVE["rollout_f32"],
                     workload="BASELINE configs[2]: 1,048,576 vehicles per GPU, fp32, 100 RK4 steps per launch, trajectory "
                              "writeback every 10 steps; inputs: 8 distinct 3.36 GB chunks resident in HBM",
                     generated=roof(leg3, CFG3, fp32_peak, "generated"), kernel="brov::rollout_kernel<float, THRUSTER8, RK4>",
                     finite=leg3["streamed"]["finite"] and leg3["generated"]["finite"]),
        "monte_carlo": mc, "rmse": rmse,
    }
    line = {
        "metric": METRIC, "value": v2, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": leg2["streamed"]["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: 65,536-vehicle ensemble per GPU, 8-thruster Fossen model with 3rd-order "
                               "thruster lag, per-vehicle smooth random thrust commands u = clip(0.98 u + 0.02 N(0,1), -1, 1), "
                               f"RK4, dt=0.02, {args.steps * CFG2['chunk']} steps ({CFG2['chunk']} per launch), fp64",
                   "vehicles_per_gpu": CFG2["n_per_gpu"], "rk4_steps_per_launch": CFG2["chunk"],
                   "l2_policy": "inputs larger than L2: 10 distinct 4.19 GB input chunks (10,000 distinct steps) resident in "
                                "HBM, each read once per launch",
                   "parallelism": f"vehicle-sharded x{world}, no data-path collective"},
        "roofline": roofline, "e2e": e2e, "gpu_launches": args.steps, "clocks": clocks,
        "finite": leg2["streamed"]["finite"] and leg2["generated"]["finite"],
        "reduced9": red9, "comparison_models": compare,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main_reference(args):
    """Reference arm: the reference's own CPU implementation of the path — fossen.BlueROV2 driven by
    training/train_tank_brov2_rk4.simulate_physics, executed from oracle/_ref (the unmodified reference, byte-compiled;
    the numpy port only where that is absent) — on all host cores.  Each step is a bounded sample of the GPU arm's
    workload: the first `cores` vehicles of rank 0's configs[1] ensemble, same x0 and command stream."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    spc = args.cpu_steps
    x0, U, how = reference_inputs(cores, spc)
    for _ in range(min(args.warmup, 1)):
        cpu_reference_rate(cores, max(spc // 8, 10), x0, U[:max(spc // 8, 10)])
    t0 = time.perf_counter()
    steps_done, kind = 0, "port"
    for k in range(args.steps):
        _, _, kind, _ = cpu_reference_rate(cores, spc, x0, U)
        steps_done += 1
        if time.perf_counter() - t0 > args.reference_budget_s:
            break
    wall = time.perf_counter() - t0
    value = cores * spc * steps_done / wall
    what = ("the UNMODIFIED reference executed from oracle/_ref" if kind == "reference" else "numpy port (oracle/_ref absent)")
    sample = (f"each step: {cores} processes x 1 vehicle x {spc} RK4 steps of configs[1] — the first {cores} vehicles of the GPU "
              f"arm's rank-0 ensemble, same x0 and commands ({how}) — {what}: simulate_physics "
              f"(training/train_tank_brov2_rk4.py:375-396) on fossen.BlueROV2; {steps_done} of {args.steps} steps within the "
              f"{args.reference_budget_s:.0f} s budget")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps_done, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * wall / max(steps_done, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BASELINE configs[1] model, x0 and command stream; bounded sample on the host CPU cores",
                       "vehicles": cores, "rk4_steps_per_vehicle": spc},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-steps", type=int, default=1000,
                    help="RK4 steps per core of the CPU baseline sample (1000 = about 2 s per vehicle of the real reference)")
    ap.add_argument("--reference-budget-s", type=float, default=120.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-rmse", action="store_true")
    ap.add_argument("--no-compare", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the final state and lag of the headline leg's last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs saves the CUDA engine's results; the reference arm has none to save")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
