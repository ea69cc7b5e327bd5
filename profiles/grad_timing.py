"""Exact coefficient gradient (brov_multistep_se_grad) against the evaluator and the central-difference sweep, on a GPU.

    python profiles/grad_timing.py [--out DIR] [--quick]

Series: the length of the reference's tank recording (45,823 rows) and the 1,000,100-row series of bench.py's evaluator
config; thruster8 fp64 RK4, H = 1/10/100, reset (one pass for the three horizons) and carried lag (one pass per
horizon).  For p in {1, 6, 18, 36} directions (K = 1: one direction per thread, the only build):
  grad     one Engine.multistep_se_grad call (se, gradient and Gauss-Newton matrix of the three horizons);
  single   one Engine.multistep_se call (default time slicing) — the cost of the objective alone;
  cd       one Engine.multistep_se_sweep call over the 2p+1 candidates a central-difference gradient needs.
Also the wall time of examples/calibrate.py's full fit (18 coefficients, 45,823 rows).  Writes DIR/grad_timing.json
(default: the current directory) with the card's name and power limit read in the same run.  The timing series are
synthetic (smooth random states and inputs in the tank's range): the cost does not depend on the values."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DT, HS = 0.02, [1, 10, 100]


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
    rng = np.random.default_rng(0)

    def synth(rows):
        walk = np.cumsum(rng.normal(0, 0.01, (rows, 12)), axis=0)
        X = 0.3 * np.tanh(walk)
        U = np.clip(np.cumsum(rng.normal(0, 0.02, (rows, 8)), axis=0) * 0.2, -1, 1)
        return X, U

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

    from bluerov2_dynamics_b200.engine import PHYS_NAMES as names
    sel = {1: ["Xu_abs"], 6: ["quad"], 18: ["added", "lin", "quad"],
           36: ["m", "W", "B", "xb", "yb", "zb", "Ix", "Iy", "Iz", "added", "lin", "quad", "current"] +
               ["Minv_u", "Minv_v", "Minv_w", "Minv_p", "Minv_q", "Minv_r"]}
    ph = B.with_minv(B.default_physical())
    ph[33:36] = 0.05             # a current, so that the current entries have a non-zero effect
    cases = []
    for rows in ((45823,) if quick else (45823, 1000100)):
        X, U = synth(rows)
        e = B.Engine("thruster8", "f64")
        Xt, Ut = e.tensor(X), e.tensor(U)
        e.set_physical(ph)
        for mode in ("reset", "carry"):
            passes = [HS] if mode == "reset" else [[h] for h in HS]
            t_single = timed(lambda: [e.multistep_se(Xt, Ut, p, dt=DT, lag_mode=mode) for p in passes])
            for p in ((1, 18) if quick else (1, 6, 18, 36)):
                rebuild = p != 36
                t_grad = timed(lambda: e.multistep_se_grad(Xt, Ut, HS, ph, sel[p], dt=DT, lag_mode=mode,
                                                           rebuild_minv=rebuild))
                idx = B.parameter_indices(sel[p])
                table = np.tile(ph, (2 * p + 1, 1))
                for j, i in enumerate(idx):
                    table[1 + 2 * j, i] *= 1 + 1e-4
                    table[2 + 2 * j, i] *= 1 - 1e-4
                t_cd = timed(lambda: [e.multistep_se_sweep(Xt, Ut, q, table, dt=DT, lag_mode=mode) for q in passes])
                r = dict(rows=rows, mode=mode, p=p, K=1, grad_ms=t_grad, single_ms=t_single, cd_sweep_ms=t_cd,
                         cd_candidates=2 * p + 1, grad_over_single=t_grad / t_single, grad_over_cd=t_grad / t_cd,
                         params=[names[i] for i in idx] if p <= 6 else sel[p])
                cases.append(r)
                print(json.dumps({k: v for k, v in r.items() if k != "params"}), flush=True)
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import calibrate
    fit = calibrate.run(verbose=True)
    res = dict(gpu=info, cases=cases, calibration=fit)
    with open(os.path.join(outdir, "grad_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("# gpu:", info)


if __name__ == "__main__":
    main()
