"""Candidate sweep (brov_multistep_se_sweep) against a serial loop of single-vehicle evaluator calls, on a GPU.

    python profiles/sweep_timing.py [--out DIR] [--quick]

Series: the length of the reference's tank recording (45,823 rows) and the 1,000,100-row series of bench.py's evaluator
config; thruster8 RK4, H = 1/10/100, fp64 and fp32, reset (one pass for the three horizons) and carried lag (one pass
per horizon).  For P in {1, 8, 64, 512}:
  sweep    one Engine.multistep_se_sweep call for the P candidates (its launches, no host sync inside);
  serial   P x (Engine.set_physical + Engine.multistep_se(time_slices=1)), the loop the sweep replaces: timed over
           min(P, 16) calls and scaled to P (every call is the same work);
  rate     window-steps per second of the sweep (P x the integrator steps all windows run) against that of the single
           evaluator on the 1M-window series (default time slicing, the bench's 6.8 ms reset figure).
Variants (built with -D knobs of csrc/brov_kernels.cuh into bluerov2_dynamics_b200/variants/ when missing): item order
candidate-major instead of window-block-major, and fp32 coefficients in registers instead of shared memory.
Writes DIR/sweep_timing.json (default: the current directory) and prints one line per case.  The series are synthetic (smooth
random states and inputs in the tank's range): the evaluator's cost does not depend on the values."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
VARIANTS = {"cand_major": ["BROV_SWEEP_CAND_MAJOR=1"], "kp_regs": ["BROV_SWEEP_KP_REGS=1"]}
VDIR = os.path.join(ROOT, "bluerov2_dynamics_b200", "variants")
DT, HS = 0.02, [1, 10, 100]


def variant_lib(name):
    out = os.path.join(VDIR, f"libbrov_{name}.so")
    if not os.path.exists(out):
        from bluerov2_dynamics_b200.build import build_lib
        os.makedirs(VDIR, exist_ok=True)
        build_lib(force=True, defines=VARIANTS[name], out=out, tag="_" + name)
    return out


def worker(cases, quick):
    import numpy as np
    import torch
    import bluerov2_dynamics_b200 as B
    from bluerov2_dynamics_b200 import _lib as L
    rng = np.random.default_rng(0)

    def synth(rows):
        X = np.zeros((rows, 12))
        walk = np.cumsum(rng.normal(0, 0.01, (rows, 12)), axis=0)
        X[:] = 0.3 * np.tanh(walk)
        U = np.clip(np.cumsum(rng.normal(0, 0.02, (rows, 8)), axis=0) * 0.2, -1, 1)
        return X, U

    def cands(P):
        ph = np.tile(B.default_physical(), (P, 1))
        for col in (L.PH_ADDED, L.PH_LIN, L.PH_QUAD):
            ph[:, col:col + 6] *= rng.uniform(0.7, 1.3, (P, 6))
        return B.with_minv(ph)

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

    def window_steps(rows, hs):   # integrator steps the windows of one pass run: window k runs min(Hmax, rows-1-k)
        k = np.arange(max(rows - hs[0], 0))
        return int(np.minimum(hs[-1], rows - 1 - k).sum())

    out = []
    series = {}
    for c in cases:
        rows, dtype, mode, Ps = c["rows"], c["dtype"], c["mode"], c["P"]
        if rows not in series:
            series[rows] = synth(rows)
        e = B.Engine("thruster8", dtype)
        X, U = e.tensor(series[rows][0]), e.tensor(series[rows][1])
        passes = [HS] if mode == "reset" else [[h] for h in HS]
        steps = sum(window_steps(rows, p) for p in passes)
        ref_ph = cands(1)

        def single():   # the single evaluator: default time slicing
            for p in passes:
                e.multistep_se(X, U, p, dt=DT, lag_mode=mode)
        t_single = timed(single) if c.get("single") else None

        def one_call():  # one iteration of the serial loop
            e.set_physical(ref_ph[0])
            for p in passes:
                e.multistep_se(X, U, p, dt=DT, lag_mode=mode, time_slices=1)
        t_serial1 = timed(one_call)
        for P in Ps:
            ph = cands(P)
            t = timed(lambda: [e.multistep_se_sweep(X, U, p, ph, dt=DT, lag_mode=mode) for p in passes])
            n = min(P, 16)
            t_ser = timed(lambda: [(e.set_physical(ph[i]), [e.multistep_se(X, U, p, dt=DT, lag_mode=mode, time_slices=1)
                                                            for p in passes]) for i in range(n)]) * P / n
            r = dict(rows=rows, dtype=dtype, mode=mode, P=P, sweep_ms=t, serial_ms=t_ser, speedup=t_ser / t,
                     serial_one_call_ms=t_serial1, sweep_window_steps_per_s=P * steps / (t * 1e-3),
                     variant=os.environ.get("SWEEP_VARIANT", "default"))
            if t_single is not None:
                r["single_evaluator_ms"] = t_single
                r["single_window_steps_per_s"] = steps / (t_single * 1e-3)
            out.append(r)
            print(json.dumps(r), flush=True)
            if quick:
                break
    return out


def main():
    args = sys.argv[1:]
    if args and args[0] == "--worker":
        res = worker(json.loads(args[1]), "--quick" in args)
        print("RESULT " + json.dumps(res))
        return
    outdir = args[args.index("--out") + 1] if "--out" in args else os.getcwd()
    quick = "--quick" in args
    os.makedirs(outdir, exist_ok=True)
    Ps = [1, 8, 64, 512]
    base = [dict(rows=45823, dtype=d, mode=m, P=Ps) for d in ("f64", "f32") for m in ("reset", "carry")]
    base += [dict(rows=1000100, dtype=d, mode=m, P=Ps, single=True) for d in ("f64", "f32") for m in ("reset", "carry")]
    runs = [("default", None, base),
            ("cand_major", "cand_major", [dict(rows=r, dtype="f64", mode="reset", P=[64, 512]) for r in (45823, 1000100)]),
            ("kp_regs", "kp_regs", [dict(rows=r, dtype="f32", mode="reset", P=[64, 512]) for r in (45823, 1000100)])]
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    results = dict(gpu=info, cases=[])
    for name, var, cases in runs:
        env = dict(os.environ, SWEEP_VARIANT=name)
        if var:
            env["BROV_LIB"] = variant_lib(var)
        t0 = time.time()
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", json.dumps(cases)] +
                           (["--quick"] if quick else []), env=env, capture_output=True, text=True)
        sys.stdout.write("".join(l for l in r.stdout.splitlines(True) if not l.startswith("RESULT ")))
        if r.returncode != 0:
            sys.stderr.write(r.stderr)
            raise SystemExit(f"variant {name} failed")
        results["cases"] += json.loads(r.stdout.split("RESULT ", 1)[1])
        print(f"# {name}: {time.time() - t0:.0f} s", flush=True)
    with open(os.path.join(outdir, "sweep_timing.json"), "w") as f:
        json.dump(results, f, indent=1)
    print("# gpu:", info)


if __name__ == "__main__":
    main()
