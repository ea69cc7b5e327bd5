"""Two builds of libbrov.so side by side on the adjoint sweeps: bitwise equality of every output, and the time of the
headline calls with the two builds alternating, on a GPU.

    python profiles/lib_compare.py --base OTHER/libbrov.so [--out DIR] [--rounds R]

  Results: seeded rollout_vjp, rollout_vjp(coef=True) with shared coefficients and with a per-vehicle table, and
      closed_loop_vjp with all three operand gradients (a tnc and a const_shared K, shared coefficients and a table),
      every model x integrator, without and with a water current, 300 vehicles x 50 steps.  gz0, gU, gkp, gK, gz_ref,
      gu_ref, z and the health counters of the two builds are compared bit for bit.
  Time: N = 65,536 x T = 1000, fp64, the calls of adjoint_timing.py / adjoint_coef_timing.py / cl_vjp_timing.py, each
      build in its own process, the builds alternating for R rounds; each entry is the median of 5 CUDA-event-timed
      calls after a warm-up call.
Each build runs in a subprocess with BROV_LIB pointing at it (the package's own library for the branch side).  Writes
DIR/lib_compare.json with the card's name, power limit and maximum SM clock."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from adjoint_timing import DT, problem, timed  # noqa: E402
from cl_vjp_timing import feedback  # noqa: E402

MODELS = ("thruster8", "wrench12", "quat13")
CURRENT = (0.12, -0.07, 0.05)
# (model, integrator, call, per-vehicle table) timed at 65,536 x 1000: the headline RK4 calls of every model, and the
# Euler closed-loop builds
TIMED = [(m, "rk4", c, t) for m in MODELS for c, t in (("vjp", False), ("coef", False), ("coef", True), ("cl", False),
                                                      ("cl", True))] + \
        [(m, "euler", "cl", t) for m in ("thruster8", "wrench12") for t in (False, True)]


def _table(B, e, n, seed, current=False):
    import numpy as np
    rng = np.random.default_rng(seed)
    ph = np.tile(B.default_physical(), (n, 1))
    ph[:, B._lib.PH_ADDED:B._lib.PH_QUAD + 6] *= rng.uniform(0.7, 1.3, (n, 18))
    if current:
        ph[:, B._lib.PH_CURRENT:B._lib.PH_CURRENT + 3] = CURRENT
    e.set_vehicle_physical(B.with_minv(ph))


def _call(B, e, call, integ, n, T, seed, k_const=False):
    """a closure running one seeded call, and its outputs as a dict of tensors"""
    import numpy as np
    import torch
    stride = 10
    g = torch.Generator(device=e.device).manual_seed(seed + 1)
    if call in ("vjp", "coef"):
        x0, U = problem(e, n, T, seed)
        gtraj = torch.randn((T // stride, n, e.nx), generator=g, device=e.device, dtype=torch.float64)
        gzT = torch.randn((n, e.nz), generator=g, device=e.device, dtype=torch.float64)

        def run():
            r = e.rollout_vjp(x0, U, gtraj=gtraj, gzT=gzT, stride=stride, dt=DT, integrator=integ, health=True,
                              coef=call == "coef")
            out = dict(gx0=r.gx0, gU=r.gU, z=r.z, health=r.health)
            if r.glag0 is not None:
                out["glag0"] = r.glag0
            if r.gkp is not None:
                out["gkp"] = r.gkp
            return out
        return run
    lim = dict(u_min=-1.0, u_max=1.0) if e.model == "thruster8" else dict(u_min=-50.0, u_max=50.0)
    x0, K, zr, ur = feedback(e, n, T, seed)
    Kt = K if k_const or n * T > 10 ** 5 else K.expand(T, n, e.nu, e.nz).clone()
    Kt = Kt + 1e-3 * torch.randn(Kt.shape, generator=g, device=e.device, dtype=torch.float64)
    gtraj = torch.randn((T // stride, n, e.nz), generator=g, device=e.device, dtype=torch.float64)
    gzT = torch.randn((n, e.nz), generator=g, device=e.device, dtype=torch.float64)
    gc = torch.full((n,), 1.0 / n, dtype=torch.float64, device=e.device)
    qw, rw = np.ones(e.nz), np.ones(e.nu)

    def run():
        r = e.closed_loop_vjp(x0, Kt, zr, ur, gtraj=gtraj, gzT=gzT, gcost=gc, stride=stride, steps=T, dt=DT,
                              integrator=integ, cost_q=qw, cost_r=rw, health=True, **lim)
        out = dict(gx0=r.gx0, gK=r.gK, gz_ref=r.gz_ref, gu_ref=r.gu_ref, z=r.z, health=r.health)
        if r.glag0 is not None:
            out["glag0"] = r.glag0
        return out
    return run


def worker(mode, out):
    import numpy as np
    import torch
    import bluerov2_dynamics_b200 as B
    res = {}
    if mode == "check":
        n, T = 300, 50
        calls = (("vjp", False, False), ("coef", False, False), ("coef", True, False), ("cl", False, False),
                 ("cl", True, False), ("cl", False, True), ("cl", True, True))
        for model in MODELS:
            for integ in ("rk4", "euler"):
                for cur in (False, True):
                    for call, table, k_const in calls:
                        e = B.Engine(model, "f64", current=CURRENT if cur and not table else None)
                        if table:
                            _table(B, e, n, 4, cur)
                        o = _call(B, e, call, integ, n, T, 11, k_const)()
                        name = f"{model}-{integ}-{call}{'-table' if table else ''}{'-kconst' if k_const else ''}"
                        for k, v in o.items():
                            res[f"{name}{'-current' if cur else ''}-{k}"] = v.cpu().numpy()
        np.savez(out, **res)
        return
    n, T = 65536, 1000
    for model, integ, call, table in TIMED:
        e = B.Engine(model, "f64")
        if table:
            _table(B, e, n, 4)
        t, ts = timed(_call(B, e, call, integ, n, T, 1), 5)
        res[f"{model}-{integ}-{call}{'-table' if table else ''}"] = dict(median_ms=t, all_ms=ts)
        del e
        torch.cuda.empty_cache()
    with open(out, "w") as f:
        json.dump(res, f)


def main():
    import numpy as np
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True, help="the other build's libbrov.so")
    ap.add_argument("--out", default=".")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--worker", choices=("check", "time"))
    ap.add_argument("--result")
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.result)
    libs = {"base": os.path.abspath(a.base), "branch": os.path.join(ROOT, "bluerov2_dynamics_b200", "libbrov.so")}
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": info[0] if info else None}

    def run(side, mode, path):
        env = dict(os.environ, BROV_LIB=libs[side])
        subprocess.run([sys.executable, os.path.abspath(__file__), "--base", a.base, "--worker", mode, "--result", path],
                       env=env, check=True)

    with tempfile.TemporaryDirectory() as d:
        outs = {}
        for side in libs:
            outs[side] = os.path.join(d, f"{side}.npz")
            run(side, "check", outs[side])
        ra, rb = np.load(outs["base"]), np.load(outs["branch"])
        assert set(ra.files) == set(rb.files)
        diff = sorted(k for k in ra.files if ra[k].tobytes() != rb[k].tobytes())
        res["bitwise"] = dict(arrays=len(ra.files), identical=len(ra.files) - len(diff), different=diff,
                              max_abs_diff={k: float(np.nanmax(np.abs(ra[k] - rb[k]))) for k in diff})
        print(json.dumps(res["bitwise"]), flush=True)
        rounds = []
        for r in range(a.rounds):
            for side in (("base", "branch") if r % 2 == 0 else ("branch", "base")):
                p = os.path.join(d, f"t{r}{side}.json")
                run(side, "time", p)
                with open(p) as f:
                    rounds.append(dict(side=side, **json.load(f)))
    res["rounds"] = rounds
    summary = {}
    for key in rounds[0]:
        if key == "side":
            continue
        s = {side: sorted(x[key]["median_ms"] for x in rounds if x["side"] == side) for side in libs}
        summary[key] = dict(base_ms=s["base"], branch_ms=s["branch"],
                            branch_over_base=float(np.median(s["branch"]) / np.median(s["base"])))
        print(key, json.dumps(summary[key]), flush=True)
    res["time"] = summary
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "lib_compare.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
