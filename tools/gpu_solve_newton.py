"""Newton against L-BFGS on long horizons (ntgb_solve_eq_newton, ntgb_solve_eq_lbfgs): lane changes of configs.kincar
over 8, 64 and 256 intervals per output (nC = 38, 262, 1030; 3 breakpoints per interval), starts from
configs.coefficients ("cfg3").  For every shape, on the CPU: the cost of the KKT solution (the oracle's gradient
at the identity columns, then [H A'; A 0]); on the device: the colours K and the half-bandwidth w.

Timed with default options (Newton: at most 100 iterations, gtol 1e-9; L-BFGS: at most 500 iterations, gtol
1e-9, memory 8), per (intervals, P), the two solvers alternated within each of --reps repetitions:
  - wall time of one call (host clock around the synchronous call), median over the repetitions;
  - mean and maximum iterations, the status counts, and at the point each problem stopped the largest
    relative cost gap to the KKT cost, |f - f_kkt| / max(1, |f_kkt|), and the median and largest relative
    projected gradient |P g|_inf / max(1, |f|);
  - device time per call by kernel family from a separate torch.profiler run of one call: the evaluator
    (cost + gradient at C, gradients at the difference points, costs at the trial points), the Newton kernels
    (k_newton_*) or the L-BFGS kernels (k_lbfgs_*), and the search (trial points, merit, picks).
Prints the card, its power limit, and one JSON object.

usage: python tools/gpu_solve_newton.py [--ninterv 8,64,256] [--P 1024,16384] [--reps N] [--out FILE]"""
import argparse
import dataclasses
import json
import os
import sys
import time
import warnings

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np
import torch

from gpu_mpc_warm import card
from ntg_b200 import Problem, configs

FAMILIES = (("eval", ("ntg_eval",)), ("newton", ("k_newton_",)), ("lbfgs", ("k_lbfgs_",)),
            ("search", ("k_ls_trial", "k_cost_merit", "k_alm_pick")))


def lane(ninterv):
    return dataclasses.replace(configs.kincar(3 * ninterv + 1, constraints=False, name=f"newton_lane{ninterv}"),
                               ninterv=[ninterv, ninterv], knots=None)


def kkt(port, spec):
    """-> (Q1 [r][nC] orthonormal rows spanning A's, cond(H on null(A)), KKT cost) of the quadratic lane change"""
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    H = port.eval(spec, np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]
    H = 0.5 * (H + H.T)
    _, s, Vt = np.linalg.svd(A)
    r = int((s > 1e-11 * s[0]).sum())
    ev = np.linalg.eigvalsh(Vt[r:] @ H @ Vt[r:].T)
    K = np.block([[H, A.T], [A, np.zeros((A.shape[0], A.shape[0]))]])
    Cref = np.linalg.solve(K, np.concatenate([np.zeros(nC), b]))[:nC]
    fref = float(port.eval(spec, Cref[None, :], mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0])
    return Vt[:r], float(ev.max() / ev.min()), fref


class Shape:
    def __init__(self, port, ninterv):
        self.spec = lane(ninterv)
        self.pb = Problem(self.spec, 0)
        Q1, self.cond, self.fref = kkt(port, self.spec)
        self.Q1 = torch.from_numpy(Q1).cuda()
        self.ninterv = ninterv

    def quality(self, C, f):
        """at the points reached: largest relative cost gap to the KKT cost, median / largest relative |P g|_inf"""
        g = self.pb.eval(C, mode_obj=2, mode_con=-1, jac=0)["g"]
        pg = g - (g @ self.Q1.T) @ self.Q1
        rel = (pg.abs().amax(dim=1) / f.abs().clamp(min=1.0)).cpu().numpy()
        gap = (np.abs(f.cpu().numpy() - self.fref) / max(1.0, abs(self.fref))).max()
        return {"fgap_max": float(gap), "pg_median": float(np.median(rel)), "pg_max": float(rel.max())}


class Case:
    def __init__(self, shape, P):
        self.shape, self.P = shape, P
        self.X = torch.from_numpy(configs.coefficients("cfg3", P, shape.spec, seed=shape.ninterv)).cuda()

    def call(self, solver, **kw):
        C = self.X.clone()
        torch.cuda.synchronize()
        t = time.perf_counter()
        f, it, st = (self.shape.pb.solve_eq_lbfgs if solver == "lbfgs" else self.shape.pb.solve_eq_newton)(C, **kw)
        dt = time.perf_counter() - t
        return dt, C, f, it.cpu().numpy(), st.cpu().numpy()


def device_us(case, solver):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        case.call(solver)
    ev = [e for e in prof.events() if e.device_type.name == "CUDA"]
    out = {name: sum(e.device_time for e in ev if any(k in e.name for k in keys)) for name, keys in FAMILIES}
    out["all"] = sum(e.device_time for e in ev)
    return out


def row(case, solver, dt, C, f, it, st):
    out = {"solver": solver, "ninterv": case.shape.ninterv, "nC": case.shape.spec.nC, "P": case.P,
           "ms": 1e3 * dt, "iters_mean": float(it.mean()), "iters_max": int(it.max()),
           "status": {int(k): int(v) for k, v in zip(*np.unique(st, return_counts=True))}}
    out.update(case.shape.quality(C, f))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ninterv", default="8,64,256")
    ap.add_argument("--P", default="1024,16384")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "gpu_solve_newton.py measures on the GPU"
    warnings.filterwarnings("ignore", module="torch.profiler")
    from oracle.oracle import Oracle
    port = Oracle("port")
    argv = sys.argv[1:]
    if args.out:
        argv = [a if a != args.out else "<dir>/" + os.path.basename(a) for a in argv]
    cmd = " ".join(["python tools/gpu_solve_newton.py"] + argv)
    print(f"# {cmd}   (one B200; card line below is from the same run)")
    res = {"card": card(), "shapes": [], "cases": []}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    shapes = {int(n): Shape(port, int(n)) for n in args.ninterv.split(",")}
    for n, s in shapes.items():
        K, w, _ = s.pb.newton_structure()
        line = {"ninterv": n, "nC": s.spec.nC, "cond_null": s.cond, "f_kkt": s.fref, "colors": K, "half_bandwidth": w}
        res["shapes"].append(line)
        print(json.dumps(line), flush=True)
    cases = [Case(shapes[int(n)], int(P)) for n in args.ninterv.split(",") for P in args.P.split(",")]
    runs = [(c, s) for c in cases for s in ("newton", "lbfgs")]
    for c, s in runs:                       # warm-up: module loading, scratch allocation
        c.call(s)
    times = {(id(c), s): [] for c, s in runs}
    last = {}
    for _ in range(args.reps):
        for c, s in runs:
            r = c.call(s)
            times[(id(c), s)].append(r[0])
            last[(id(c), s)] = r
    for c, s in runs:
        out = row(c, s, *last[(id(c), s)])
        out["ms"] = 1e3 * float(np.median(times[(id(c), s)]))
        out["device_us"] = device_us(c, s)
        res["cases"].append(out)
        print(json.dumps(out), flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
