"""Cost of per-problem bounds in the batched solvers: ntgb_solve_eq against ntgb_solve_eq_bounds on
65 536 lane changes (configs.kincar(64), no nonlinear rows) with distinct initial / final states, and
ntgb_solve_sqp against ntgb_solve_sqp_bounds on 16 384 lane changes with active speed / curvature bounds
(tests/test_gpu_next.py _kincar_active_constraints) with distinct states and limits.  Each solver runs
three ways, alternately, from the same starts: shared bounds, per-problem bounds that replicate the
setup's (same problems: the cost of the path itself) and distinct per-problem bounds (different problems,
so the iteration counts differ too).  Each call is timed with CUDA events around it (it ends in a stream
synchronise).  k_bounds_prep alone is timed from a torch.profiler trace of separate calls.
Prints the card, its power limit, and one JSON object.

usage: python tools/gpu_mpc.py [--reps N] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

from ntg_b200 import Problem, configs


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), r


def alternate(name, calls, reps):
    """calls: {label: fn}, run in turn reps times after one warm-up each; each fn clones the same starts"""
    for fn in calls.values():
        fn()  # warm-up: reduction, scratch, module load
    t = {k: [] for k in calls}
    for _ in range(reps):
        for k, fn in calls.items():
            t[k].append(timed(fn)[0])
    r = {}
    for k, v in t.items():
        v = np.array(v)
        r[k] = {"ms_median": float(np.median(v)), "ms_min": float(v.min()), "ms": [round(float(x), 3) for x in v]}
    base = r["shared"]["ms_median"]
    print(f"{name}: " + ", ".join(f"{k} {v['ms_median']:.2f} ms (x{v['ms_median'] / base:.3f})" for k, v in r.items()),
          flush=True)
    return r


def prep_kernel_us(call, n=10):
    """mean device time of k_bounds_prep over n calls, from a profiler trace"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            call()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "k_bounds_prep" in e.name and e.device_type.name == "CUDA"]
    if not ev:
        return None
    return float(np.mean([e.device_time for e in ev]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "gpu_mpc.py measures on the GPU"
    out = {"card": card(), "device": torch.cuda.get_device_name(0)}
    print("card (name, power limit, max SM clock):", out["card"], flush=True)

    from test_gpu_mpc import _active_specs, _lane_changes
    # ---- eq: 65 536 lane changes, each with its own x0 / xf
    spec = configs.kincar(64, constraints=False, name="mpc_bench_eq")
    P = 65536
    X = torch.from_numpy(configs.coefficients("cfg4", P, spec, seed=41)).cuda()
    b = torch.from_numpy(_lane_changes(P, seed=42)).cuda()
    pb = Problem(spec, 0, fast=True)

    def eq_shared():
        C = X.clone()
        return pb.solve_eq(C)

    def eq_bounds():
        C = X.clone()
        return pb.solve_eq(C, lowerb=b, upperb=b)

    brep = torch.from_numpy(np.tile(spec.lowerb, (P, 1))).cuda()

    def eq_replicated():
        C = X.clone()
        return pb.solve_eq(C, lowerb=brep, upperb=brep)

    calls = {"shared": eq_shared, "bounds_replicated": eq_replicated, "bounds_distinct": eq_bounds}
    out["eq"] = alternate(f"solve_eq kincar64 x{P}", calls, args.reps)
    for k, fn in calls.items():
        f, it, st = fn()
        out["eq"][k].update(iters_mean=float(it.float().mean()), status1=float((st == 1).float().mean()))
    out["eq"].update(P=P, k_bounds_prep_us=prep_kernel_us(eq_bounds, 5))
    pb.close()

    # ---- sqp: 16 384 active-bound lane changes, own x0 and limits
    P = 16384
    spec, lo, up = _active_specs(P, seed=43)
    X = torch.from_numpy(configs.coefficients("cfg3", P, spec, seed=44)).cuda()
    lo, up = torch.from_numpy(lo).cuda(), torch.from_numpy(up).cuda()
    pb = Problem(spec, 0, fast=True)

    def sqp_shared():
        C = X.clone()
        return pb.solve_sqp(C)

    def sqp_bounds():
        C = X.clone()
        return pb.solve_sqp(C, lowerb=lo, upperb=up)

    lrep = torch.from_numpy(np.tile(spec.lowerb, (P, 1))).cuda()
    urep = torch.from_numpy(np.tile(spec.upperb, (P, 1))).cuda()

    def sqp_replicated():
        C = X.clone()
        return pb.solve_sqp(C, lowerb=lrep, upperb=urep)

    calls = {"shared": sqp_shared, "bounds_replicated": sqp_replicated, "bounds_distinct": sqp_bounds}
    out["sqp"] = alternate(f"solve_sqp active-bound kincar40 x{P}", calls, args.reps)
    for k, fn in calls.items():
        f, v, it, st = fn()
        out["sqp"][k].update(iters_mean=float(it.float().mean()), status1=float((st == 1).float().mean()))
    out["sqp"].update(P=P, k_bounds_prep_us=prep_kernel_us(sqp_bounds, 3))
    pb.close()
    print(f"k_bounds_prep: {out['eq']['k_bounds_prep_us']} us (eq, 65 536), "
          f"{out['sqp']['k_bounds_prep_us']} us (sqp, 16 384)", flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
