"""What the SQP warm start (ntgb_solve_sqp_warm) saves in receding-horizon MPC: 16 384 lane changes with
active speed / curvature bounds, each with its own state and limits (tests/test_gpu_mpc.py _active_specs),
over a 10-step horizon.  Each step solves, then moves every problem's initial state to its own solution's
flat state at dt (ntgb_spline_interp, on the device).  Two loops run from the same starts, alternated over
--reps repetitions: "cold" (ntgb_solve_sqp_bounds, B = I every step) and "warm" (ntgb_solve_sqp_warm, the
warm array carried from step to step).  Per step: ms (CUDA events around the call, which ends in a stream
synchronise; median over the repetitions), mean iterations, the fraction with status 1, and the largest
relative warm-vs-cold cost difference (the median too).  A call lasts as long as its slowest problem,
so the largest iteration count is printed beside the mean.  One more loop is real-time iteration: a full
warm solve at step 1, then max_iter = 2 per step with the warm array carried.  k_sqp_warm_store and
k_sqp_init (warm and cold) are timed from a torch.profiler trace of separate calls.  Prints the card, its
power limit, and one JSON object.

usage: python tools/gpu_mpc_warm.py [--reps N] [--steps K] [--out FILE]"""
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


def run_loop(pb, X, lo0, up0, steps, dt, mode):
    """one receding-horizon loop from the starts X; mode cold / warm / rti -> per step (ms, f, iters, status)"""
    Cd, lo, up = X.clone(), lo0.clone(), up0.clone()
    W = pb.sqp_warm_state(X.shape[0]) if mode != "cold" else None
    tq = torch.tensor([dt], dtype=torch.float64, device=X.device)
    out = []
    for k in range(steps):
        max_iter = 2 if (mode == "rti" and k > 0) else 0
        ms, (f, v, it, st) = timed(lambda: pb.solve_sqp(Cd, max_iter=max_iter, lowerb=lo, upperb=up, warm=W))
        out.append((ms, f.cpu().numpy(), it.cpu().numpy(), st.cpu().numpy()))
        z = pb.spline_interp(Cd, tq)[:, 0, :]
        lo[:, :6] = z
        up[:, :6] = z
    return out


def kernel_us(call, names, n=3):
    """mean device time per launch of each kernel named in names, from a profiler trace of n calls"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            call()
        torch.cuda.synchronize()
    r = {}
    for nm in names:
        ev = [e for e in prof.events() if nm in e.name and e.device_type.name == "CUDA"]
        r[nm] = float(np.mean([e.device_time for e in ev])) if ev else None
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--P", type=int, default=16384)
    ap.add_argument("--dt", type=float, default=0.1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "gpu_mpc_warm.py measures on the GPU"
    out = {"card": card(), "device": torch.cuda.get_device_name(0), "P": args.P, "steps": args.steps, "dt": args.dt}
    print("card (name, power limit, max SM clock):", out["card"], flush=True)

    from test_gpu_mpc import _active_specs
    P = args.P
    spec, lo, up = _active_specs(P, seed=43)
    X = torch.from_numpy(configs.coefficients("cfg3", P, spec, seed=44)).cuda()
    lo, up = torch.from_numpy(lo).cuda(), torch.from_numpy(up).cuda()
    pb = Problem(spec, 0, fast=True)
    modes = ("cold", "warm", "rti")
    for m in modes:
        run_loop(pb, X, lo, up, 2, args.dt, m)  # warm-up: reduction, scratch, module load
    ms = {m: [] for m in modes}
    res = {}
    for _ in range(args.reps):
        for m in modes:
            r = run_loop(pb, X, lo, up, args.steps, args.dt, m)
            ms[m].append([x[0] for x in r])
            res[m] = r  # deterministic: every repetition computes the same
    for m in modes:
        t = np.median(np.array(ms[m]), axis=0)
        ref = res["cold"]
        rows = []
        for k in range(args.steps):
            _, f, it, st = res[m][k]
            fc = ref[k][1]
            d = np.abs(f - fc) / np.maximum(1.0, np.abs(fc))
            rows.append({"ms": round(float(t[k]), 3), "iters_mean": float(it.mean()), "iters_max": int(it.max()),
                         "status1": float((st == 1).mean()), "dcost_vs_cold_median": float(np.median(d)),
                         "dcost_vs_cold_max": float(d.max())})
        out[m] = {"steps": rows, "ms_total": round(float(t.sum()), 3),
                  "ms_steps_2_on": round(float(t[1:].sum()), 3),
                  "iters_steps_2_on": float(sum(r["iters_mean"] for r in rows[1:]))}
        print(f"{m:4s}: total {out[m]['ms_total']:.2f} ms, steps 2..{args.steps} {out[m]['ms_steps_2_on']:.2f} ms, "
              f"{out[m]['iters_steps_2_on']:.2f} iterations per problem", flush=True)
        for k, r in enumerate(rows):
            print(f"  step {k + 1:2d}: {r['ms']:7.2f} ms  iters mean {r['iters_mean']:6.2f} max {r['iters_max']:3d}  "
                  f"status1 {r['status1']:.4f}  |f - f_cold| / max(1, |f_cold|) median {r['dcost_vs_cold_median']:.1e} "
                  f"max {r['dcost_vs_cold_max']:.1e}", flush=True)
    c, w = out["cold"], out["warm"]
    print(f"warm / cold, steps 2..{args.steps}: time {w['ms_steps_2_on'] / c['ms_steps_2_on']:.3f}, "
          f"iterations {w['iters_steps_2_on'] / c['iters_steps_2_on']:.3f}", flush=True)

    # kernel times, separate calls under the profiler: re-solves at a solution, with its rows and cold
    W = pb.sqp_warm_state(P)
    C1 = X.clone()
    pb.solve_sqp(C1, lowerb=lo, upperb=up, warm=W)
    Wsave, C1save = W.clone(), C1.clone()

    def warm_call():
        W.copy_(Wsave)
        return pb.solve_sqp(C1save.clone(), lowerb=lo, upperb=up, warm=W)

    def cold_call():
        return pb.solve_sqp(C1save.clone(), lowerb=lo, upperb=up)

    out["kernels_us_warm"] = kernel_us(warm_call, ["k_sqp_init", "k_sqp_warm_store", "k_sqp_step"])
    out["kernels_us_cold"] = kernel_us(cold_call, ["k_sqp_init", "k_sqp_step"])
    print(f"kernels (us per launch): warm {out['kernels_us_warm']}, cold {out['kernels_us_cold']}", flush=True)
    pb.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
