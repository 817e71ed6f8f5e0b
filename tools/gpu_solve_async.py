"""What the stream-ordered SQP solver (ntgb_solve_sqp_async) and a CUDA graph save in a real-time-iteration
control step: the active-bound lane changes of tools/gpu_mpc_warm.py (tests/test_gpu_mpc.py _active_specs),
warm state carried, max_iter = 2.  One step = solve, ntgb_spline_interp at dt, the new initial state copied
into both bound arrays.  Three ways, alternated over --reps repetitions of --steps steps each, from the state a
full warm solve reached:
  sync   ntgb_solve_sqp_warm (synchronizes inside), then the interpolation and the copy
  async  ntgb_solve_sqp_async, the interpolation and the copy, one stream synchronize per step
  graph  the whole step captured once with torch.cuda.graph and replayed, one synchronize per step
Per step: wall time (host clock around the step, which ends in a synchronize), median over all steps of all
repetitions, and the 10th / 90th percentiles.  The three ways must end in the same bits (checked).  At the
largest P, the GPU time of one step (sum of the device time of every kernel, copy and memset in a
torch.profiler trace of separate steps) for sync and async: the async line search evaluates all 16 steps of
every problem where the synchronous one evaluates 4 and then 12 for the problems that need them.  Prints the
card, its power limit, and one JSON object.

usage: python tools/gpu_solve_async.py [--P 1,64,1024,16384] [--reps N] [--steps K] [--out FILE]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np
import torch

from gpu_mpc_warm import card
from ntg_b200 import Problem, configs

MODES = ("sync", "async", "graph")


class Loop:
    """one fleet of P problems: the state after a full warm solve, and the step in the three ways"""

    def __init__(self, P, dt, seed=43):
        from test_gpu_mpc import _active_specs
        spec, lo, up = _active_specs(P, seed=seed)
        X = torch.from_numpy(configs.coefficients("cfg3", P, spec, seed=seed + 1)).cuda()
        self.pb = pb = Problem(spec, 0, fast=True)
        self.tq = torch.tensor([dt], dtype=torch.float64, device="cuda")
        self.C, self.lo, self.up = X, torch.from_numpy(lo).cuda(), torch.from_numpy(up).cuda()
        self.W = pb.sqp_warm_state(P)
        pb.solve_sqp(self.C, lowerb=self.lo, upperb=self.up, warm=self.W)      # step 1: a full warm solve
        self.step(True)
        self.start = [t.clone() for t in self.state()]
        pb.solver_reserve("sqp", P)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.step(False)

    def state(self):
        return (self.C, self.lo, self.up, self.W)

    def step(self, sync):
        self.pb.solve_sqp(self.C, max_iter=2, lowerb=self.lo, upperb=self.up, warm=self.W, sync=sync)
        z = self.pb.spline_interp(self.C, self.tq)[:, 0, :]
        self.lo[:, :6] = z
        self.up[:, :6] = z

    def run(self, mode):
        if mode == "graph":
            self.graph.replay()
        else:
            self.step(mode == "sync")
        torch.cuda.synchronize()

    def reset(self):
        for t, s in zip(self.state(), self.start):
            t.copy_(s)
        torch.cuda.synchronize()


def gpu_us(loop, mode, n):
    """device time per step: every CUDA kernel, copy and memset of n steps in a profiler trace"""
    from torch.profiler import ProfilerActivity, profile
    loop.reset()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            loop.run(mode)
    ev = [e for e in prof.events() if e.device_type.name == "CUDA"]
    ev_eval = [e for e in ev if "ntg_eval" in e.name]
    return {"us_per_step": sum(e.device_time for e in ev) / n, "eval_us_per_step": sum(e.device_time for e in ev_eval) / n,
            "launches_per_step": len(ev) / n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--P", default="1,64,1024,16384")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--dt", type=float, default=0.1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "gpu_solve_async.py measures on the GPU"
    Ps = [int(p) for p in args.P.split(",")]
    out = {"card": card(), "device": torch.cuda.get_device_name(0), "steps": args.steps, "reps": args.reps,
           "dt": args.dt, "max_iter": 2, "P": {}}
    print("card (name, power limit, max SM clock):", out["card"], flush=True)
    for P in Ps:
        loop = Loop(P, args.dt)
        ms = {m: [] for m in MODES}
        final = {}
        for m in MODES:                      # warm-up: module load, launch plans
            loop.reset()
            loop.run(m)
        for _ in range(args.reps):
            for m in MODES:
                loop.reset()
                for _ in range(args.steps):
                    t0 = time.perf_counter()
                    loop.run(m)
                    ms[m].append(1e3 * (time.perf_counter() - t0))
                final[m] = [t.cpu().numpy() for t in loop.state()]
        same = all(np.array_equal(a.view(np.uint8), b.view(np.uint8))
                   for m in MODES[1:] for a, b in zip(final[m], final["sync"]))
        r = {m: {"ms_median": round(float(np.median(ms[m])), 4), "ms_p10": round(float(np.percentile(ms[m], 10)), 4),
                 "ms_p90": round(float(np.percentile(ms[m], 90)), 4)} for m in MODES}
        r["same_bits"] = bool(same)
        out["P"][P] = r
        print(f"P = {P:6d}: " + ", ".join(f"{m} {r[m]['ms_median']:.3f} ms [{r[m]['ms_p10']:.3f}, {r[m]['ms_p90']:.3f}]"
                                          for m in MODES) + f" per step; same bits: {same}", flush=True)
        if P == max(Ps):
            g = {m: gpu_us(loop, m, 5) for m in ("sync", "async")}
            out["gpu_time_largest_P"] = {"P": P, **g}
            print(f"P = {P}: GPU time per step sync {g['sync']['us_per_step']:.1f} us "
                  f"(evaluator {g['sync']['eval_us_per_step']:.1f}), async {g['async']['us_per_step']:.1f} us "
                  f"(evaluator {g['async']['eval_us_per_step']:.1f})", flush=True)
        loop.pb.close()
        del loop
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
