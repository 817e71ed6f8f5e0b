#!/usr/bin/env python
"""bench.py -- collocation evals/sec (cost + constraints + Jacobian, batched)
and % of the HBM roofline, on 1..8 B200 (BASELINE.json `metric`).

    python bench.py --gpus N --steps K --warmup W [--workload cfg4] [--scaling weak|strong]
                    [--launch graph|stream] [--gather fused|nccl] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic coefficient
vectors: a single launch of the fused evaluator (funobj mode 2 + funcon mode 2
for every problem of the batch: cost, gradient, constraints, banded Jacobian).
At N > 1 the step includes the gather of the per-problem (objective,
violation) table: fused into the evaluator's epilogue as peer stores (default)
or one NCCL all_gather (--gather nccl).  The batch shards by problem index; no
data-path collective.

Headline workload (DESIGN.md "Measurement"): CFG-4, the kincar MPC shape with
64 breakpoints x 65536 problems per GPU (weak scaling: the driver's scaling run
compares per-N values).  The named multi-GPU configs -- 65536 horizons and the
16384 high-order problems IN TOTAL, sharded over the GPUs -- are measured at
every N under "strong_scaling"; CFG-2/3/5, the exact variant, the dense NPSOL
Jacobian layout and the general kernel are reported under "other_workloads" at
N = 1.

Timing: the K timed steps are ONE CUDA graph of K launches (value, ms_per_step);
the same K steps are then launched on the stream with an event pair around each
launch (roofline.kernel_ms, ms_per_step_stream_launch).  Both regions sit
between barrier + synchronize; maximum over ranks.

Rank 0 prints ONE JSON line.  `--impl reference` times the reference's own CPU
implementation (oracle/_ref: the unmodified reference C sources) on all host
cores for the same metric and config.
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
sys.path.insert(0, ROOT)

from ntg_b200 import JAC_BAND, JAC_DENSE, configs  # noqa: E402

L2_BYTES = 126e6
KERNEL_OF = {"cfg2": "ntgb::ntg_eval_small_kernel<vdp> (K1s)", "cfg3": "ntgb::ntg_eval_small_kernel<kincar> (K1s)",
             "cfg4": "ntgb::ntg_eval_small_kernel<kincar> (K1s)", "cfg5": "ntgb::ntg_eval_cluster_kernel<syn6> (K1c)"}
METRIC = "collocation_evals_per_sec"
UNIT = "evals/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# --------------------------------------------------------------------------- CPU reference arm
def _ref_worker(args):
    cfg, lo, hi, P, kind, shipped = args
    from oracle.oracle import Oracle
    spec, _ = configs.get(cfg)
    X = configs.coefficients(cfg, P, spec)[lo:hi]
    o = Oracle(kind, shipped_flags=shipped) if kind == "ref" else Oracle(kind)
    t0 = time.perf_counter()
    r = o.eval(spec, X, dense=False, band=False, outputs=False, reps=1)
    return time.perf_counter() - t0, r["seconds"], hi - lo


class CpuReference:
    """The reference's CPU implementation of the path on the host cores: one
    process per core (the reference is non-re-entrant: file-static globals,
    src/ntg.c:17-41), disjoint slices of the sample."""

    def __init__(self, cfg: str, cores: int | None = None, shipped: bool = False):
        from oracle import oracle
        self.cfg = cfg
        self.shipped = shipped   # the reference's own CFLAGS=-g (Makefile:18) instead of -O2
        self.kind = "ref" if oracle.have_ref() else "port"
        self.cores = cores or len(os.sched_getaffinity(0))
        import multiprocessing as mp
        self.pool = mp.get_context("spawn").Pool(self.cores)

    def sample_size(self, target_seconds: float) -> int:
        spec, P = configs.get(self.cfg)
        # calibrate on one core
        n0 = 4 if self.cfg == "cfg5" else 512
        w, s, n = _ref_worker((self.cfg, 0, n0, n0, self.kind, self.shipped))
        per_eval = max(s, 1e-9) / n
        n_target = int(target_seconds * self.cores / per_eval)
        per_core = max(1, min(n_target, P) // self.cores)
        return per_core * self.cores

    def step(self, nsample: int):
        from ntg_b200.shard import shard_range
        jobs = [(self.cfg, *shard_range(nsample, r, self.cores), nsample, self.kind, self.shipped)
                for r in range(self.cores)]
        t0 = time.perf_counter()
        res = self.pool.map(_ref_worker, jobs)
        wall = time.perf_counter() - t0
        inner = max(r[1] for r in res)   # slowest worker, funcon+funobj time only
        return wall, inner

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline(cfg: str, target_seconds: float = 4.0):
    ref = CpuReference(cfg)
    try:
        n = ref.sample_size(target_seconds)
        ref.step(min(n, ref.cores * 2))  # warm the workers (imports, table build)
        wall, inner = min((ref.step(n) for _ in range(3)), key=lambda t: t[1])  # best of 3 passes
        one = CpuReference(cfg, cores=1)
        n1 = max(1, n // ref.cores)
        one.step(1)
        _, inner1 = one.step(n1)
        one.close()
        shipped = {}
        if ref.kind == "ref" and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libntg_ref_g.so")):
            # as shipped: the reference's Makefile builds with CFLAGS=-g (no optimisation)
            g = CpuReference(cfg, shipped=True)
            try:
                ng = max(g.cores, (n // 4) // g.cores * g.cores)
                g.step(min(ng, g.cores * 2))
                _, inner_g = min((g.step(ng) for _ in range(2)), key=lambda t: t[1])
                shipped = {"value_shipped_flags": ng / inner_g,
                           "shipped_flags": "-g (reference Makefile:18), same sources, all cores"}
            finally:
                g.close()
        spec, P = configs.get(cfg)
        return {**shipped, "value": n / inner, "unit": UNIT, "cores": ref.cores,
                "kind": "reference" if ref.kind == "ref" else "port",
                "sample": f"{n} of {P} problems of {spec.name} (same seeded coefficients), one process per "
                          f"core, -O2 -ffp-contract=off; funobj mode 2 + funcon mode 2 per problem",
                "value_1core": n1 / inner1, "wall_value": n / wall}
    finally:
        ref.close()


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ref = CpuReference(a.workload)
    spec, P = configs.get(a.workload)
    if a.problems:
        P = a.problems
    n = ref.sample_size(a.ref_step_seconds)
    for _ in range(max(a.warmup, 1)):
        ref.step(n)
    t, tw = [], []
    for _ in range(a.steps):
        wall, inner = ref.step(n)
        t.append(inner)   # slowest worker's time inside funcon+funobj: the path itself,
        tw.append(wall)   # without this harness's process dispatch and input generation
    ref.close()
    per_step = float(np.mean(t))
    value = n / per_step
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": a.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(a, spec, P if a.scaling == "weak" else (P + a.gpus - 1) // a.gpus,
                                  P * a.gpus if a.scaling == "weak" else P, a.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores,
                         "kind": "reference" if ref.kind == "ref" else "port",
                         "sample": f"each step = {n} of {P} problems of {spec.name}, one process per core, "
                                   f"step time = slowest worker's time inside funcon+funobj",
                         "wall_value": n / float(np.mean(tw))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)
    return 0


def workload_config(a, spec, P, Ptot, ngpus):
    """The SAME dictionary in both arms (everything in it follows from the command line): the
    reference arm is the CPU baseline OF this configuration."""
    per_set = P * spec.bytes_per_eval()
    nset = 1 if per_set >= 2 * L2_BYTES else min(64, int(np.ceil(2 * L2_BYTES / per_set)))
    fast = a.variant == "fast"
    return {"workload": spec.name, "cfg": a.workload, "problems_per_gpu": P, "total_problems": Ptot,
            "nout": spec.nout, "nbps": spec.nbps, "order": spec.order[0], "nC": spec.nC,
            "ncnln": spec.ncnln, "jacobian": "band-compact",
            "bytes_per_eval": spec.bytes_per_eval(), "parallelism": f"problem-sharded x{ngpus}",
            "variant": ("fast (FMA contraction, node-weight quadrature with 4 partial sums; within 1e-12 of the "
                        "CPU reference -- the bit-identical `exact` variant is timed under other_workloads.cfg4_exact)"
                        if fast else
                        "exact (-fmad=false, reference summation order, bit-identical to the CPU reference)"),
            "l2": (f"inputs+outputs of one step = {per_set * nset / 1e6:.0f} MB over a ring of {nset} "
                   f"buffer set(s), larger than the 126 MB L2"),
            "launch": (f"the {a.steps} timed steps are ONE CUDA graph of {a.steps} evaluator launches"
                       if a.launch == "graph" else f"{a.steps} stream launches")}


# --------------------------------------------------------------------------- GPU arm
def jac_bytes_per_eval(spec, jac):
    """SURVEY.md section 8(d): 8*(nC + 1 + nC + ncnln + nnzJ); nnzJ = ncnln*S (band) or ncnln*nC (dense NPSOL layout)"""
    if jac == JAC_BAND:
        return spec.bytes_per_eval()
    return 8 * (2 * spec.nC + 1 + spec.ncnln + spec.ncnln * spec.nC)


def make_ring(torch, pb, spec, Xnp, jac=JAC_BAND):
    """Ring of buffer sets larger than 2 x L2 when one set is not (every set holds the same
    coefficients, so every launch computes the same results into different memory)."""
    dev = torch.device("cuda", pb.device)
    P = int(Xnp.shape[0])
    per_set = P * jac_bytes_per_eval(spec, jac)
    nset = 1 if per_set >= 2 * L2_BYTES else min(64, int(np.ceil(2 * L2_BYTES / per_set)))
    X0 = torch.from_numpy(np.ascontiguousarray(Xnp)).to(dev)
    sets = [(X0.clone() if i else X0, pb.alloc_outputs(P, jac, zero=False)) for i in range(nset)]
    return {"sets": sets, "nset": nset, "P": P, "per_set": per_set, "jac": jac,
            "footprint_mb": per_set * nset / 1e6}


def time_graph(torch, pb, ring, steps, warmup, dist=None, peers=None):
    """EXACTLY `steps` launches captured in ONE CUDA graph (cycling over the ring), replayed once
    between barrier + synchronize; -> ms per step.  With the fused gather (peers) the launches carry
    the peer stores, so a step is complete (every rank's table written) when its kernel retires."""
    dev = torch.device("cuda", pb.device)
    sets, nset, jac = ring["sets"], ring["nset"], ring["jac"]
    st = torch.cuda.current_stream(dev).cuda_stream
    for i in range(max(warmup, 1)):
        pb.launch(pb.eval_args(sets[i % nset][0], sets[i % nset][1], 2, 2, jac, 0, st, peers=peers))
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cs = torch.cuda.current_stream(dev).cuda_stream
        for i in range(steps):
            pb.launch(pb.eval_args(sets[i % nset][0], sets[i % nset][1], 2, 2, jac, 0, cs, peers=peers))
    g.replay()                       # untimed: the graph is uploaded here
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    chk = float(sets[(steps - 1) % nset][1]["result"][:, 0].sum().item())
    assert np.isfinite(chk), "non-finite objective in the timed run"
    del g
    return e0.elapsed_time(e1) / steps


def check_gather(torch, dist, peers, local_result, P_total):
    """The fused gather against the collective it replaces: after the timed run, ONE NCCL
    all_gather of this rank's (objective, violation) rows must equal, bit for bit, the table the
    evaluators' peer stores wrote into this rank's HBM."""
    from ntg_b200.shard import gather_results
    peers.fence()
    want = gather_results(local_result, P_total)
    got = peers.table()
    ok = torch.tensor([1 if torch.equal(got, want) else 0], dtype=torch.int32, device=local_result.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    assert int(ok.item()) == 1, "fused gather: a rank's gathered table differs from NCCL all_gather"
    return True


def time_stream(torch, pb, ring, steps, warmup, dist=None, world=1, peers=None):
    """One stream launch per step, an event pair around every launch.
    -> dict(ms_per_step, kernel_ms = mean launch duration).
    N > 1 without the fused gather: the 16 B/problem NCCL all_gather of step i runs asynchronously
    on NCCL's stream while later kernels run; four result tables rotate so that a gather never reads
    a table a kernel is writing."""
    dev = torch.device("cuda", pb.device)
    sets, nset, jac, P = ring["sets"], ring["nset"], ring["jac"], ring["P"]
    stream = torch.cuda.current_stream(dev)
    nccl = dist is not None and peers is None
    NB = 4
    if nccl:
        res2 = [torch.empty((P, 2), dtype=torch.float64, device=dev) for _ in range(NB)]
        gath2 = [torch.empty((world * P, 2), dtype=torch.float64, device=dev) for _ in range(NB)]
        args = [[pb.eval_args(x, dict(o, result=res2[b]), 2, 2, jac, 0, stream.cuda_stream) for x, o in sets]
                for b in range(NB)]
    else:
        args = [[pb.eval_args(x, o, 2, 2, jac, 0, stream.cuda_stream, peers=peers) for x, o in sets]]
    pending = [None] * NB

    def step(i, ev=None):
        b = i % NB if nccl else 0
        if nccl and pending[b] is not None:
            pending[b].wait()          # the gather that last read res2[b] is done
        if ev is not None:
            ev[0].record()
        pb.launch(args[b][i % nset])
        if ev is not None:
            ev[1].record()
        if nccl:
            pending[b] = dist.all_gather_into_tensor(gath2[b], res2[b], async_op=True)

    def drain():
        for b in range(NB):
            if pending[b] is not None:
                pending[b].wait()
                pending[b] = None
        if peers is not None:
            peers.fence()   # fused gather: the tables are complete once every rank's stream has drained

    for i in range(warmup):
        step(i)
    drain()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(steps):
        step(i, ev[i])
    drain()
    e1.record()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    if nccl:
        r0 = dist.get_rank()
        b = (steps - 1) % NB
        assert torch.equal(gath2[b][r0 * P:(r0 + 1) * P], res2[b]), "gathered table does not hold this rank's rows"
    total_ms = e0.elapsed_time(e1)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    chk = float((res2[0] if nccl else sets[0][1]["result"])[:, 0].sum().item())
    assert np.isfinite(chk), "non-finite objective in the timed run"
    return {"ms_per_step": total_ms / steps, "kernel_ms": kernel_ms}


def time_small(torch, pb, ring, steps, warmup):
    """Launch-bound workloads (a few microseconds of GPU time per step): ONE CUDA graph holds a whole
    lap over the ring of buffer sets, so the host launch cost is paid once per lap."""
    dev = torch.device("cuda", pb.device)
    sets, nset, jac = ring["sets"], ring["nset"], ring["jac"]
    st = torch.cuda.current_stream(dev).cuda_stream
    for x, o in sets:
        pb.launch(pb.eval_args(x, o, 2, 2, jac, 0, st))
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cs = torch.cuda.current_stream(dev).cuda_stream
        for x, o in sets:
            pb.launch(pb.eval_args(x, o, 2, 2, jac, 0, cs))
    laps_w = max(1, warmup // nset + 1)
    laps = max(1, (steps + nset - 1) // nset)
    for _ in range(laps_w):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(laps):
        g.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / (laps * nset)
    assert np.isfinite(float(sets[0][1]["result"][:, 0].sum().item())), "non-finite objective in the timed run"
    return {"ms_per_step": ms, "kernel_ms": ms, "launches": laps * nset}


DUMP_BYTES = 64 << 20


def dump_outputs(torch, out, ncnln, path):
    """What a caller of the timed path receives from one step -- f [P], g [P][nC], c [P][ncnln],
    J [P][ncnln*S] in the device band layout, result [P][2] -- as path/<name>.npy, float64.  When
    the batch holds more than DUMP_BYTES of them, the rows of a sorted sample of problems drawn with
    a fixed seed are written, so two runs with the same arguments write the same problems."""
    arrays = {"f": out["f"], "g": out["g"], "c": out["c"][:, :ncnln], "J": out["J"], "result": out["result"]}
    arrays = {k: v for k, v in arrays.items() if v is not None}
    P = int(out["f"].shape[0])
    row_bytes = sum(v[0].numel() * v.element_size() for v in arrays.values())
    n = min(P, DUMP_BYTES // row_bytes)
    idx = None
    if n < P:
        rows = np.sort(np.random.default_rng(0).choice(P, n, replace=False))
        idx = torch.from_numpy(rows).to(out["f"].device)
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), (v if idx is None else v.index_select(0, idx)).cpu().numpy())


def d2h_ceiling(torch, device, nbytes, reps=3):
    """What the link gives: ONE plain cudaMemcpyAsync of `nbytes` from HBM into pinned host memory
    (torch's non_blocking copy_), best of `reps`; -> GB/s"""
    dev = torch.device("cuda", device)
    n = max(1, int(nbytes) // 8)
    src = torch.empty(n, dtype=torch.float64, device=dev)
    dst = torch.empty(n, dtype=torch.float64).pin_memory()
    best = None
    for _ in range(reps + 1):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    del src, dst
    return n * 8 / best / 1e9


def time_e2e(torch, pb, spec, cfg, P, steps, warmup, full: bool):
    """Same metric end to end with HOST buffers: every step copies that step's coefficients from
    pinned host memory, evaluates, and copies results back to pinned host memory.
    full=True: ONE call of the C ABI's host-buffer entry point `ntgb_eval_host` per step -- f, g, c
    and the whole Jacobian band come back (what a host-side consumer such as NPSOL needs); the
    library chunks the batch and overlaps copies with compute on two streams.
    full=False ("resident"): only the per-problem (objective, violation) table comes back; g, c, J
    are still computed and written to HBM, where a GPU-side consumer would read them.  Steps are
    independent batches, so they are pipelined: four chunks per step alternate between two streams
    and the host only waits at the end (in-stream order protects the two device buffer sets)."""
    dev = torch.device("cuda", pb.device)
    d = pb.dims
    Xh = torch.from_numpy(configs.coefficients(cfg, P, spec)).pin_memory()
    if full:
        host = {"f": torch.empty(P, dtype=torch.float64).pin_memory(),
                "result": torch.empty((P, 2), dtype=torch.float64).pin_memory(),
                "g": torch.empty((P, d.nC), dtype=torch.float64).pin_memory(),
                "c": torch.empty((P, d.ncnln), dtype=torch.float64).pin_memory(),
                "J": torch.empty((P, d.ncnln * d.sorder), dtype=torch.float64).pin_memory()}
        h2d = P * d.nC * 8
        d2h = sum(v.numel() * 8 for v in host.values())

        def one_step():
            pb.eval_host_tensors(Xh, host, 2, 2, JAC_BAND)

        def finish():
            pass
    else:
        nchunk = 4 if P >= 8192 else 1
        Pc = P // nchunk
        host = {"result": torch.empty((P, 2), dtype=torch.float64).pin_memory()}
        streams = [torch.cuda.Stream(dev) for _ in range(2)]
        bufs = []
        for s in range(2):
            with torch.cuda.stream(streams[s]):
                bufs.append((torch.empty((Pc, d.nC), dtype=torch.float64, device=dev),
                             pb.alloc_outputs(Pc, JAC_BAND, zero=False)))
        h2d = P * d.nC * 8
        d2h = host["result"].numel() * 8

        # everything that does not change from step to step is prepared once: the host side of a
        # step is 4 x (copy, launch, copy)
        plan = []
        for ci in range(nchunk):
            s = ci % 2
            lo, hi = ci * Pc, (ci + 1) * Pc
            xd, out = bufs[s]
            plan.append((streams[s], xd, Xh[lo:hi], pb.eval_args(xd, out, 2, 2, JAC_BAND, 0, streams[s].cuda_stream),
                         host["result"][lo:hi], out["result"]))

        def one_step():
            for st, xd, xh, args, rh, rd in plan:
                with torch.cuda.stream(st):
                    xd.copy_(xh, non_blocking=True)
                    pb.launch(args)
                    rh.copy_(rd, non_blocking=True)

        def finish():
            for st in streams:
                st.synchronize()

    for _ in range(warmup):
        one_step()
    finish()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    finish()
    torch.cuda.synchronize(dev)
    dt = (time.perf_counter() - t0) / steps
    assert np.isfinite(float(host["result"][:, 0].sum())), "non-finite objective in the e2e run"
    return {"value": P / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_step": dt * 1e3,
            "what": ("one ntgb_eval_host() call per step: all outputs (f, g, c, Jacobian band) to pinned host memory"
                     if full else
                     "(objective, violation) table to host every step; g, c, J computed and left resident in HBM; "
                     "4 chunks per step on 2 streams, steps pipelined (host waits once, after the last step)")}


def time_solvers(torch, device, fast):
    """Wall time of the batched solvers on the lane-change problem of examples/kincar.c:
    ntgb_solve_eq (linear equalities only, as shipped), ntgb_solve_nlp and ntgb_solve_sqp (active speed
    and curvature bounds).  Host wall clock around the synchronous C call, after one warm-up solve."""
    import dataclasses
    from ntg_b200 import Problem
    out = {}
    s1 = configs.kincar(64, constraints=False, name="solve_kincar_64bps")
    P1 = 65536
    X1 = torch.from_numpy(configs.coefficients("cfg3", P1, s1, seed=3)).to(f"cuda:{device}")
    pb = Problem(s1, device, fast=fast)
    pb.solve_eq(X1.clone(), max_iter=100)
    C1 = X1.clone()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, it, st = pb.solve_eq(C1, max_iter=100)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["solve_eq"] = {"workload": "kincar lane change, 64 breakpoints, linear equalities only", "problems": P1,
                       "ms": dt * 1e3, "problems_per_s": P1 / dt, "iterations_mean": float(it.float().mean()),
                       "converged_frac": float((st >= 1).float().mean())}
    pb.close()
    base = configs.kincar(40, constraints=True, name="solve_kincar_active")
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(ninterv=[4, 4], knots=None, bps=None)
    s2 = type(base)(**kw)
    lo, up = s2.lowerb.copy(), s2.upperb.copy()
    lo[-2], up[-2], lo[-1], up[-1] = 0.0, 66.2, -7.2, 7.2
    s2.lowerb, s2.upperb = lo, up
    P2 = 16384
    X2 = torch.from_numpy(configs.coefficients("cfg3", P2, s2, seed=5)).to(f"cuda:{device}")
    pb = Problem(s2, device, fast=fast)
    pb.solve_nlp(X2.clone())   # warm-up at full size: the scratch is allocated here, not in the timed call
    C2 = X2.clone()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, v, it, st = pb.solve_nlp(C2)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["solve_nlp"] = {"workload": "kincar lane change, 40 breakpoints, 4 intervals, active speed^2 / curvature bounds",
                        "problems": P2, "ms": dt * 1e3, "problems_per_s": P2 / dt,
                        "iterations_mean": float(it.float().mean()), "converged_frac": float((st >= 1).float().mean()),
                        "violation_max": float(v.max())}
    pb.solve_sqp(X2.clone())
    C3 = X2.clone()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, v, it, st = pb.solve_sqp(C3)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["solve_sqp"] = {"workload": "the same 16384 problems and starts; SQP (dual active-set QP per problem in shared memory, BFGS)",
                        "problems": P2, "ms": dt * 1e3, "problems_per_s": P2 / dt,
                        "iterations_mean": float(it.float().mean()), "converged_frac": float((st == 1).float().mean()),
                        "violation_max": float(v[st == 1].max()) if bool((st == 1).any()) else None}
    pb.close()
    torch.cuda.empty_cache()
    return out


_REAL_STDOUT = None


def _quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version
    banner on stdout when NCCL_DEBUG is set), so file descriptor 1 is pointed at stderr for the run
    and the line goes to the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def kernel_source_hash(cfg: str) -> str:
    """sha256 over the sources that define the workload's dominant kernel: profiles/traffic.json is
    stamped with it, and a stamp that no longer matches means the ncu capture describes an older
    kernel (the .git directory does not travel to the GPU box, so the working tree is hashed)."""
    import hashlib
    files = ["ntg_b200/csrc/ntg_kernel_args.h", "ntg_b200/csrc/ntg_eval_kernel.cuh", "ntg_b200/csrc/ntg_eval_small.cuh",
             "ntg_b200/csrc/ntg_small_plan.h", "include/ntg_b200.h"]
    files += {"cfg2": ["ntg_b200/packs/vdp.c"], "cfg3": ["ntg_b200/packs/kincar.c"], "cfg4": ["ntg_b200/packs/kincar.c"],
              "cfg5": ["ntg_b200/csrc/ntg_eval_cluster.cuh", "ntg_b200/csrc/ntg_eval_cluster_hot.cuh",
                       "ntg_b200/packs/syn6.c"]}[cfg]
    h = hashlib.sha256()
    for f in files:
        h.update(open(os.path.join(ROOT, f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(cfg: str):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture, or
    None when there is none for the kernel as it is now."""
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        e = json.load(open(tr)).get(cfg)
        if isinstance(e, dict) and e.get("kernel_source_hash") == kernel_source_hash(cfg):
            return e.get("dram_bytes_per_launch")
    except Exception:
        pass
    return None


def strong_scaling(torch, dist, world, rank, local, fast, peak, gather):
    """BASELINE.json configs[3] / configs[4] as named: the TOTAL batch is fixed (65 536 horizons,
    16 384 high-order problems) and sharded over the ranks by problem index (shard_range); every
    rank's evaluator stores its result pairs into all ranks' tables (fused gather) and the tables
    are checked against an NCCL all_gather after the timed run.  Steps are captured in one CUDA
    graph: at 8 GPUs a step is ~16 us of kernel."""
    from ntg_b200 import Problem
    from ntg_b200.shard import PeerGather, shard_range
    out = {}
    for cfg, steps in (("cfg4", 50), ("cfg5", 10)):
        spec, Ptot = configs.get(cfg)
        lo, hi = shard_range(Ptot, rank, world)
        X = configs.coefficients(cfg, Ptot, spec)[lo:hi]
        pb = Problem(spec, local, fast=fast)
        peers, how = None, "none (1 GPU)"
        if world > 1:
            how = "nccl all_gather after the run only (no fused gather)"
            if gather == "fused":
                try:
                    peers = PeerGather(pb, Ptot)
                    how = "fused peer stores, checked against NCCL all_gather"
                except Exception as e:
                    sys.stderr.write(f"bench: fused gather unavailable ({e})\n")
        ring = make_ring(torch, pb, spec, X)
        del X
        ms = time_graph(torch, pb, ring, steps, 3, dist, peers)
        if peers is not None:
            check_gather(torch, dist, peers, ring["sets"][(steps - 1) % ring["nset"]][1]["result"], Ptot)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        pmax = (Ptot + world - 1) // world
        gbs = pmax * spec.bytes_per_eval() / (ms * 1e-3) / 1e9
        out[cfg] = {"workload": spec.name, "total_problems": Ptot, "problems_per_gpu": pmax, "n_gpus": world,
                    "steps": steps, "ms_per_step": ms, "evals_per_s": Ptot / (ms * 1e-3),
                    "algorithmic_gbs_per_gpu": gbs, "roofline_frac_per_gpu": gbs / peak, "gather": how,
                    "launch": f"one CUDA graph of {steps} launches over a ring of {ring['nset']} buffer set(s)",
                    "kernel": KERNEL_OF[cfg]}
        if peers is not None:
            peers.close()
        del ring
        pb.close()
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--variant", default=os.environ.get("NTG_BENCH_VARIANT", "fast"), choices=["exact", "fast"])
    ap.add_argument("--problems", type=int, default=0, help="override problems per GPU (weak) / in total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the named batch PER GPU; strong: the named batch in total, sharded by problem index")
    ap.add_argument("--launch", default=os.environ.get("NTG_BENCH_LAUNCH", "graph"), choices=["graph", "stream"],
                    help="graph: the K timed steps are ONE CUDA graph; stream: K stream launches")
    ap.add_argument("--no-others", action="store_true", help="skip the other workloads / baselines")
    ap.add_argument("--gather", default=os.environ.get("NTG_BENCH_GATHER", "fused"), choices=["fused", "nccl"],
                    help="N > 1: how the 16 B/problem result table reaches every rank")
    ap.add_argument("--ref-step-seconds", type=float, default=1.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                         f"(rank 0; a fixed sample of problems when the batch holds more than {DUMP_BYTES >> 20} MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3)
    _quiet_stdout()

    if a.impl == "reference":
        return run_reference_arm(a)

    import torch
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the evaluator has no CPU fallback "
                         "(use --impl reference for the CPU reference arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        # --gather fused (default): the evaluator's epilogue stores each rank's (objective, violation)
        # rows into EVERY rank's gathered table over NVLink (CUDA IPC peer tables, ntg_b200/shard.py::
        # PeerGather); no collective kernel runs beside the persistent evaluator.
        # --gather nccl: one asynchronous all_gather per step.  The persistent evaluator fills every
        # SM, so the NCCL kernel can only start when evaluator CTAs retire and then holds back a few
        # CTAs of the NEXT launch, which finish last (N = 2: 144 us per step; with four SMs left
        # free and four NCCL channels 139 us; at N = 4 / 8 the 4 / 8 MB table needs NCCL's default
        # channel count: 138 / 149 us).
        if a.gather == "nccl" and world == 2:
            os.environ.setdefault("NTG_B200_SM_RESERVE", "4")
            os.environ.setdefault("NCCL_MAX_NCHANNELS", "4")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from ntg_b200 import Problem
    from ntg_b200.shard import shard_range

    spec, P = configs.get(a.workload)
    if a.problems:
        P = a.problems
    strong = a.scaling == "strong"
    Ptot = P if strong else world * P
    lo, hi = shard_range(Ptot, rank, world)
    Xnp = configs.coefficients(a.workload, P, spec)
    if strong:
        Xnp = Xnp[lo:hi]
    Ploc = int(Xnp.shape[0])
    fast = a.variant == "fast"
    pb = Problem(spec, local, fast=fast)
    peak, peak_src = measured_peaks()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    peers = None
    gather_how = "none"
    if world > 1:
        gather_how = "nccl all_gather_into_tensor, asynchronous, 4 rotating tables"
        if a.gather == "fused":
            try:
                from ntg_b200.shard import PeerGather
                peers = PeerGather(pb, Ptot)
                gather_how = ("fused: peer stores from the evaluator's epilogue into every rank's table (CUDA IPC, "
                              "NVLink), one 16-byte store per problem and table; checked bit for bit against an NCCL "
                              "all_gather after the timed run")
            except Exception as e:  # no peer access between these GPUs: the collective still works
                sys.stderr.write(f"bench: fused gather unavailable ({e}); using NCCL\n")
                peers = None
    ring = make_ring(torch, pb, spec, Xnp)
    use_graph = a.launch == "graph" and (world == 1 or peers is not None)
    ms_graph = time_graph(torch, pb, ring, a.steps, a.warmup, dist, peers) if use_graph else None
    rs = time_stream(torch, pb, ring, a.steps, a.warmup, dist, world, peers)
    gather_checked = False
    if peers is not None:
        gather_checked = check_gather(torch, dist, peers, ring["sets"][(a.steps - 1) % ring["nset"]][1]["result"], Ptot)
    if a.dump_outputs and rank == 0:
        dump_outputs(torch, ring["sets"][(a.steps - 1) % ring["nset"]][1], pb.dims.ncnln, a.dump_outputs)

    ms = torch.tensor([ms_graph if use_graph else rs["ms_per_step"], rs["kernel_ms"], rs["ms_per_step"]],
                      dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step, ms_kernel_ev, ms_stream = float(ms[0]), float(ms[1]), float(ms[2])
    # average launch duration: inside the graph the launches run back to back, so (time of the graph)
    # / K is the kernel's duration plus the gap to the next launch -- an upper bound of the kernel
    # time; an event pair around a stream launch also spans the launch latency of the kernel
    ms_kernel = min(ms_step, ms_kernel_ev) if use_graph else ms_kernel_ev
    value = Ptot / (ms_step * 1e-3)
    nset, footprint_mb = ring["nset"], ring["footprint_mb"]
    del ring
    torch.cuda.empty_cache()

    e2e = time_e2e(torch, pb, spec, a.workload, Ploc, max(3, min(a.steps, 10)), 3, full=True)
    e2e_res = time_e2e(torch, pb, spec, a.workload, Ploc, max(3, min(a.steps, 20)), 3, full=False)
    if dist is not None:
        dist.barrier()
    ceil_gbs = d2h_ceiling(torch, local, e2e["d2h_bytes_per_step"])   # every rank at the same time
    if dist is not None:
        t = torch.tensor([e2e["value"], e2e_res["value"], ceil_gbs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        e2e["value"], e2e_res["value"], ceil_gbs = float(t[0]) * world, float(t[1]) * world, float(t[2])
    e2e["d2h_ceiling_gbs_per_gpu"] = ceil_gbs
    e2e["d2h_achieved_gbs_per_gpu"] = e2e["d2h_bytes_per_step"] / (Ploc / (e2e["value"] / world)) / 1e9
    e2e["frac_of_d2h_ceiling"] = e2e["d2h_achieved_gbs_per_gpu"] / ceil_gbs
    e2e["ceiling_how"] = ("one plain pinned cudaMemcpyAsync of the step's d2h bytes, best of 3" +
                          (f", all {world} ranks at the same time (minimum over ranks)" if world > 1 else ""))
    clocks = sampler.stop() if sampler else None

    if peers is not None:
        peers.close()
        peers = None
    strong_lines = None
    if not a.no_others:
        pb.close()
        pb = None
        torch.cuda.empty_cache()
        strong_lines = strong_scaling(torch, dist, world, rank, local, fast, peak, a.gather)

    others = {}
    if rank == 0 and world == 1 and not a.no_others:
        for cfg in ("cfg2", "cfg3", "cfg4", "cfg5"):
            if cfg == a.workload:
                continue
            s2, P2 = configs.get(cfg)
            pb2 = Problem(s2, local, fast=fast)
            small = cfg in ("cfg2", "cfg3")
            st = 200 if small else (5 if cfg == "cfg5" else 20)
            ring2 = make_ring(torch, pb2, s2, configs.coefficients(cfg, P2, s2))
            r2 = time_small(torch, pb2, ring2, st, 5) if small else time_stream(torch, pb2, ring2, st, 5)
            gbs = P2 * s2.bytes_per_eval() / (r2["kernel_ms"] * 1e-3) / 1e9
            others[cfg] = {"workload": s2.name, "problems": P2, "evals_per_s": P2 / (r2["ms_per_step"] * 1e-3),
                           "ms_per_step": r2["ms_per_step"], "kernel_ms": r2["kernel_ms"],
                           "algorithmic_gbs": gbs, "roofline_frac": gbs / peak,
                           "launch": "one CUDA graph per lap over the buffer ring" if small else "stream launch", "kernel": KERNEL_OF[cfg],
                           "l2": f"ring of {ring2['nset']} buffer sets, {ring2['footprint_mb']:.0f} MB"}
            del ring2
            pb2.close()
            torch.cuda.empty_cache()
        # the same workload two more ways: bit-identical variant, NPSOL's dense column-major
        # Jacobian layout (src/ntg.c:217-220); then outputs with DIFFERENT spline setups (no cluster
        # kernel) on longer horizons: 320 breakpoints (K1s on CTAs of 512 threads) and 640 (the
        # general kernel K1, the fallback for everything the register-table kernels do not take)
        extra = [("cfg4_exact", a.workload, None, False, JAC_BAND, 20, None),
                 ("cfg4_dense_npsol_layout", a.workload, None, fast, JAC_DENSE, 20, None),
                 ("nonuniform_endpoint_320bps", "endpt", configs.endpoint(320, name="endpoint_320bps_x16384"), fast, JAC_BAND, 10,
                  "ntgb::ntg_eval_small_kernel<endpt, BLOCK=512> (K1s, one CTA of 512 threads per SM)"),
                 ("k1_general_endpoint_640bps", "endpt", configs.endpoint(640, name="endpoint_640bps_x8192"), fast, JAC_BAND, 10,
                  "ntgb::ntg_eval_kernel<endpt> (K1 general)")]
        for key, cfg, s3, fst, jac, st, kname in extra:
            try:
                if s3 is None:
                    s3, P3 = configs.get(cfg)
                    X3 = configs.coefficients(cfg, P3, s3)
                else:
                    P3 = 16384 if s3.nbps <= 512 else 8192
                    X3 = configs.coefficients("other", P3, s3)
                pb3 = Problem(s3, local, fast=fst)
                ring3 = make_ring(torch, pb3, s3, X3, jac)
                r3 = time_stream(torch, pb3, ring3, st, 5)
                # numerator = the band figure in both layouts: out-of-band zeros of the dense layout are
                # written once at allocation, exactly as the reference does (SURVEY.md section 8(d))
                bpe = s3.bytes_per_eval()
                gbs = P3 * bpe / (r3["kernel_ms"] * 1e-3) / 1e9
                others[key] = {"workload": s3.name, "problems": P3, "variant": "fast" if fst else "exact",
                               "jacobian": "band-compact" if jac == JAC_BAND else "dense column-major (NPSOL), band entries written",
                               "bytes_per_eval": bpe, "evals_per_s": P3 / (r3["ms_per_step"] * 1e-3),
                               "ms_per_step": r3["ms_per_step"], "kernel_ms": r3["kernel_ms"],
                               "algorithmic_gbs": gbs, "roofline_frac": gbs / peak}
                if kname:
                    others[key]["kernel"] = kname
                del ring3, X3
                pb3.close()
                torch.cuda.empty_cache()
            except Exception as e:
                others[key] = {"error": str(e)[:200]}
        try:   # the batched solvers built on the evaluator (informative, not the metric)
            others["solvers"] = time_solvers(torch, local, fast)
        except Exception as e:  # never let an extra take the bench line down
            others["solvers"] = {"error": str(e)[:200]}

    if rank == 0:
        bytes_launch = Ploc * spec.bytes_per_eval()
        ach = bytes_launch / (ms_kernel * 1e-3) / 1e9
        cfgd = workload_config(a, spec, (Ptot + world - 1) // world, Ptot, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfgd, "clocks": clocks,
            "e2e": e2e, "e2e_resident": e2e_res, "gpu_launches": a.steps,
            "ms_per_step_stream_launch": ms_stream,
            "launch_used": "graph" if use_graph else "stream",
            "gather": {"how": gather_how, "checked_against_nccl_all_gather": gather_checked} if world > 1 else None,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": measured_traffic(a.workload), "peak_source": peak_src,
                         "kernel": KERNEL_OF.get(a.workload, "ntgb::ntg_eval_kernel"),
                         "kernel_ms": ms_kernel,
                         "kernel_ms_how": ("(CUDA-event time of the graph of K back-to-back launches) / K" if use_graph and ms_step <= ms_kernel_ev
                                           else "mean over the event pairs around each of the K stream launches"),
                         "kernel_ms_event_pairs": ms_kernel_ev,
                         "algorithmic_bytes_per_launch": bytes_launch},
            "other_workloads": others,
        }
        if strong_lines is not None:
            line["strong_scaling"] = strong_lines
        if world == 1 and not a.no_others:
            line["cpu_baseline"] = cpu_baseline(a.workload)
        _emit(line)
    if peers is not None:
        peers.close()
    if pb is not None:
        pb.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
