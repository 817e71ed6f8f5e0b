"""GPU tests of the batched SQP solver iteration by iteration: ntgb_solve_sqp / _bounds / _warm stopped after
K = 1..6 iterations against the same K iterations of the lock-step host driver (tests/tools/sqp_lockstep.py:
the library's own reduced basis restated bit for bit, the g++-compiled core of ntg_sqp.cuh, the CPU oracle's
evaluations).  The end-result tests of test_gpu_sqp.py cannot see a slightly wrong row gradient or a lost
share of a reduction, because SQP corrects itself; a comparison after each iteration can.

The shapes are where k_sqp_step changes path: a tiled band Jacobian (K1c/H, nbps > 256), CTAs of 32 and 64
threads, more reduced variables than threads, every row kind, per-problem bounds, ragged 128-thread grids
(P = 129), and both sides of the shared-memory limit.  The exact build (fast=False) is used throughout."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from ntg_b200 import configs

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools"))
from sqp_lockstep import Core, Reduced, lockstep, rel_diff, rounding_spread, sqp_smem_bytes, warm_row_state  # noqa: E402

TAG = float(0x4E545731)
KS = (1, 2, 3, 4, 5, 6)


@pytest.fixture(scope="module")
def core(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("lockstep") / "sqp_host.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-I", os.path.join(os.path.dirname(HERE), "ntg_b200", "csrc"),
                           "-o", so, os.path.join(HERE, "tools", "sqp_host.cpp")])
    return Core(C.CDLL(so))


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _kincar(nbps=40, ninterv=4):
    from test_gpu_next import _kincar_active_constraints
    return _kincar_active_constraints(nbps=nbps, ninterv=ninterv)


def _setup(name):
    """-> (spec, starts [P][nC], per-problem (lowerb, upperb) or None)"""
    def small(spec, P, r, seed=1):
        return spec, np.random.default_rng(seed).uniform(-r, r, (P, spec.nC)), None

    def cfg3(spec, P):
        return spec, configs.coefficients("cfg3", P, spec, seed=5), None

    if name == "kincar_bounds":
        from test_gpu_mpc import _active_specs
        spec, lo, up = _active_specs(129, seed=3)
        return spec, configs.coefficients("cfg3", 129, spec, seed=5), (lo, up)
    return {
        "kincar_tiled301": lambda: cfg3(_kincar(301, 4), 5),
        "kincar_nr30": lambda: cfg3(_kincar(40, 9), 5),
        "kincar_nr34": lambda: cfg3(_kincar(40, 10), 5),
        "hi_nr31": lambda: small(configs.high_order(5, 3, 14, 33, name="lock_hi31"), 5, 0.01),
        "hi_nr32": lambda: small(configs.high_order(4, 2, 15, 33, name="lock_hi32"), 5, 0.05),
        "hi_nr63": lambda: small(configs.high_order(6, 3, 20, 65, name="lock_hi63"), 1, 0.01),
        "hi_nr64": lambda: small(configs.high_order(4, 2, 31, 65, name="lock_hi64"), 1, 0.05),
        "hi_nr66": lambda: small(configs.high_order(4, 2, 32, 81, name="lock_hi66"), 1, 0.01),
        "hi_nr70": lambda: small(configs.high_order(4, 2, 34, 81, name="lock_hi70"), 1, 0.05),
        "endpoint": lambda: small(configs.endpoint(), 129, 0.5, seed=3),
    }[name]()


SETUPS = ["kincar_tiled301", "kincar_nr30", "kincar_nr34", "hi_nr31", "hi_nr32", "hi_nr63", "hi_nr64", "hi_nr66",
          "hi_nr70", "endpoint", "kincar_bounds"]


def _gpu(pb, X, K, bounds, warm=None, **kw):
    """solve_sqp(max_iter=K) from X with a warm array (zeros: a cold start); every output on the host"""
    Cd = _cuda(X)
    W = pb.sqp_warm_state(X.shape[0]) if warm is None else _cuda(warm)
    lo, up = (None, None) if bounds is None else (_cuda(bounds[0]), _cuda(bounds[1]))
    f, v, it, st, lam, ist = pb.solve_sqp(Cd, max_iter=K, multipliers=True, warm=W, lowerb=lo, upperb=up, **kw)
    out = dict(C=Cd, f=f, viol=v, iters=it, status=st, lam=lam, istate=ist, W=W)
    return {k: t.cpu().numpy() for k, t in out.items()}


def _references(core, red, X, bounds, K, warm=None, **opts):
    """the lock-step reference of every problem, with its rounding spread (sqp_lockstep.rounding_spread)"""
    refs = []
    for p in range(X.shape[0]):
        kw = dict(opts)
        if bounds is not None:
            kw["hl"], kw["hu"], kw["Cpart"] = red.problem_bounds(bounds[0][p], bounds[1][p])
        if warm is not None:
            kw["B0"], kw["nu0"] = warm_row_state(warm[p], red.nr)
        r = lockstep(core, red, X[p], K, **kw)
        r["spread"], r["flip"] = rounding_spread(core.lib, red, X[p], K, r, **kw)
        refs.append(r)
    return refs


# the bars: C, f and violation; B and nu; multipliers -- for K <= 3 and for K = 4..6.  A problem whose own
# rounding spread times SPREAD_FACTOR exceeds a bar is held to that instead: the GPU sums in another order.
BARS = {True: (1e-10, 1e-9, 1e-8), False: (1e-8, 1e-7, 1e-8)}
SPREAD_FACTOR = 100.0


def _compare(name, red, gpu, refs):
    """gpu[K] against the reference snapshots.  A problem is compared only up to the iteration where its
    reference decided a line search within 1e-12 of the Armijo threshold, or where a rerun with one-ulp
    noise decided anything differently; such drops are counted, at most 1 in 20."""
    nr = red.nr
    drops, widened = 0, 0
    for p, ref in enumerate(refs):
        last = max(KS)
        close = next((j for j, s in enumerate(ref["steps"]) if s["margin"] < 1e-12), None)
        if close is not None:
            last = min(last, close)
        if ref["flip"] is not None:
            last = min(last, ref["flip"] - 1)
        drops += last < max(KS)
        for K in KS:
            if K > last:
                break
            g, s = {k: v[p] for k, v in gpu[K].items()}, ref["snaps"][K]
            tag = f"{name} p={p} K={K}"
            bc, bb, bl = BARS[K <= 3]
            tol = {q: max(bar, SPREAD_FACTOR * ref["spread"][(K, q)])
                   for q, bar in (("C", bc), ("f", bc), ("viol", bc), ("B", bb), ("nu", bb), ("lam", bl))}
            widened += any(tol[q] > bar for q, bar in (("C", bc), ("B", bb), ("lam", bl)))
            assert g["status"] == s["status"] and g["iters"] == s["iters"], (tag, g["status"], s["status"], g["iters"], s["iters"])
            assert np.array_equal(g["istate"], s["istate"]), (tag, g["istate"], s["istate"])
            # the step index the K-th line search chose, read off the GPU's steps
            st = ref["steps"][K - 1] if K - 1 < len(ref["steps"]) else None
            if st is not None:
                dg = g["C"] - (gpu[K - 1]["C"][p] if K > 1 else ref["C0"])
                dr = s["C"] - ref["snaps"][K - 1]["C"]
                if not st["accepted"]:
                    assert not dg.any(), (tag, "the GPU took a step the reference rejected")
                else:
                    ng, nrf = np.abs(dg).max(), np.abs(dr).max()
                    assert ng > 0, (tag, "the GPU rejected the step")
                    a_gpu = st["a"] + int(round(np.log2(nrf / ng)))
                    assert a_gpu == st["a"], (tag, "step index", a_gpu, st["a"])
            row = g["W"]
            assert row[0] == TAG and row[1] == nr and row[2] == red.m, tag
            got = dict(C=g["C"], f=g["f"], viol=g["viol"], B=row[6:].reshape(nr, nr), nu=row[5], lam=g["lam"])
            for q, v in got.items():
                assert rel_diff(v, s[q]) <= tol[q], (tag, q, rel_diff(v, s[q]), tol[q])
    assert drops * 20 <= max(len(refs), 20), (name, drops, len(refs))
    return drops, widened


@pytest.mark.parametrize("name", SETUPS)
def test_iterations_match_lockstep_reference(core, port, name):
    """cold solves stopped after K = 1..6 iterations: status, iterations, active set and the chosen step
    equal; C, f, violation, B, nu and the multipliers (eliminated equality rows included) within 1e-10 ..
    1e-7.  The warm row's header carries the digest of the restated basis: the reference's N is the
    library's N bit for bit."""
    from ntg_b200 import Problem
    spec, X, bounds = _setup(name)
    red = Reduced(port, spec)
    pb = Problem(spec, 0)
    assert not pb.fast
    if name == "kincar_tiled301":
        tile = pb.dims.band_tile
        assert tile < spec.nbps and spec.nbps % tile != 0, "the band Jacobian is stored in tiles, the last one shorter"
    gpu = {K: _gpu(pb, X, K, bounds) for K in KS}
    row = gpu[1]["W"][0]
    assert int(row[3]) + (int(row[4]) << 32) == red.digest(), "the restated basis is not the library's"
    refs = _references(core, red, X, bounds, max(KS))
    drops, widened = _compare(name, red, gpu, refs)
    print(f"{name}: nr {red.nr} m {red.m} P {X.shape[0]}: {drops} problems compared only up to a close decision, "
          f"{widened} comparisons held to their rounding spread")
    pb.close()


@pytest.mark.parametrize("name", ["kincar_bounds", "endpoint", "kincar_tiled301", "kincar_nr34", "hi_nr32"])
def test_warm_iterations_match_lockstep_reference(core, port, name):
    """the same comparison from a warm row an earlier call filled: the reference starts from that row's B
    and nu, at the point that call returned"""
    from ntg_b200 import Problem
    spec, X, bounds = _setup(name)
    red = Reduced(port, spec)
    pb = Problem(spec, 0)
    first = _gpu(pb, X, 3, bounds)
    X1, W1 = first["C"], first["W"]
    gpu = {K: _gpu(pb, X1, K, bounds, warm=W1) for K in KS}
    refs = _references(core, red, X1, bounds, max(KS), warm=W1)
    _compare(name + "_warm", red, gpu, refs)
    pb.close()


@pytest.mark.parametrize("name", ["endpoint", "kincar_bounds"])
def test_line_search_without_armijo_point(core, port, name):
    """c1 = 0.999 leaves most line searches without an Armijo point: stage 2 runs, and the step is the first
    strict minimum over both stages -- mostly one of stage 1, which k_alm_pick2 must keep"""
    from ntg_b200 import Problem
    spec, X, bounds = _setup(name)
    red = Reduced(port, spec)
    pb = Problem(spec, 0)
    gpu = {K: _gpu(pb, X, K, bounds, c1=0.999) for K in KS}
    refs = _references(core, red, X, bounds, max(KS), c1=0.999)
    kept = sum(s["stage2"] and s["a"] < 4 for r in refs for s in r["steps"])
    assert kept >= 3, kept
    _compare(name + "_c1", red, gpu, refs)
    pb.close()


@pytest.mark.parametrize("name", ["hi_nr32", "kincar_nr34", "hi_nr70"])
def test_cta_of_64_threads_is_deterministic(name):
    """nr >= 32 (two warps, cross-warp reductions; nr > 64 also gives threads several columns): repeated
    calls are bit-identical, a permuted batch gives permuted outputs, and checking for the end of the batch
    every iteration or every fourth gives the same bits -- finished problems do not change after they finish"""
    from ntg_b200 import Problem
    spec, X, _ = _setup(name)
    if X.shape[0] < 8:
        X = np.vstack([X, np.random.default_rng(11).uniform(-0.01, 0.01, (8 - X.shape[0], spec.nC))]) \
            if name.startswith("hi") else configs.coefficients("cfg3", 8, spec, seed=5)
    pb = Problem(spec, 0)

    def run(Xr, **kw):
        o = _gpu(pb, Xr, 250, None, **kw)
        return [o[k] for k in ("C", "f", "viol", "iters", "status", "lam", "istate", "W")]

    a = run(X)
    assert (a[4] == 1).mean() >= 0.75, a[4]
    for x, y in zip(a, run(X)):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    perm = np.random.default_rng(2).permutation(X.shape[0])
    for x, y in zip(a, run(X[perm])):
        assert np.array_equal(x[perm].view(np.uint8), y.view(np.uint8))
    for x, y in zip(run(X, check_every=1), run(X, check_every=4)):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    pb.close()


def test_shared_memory_limit(core, port):
    """the largest high-order shape whose CTA fits the device's opt-in shared memory solves and follows the
    reference; the next size up and endpoint(300) (m = 1207) are refused with C untouched"""
    import torch
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    limit = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    fam = {n: configs.high_order(4, 2, n, 81, name=f"lock_hi_n{n}") for n in range(20, 40)}   # nr = 2n + 2 < nbps
    fits = [n for n, s in fam.items() if sqp_smem_bytes(s.nC, s.nbps) <= limit]
    n = max(fits)
    assert n + 1 in fam and n + 1 not in fits, "the limit falls inside the family"
    spec = fam[n]
    red = Reduced(port, spec)
    assert red.nr == spec.nC and red.m == spec.nbps
    X = np.random.default_rng(1).uniform(-0.01, 0.01, (1, spec.nC))
    pb = Problem(spec, 0)
    gpu = {K: _gpu(pb, X, K, None) for K in KS}
    _compare(f"hi_n{n}", red, gpu, _references(core, red, X, None, max(KS)))
    Cd = _cuda(X)
    f, v, it, st = pb.solve_sqp(Cd, max_iter=400)
    assert int(st[0]) == 1
    pb.close()
    for spec in (fam[n + 1], configs.endpoint(300, name="lock_ep300")):
        X = np.random.default_rng(2).uniform(-0.5, 0.5, (3, spec.nC))
        pb = Problem(spec, 0)
        Cd = _cuda(X)
        with pytest.raises(NtgError, match="shared memory"):
            pb.solve_sqp(Cd)
        assert np.array_equal(Cd.cpu().numpy().view(np.int64), X.view(np.int64))
        pb.close()


def _hi_eq(order, mult, ninterv, name):
    """high_order without its nonlinear row, z(0) = 1 and z'(0) = 0.5 pinned: a convex quadratic cost under
    two linear equalities, nr = nC - 2"""
    import dataclasses
    base = configs.high_order(order, mult, ninterv, 33, name=name)
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(callbacks={"ucf": "hi20_ucf", "nltcf": ""}, nnltc=0, trajectoryconstrav=[],
              lic=np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]), lowerb=np.array([1.0, 0.5]), upperb=np.array([1.0, 0.5]))
    return type(base)(**kw)


def test_solve_eq_at_its_per_thread_limit(port):
    """k_solve_dir keeps kSolveMaxNr = 32 reduced variables per thread: nr = 32 reaches the minimiser of the
    quadratic (its KKT system solved with numpy), nr = 33 is refused"""
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    spec = _hi_eq(4, 2, 16, "lock_eq32")
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    assert nC - np.linalg.matrix_rank(A) == 32
    H = port.eval(spec, np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]   # g(C) = H C
    H = 0.5 * (H + H.T)
    K = np.block([[H, A.T], [A, np.zeros((A.shape[0], A.shape[0]))]])
    Cref = np.linalg.solve(K, np.concatenate([np.zeros(nC), b]))[:nC]
    fref = float(port.eval(spec, Cref[None, :], mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0])
    X = np.random.default_rng(4).uniform(-0.5, 0.5, (5, nC))
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    f, it, st = pb.solve_eq(Cd, max_iter=500)
    Cs = Cd.cpu().numpy()
    assert (st.cpu().numpy() != 0).all(), (st, it)   # converged, or no further decrease at rounding level
    assert np.abs(Cs @ A.T - b).max() <= 1e-10
    assert (np.abs(f.cpu().numpy() - fref) <= 1e-9 * max(1.0, abs(fref))).all(), (f, fref)
    assert np.abs(Cs - Cref).max() <= 1e-4 * max(1.0, np.abs(Cref).max()), np.abs(Cs - Cref).max()
    pb.close()
    spec = _hi_eq(5, 2, 11, "lock_eq33")
    assert spec.nC - 2 == 33
    pb = Problem(spec, 0)
    with pytest.raises(NtgError, match="33 free directions"):
        pb.solve_eq(_cuda(np.zeros((2, spec.nC))))
    pb.close()
