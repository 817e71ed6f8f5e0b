"""GPU tests of the banded Newton solver iteration by iteration: ntgb_solve_eq_newton stopped after K = 1..Kmax
iterations against the same K iterations of the lock-step reference (tests/tools/newton_lockstep.py: the
library's reduced form restated bit for bit, the band assembled in numpy, the g++ build of ntg_newton.h's factor
and range-space step, the CPU oracle's evaluations, every CTA reduction in the CTA's order).  On the libm-free
packs every input of an iteration is reproducible, so C, f, iters and status must equal the reference bit for bit
at every K.  The end-result tests of
test_gpu_solve_newton.py cannot see a wrong band entry or a lost update of the factor: a Levenberg-Marquardt
Newton method with a line search converges with a wrong Hessian too, only more slowly.

The setups reach the band and row limits (w = 64 and 63, r = 128 and 127, r = 0, nC = w + 1), long rows
(nC = 1030), per-problem bounds with rejected problems, ragged grids (P = 129), the shifted refactorization, the
-P g fallback and both stopping rules.  The exact build is used throughout."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools"))
import newton_lockstep as nl  # noqa: E402

MARGIN = 1e-13


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    return nl.load_host(tmp_path_factory.mktemp("newton_lockstep_gpu"))


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _gpu(pb, X, K, bounds):
    Cd = _cuda(X)
    kw = {} if bounds is None else dict(lowerb=_cuda(bounds[0]), upperb=_cuda(bounds[1]))
    f, it, st = pb.solve_eq_newton(Cd, max_iter=K, **kw)
    return dict(C=Cd.cpu().numpy(), f=f.cpu().numpy(), iters=it.cpu().numpy(), status=st.cpu().numpy())


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _diagnose(nw, pb, gpu, ref, p, K, Cpart):
    """the first stage of iteration K that differs, from the device's own C_{K-1} (teacher-forced)"""
    import torch
    prev = ref["snaps"][K - 1]
    Cprev = gpu[K - 1]["C"][p] if K > 1 else prev["C"]
    if K > 1 and not np.array_equal(_bits(Cprev), _bits(prev["C"])):
        return f"C_{K - 1} already differs"
    st = nl.State(Cprev.copy(), prev["state"].tau, prev["state"].beta, prev["state"].stall, 0, prev["iters"])
    rec = {}
    want = nw.iterate(st, Cpart, rec)
    dev = pb.eval(torch.from_numpy(Cprev[None, :]).cuda())
    if not (np.array_equal(_bits(dev["f"].cpu().numpy()[0]), _bits(rec["f"]))
            and np.array_equal(_bits(dev["g"].cpu().numpy()[0]), _bits(rec["g"]))):
        return "f, g at C (the evaluator)"
    if "G" in rec:
        Gd = pb.eval(torch.from_numpy(nw.points(Cprev)).cuda())["g"].cpu().numpy()
        if not np.array_equal(_bits(Gd), _bits(rec["G"])):
            return "G (the evaluator at the difference points)"
    dC_dev, dC_ref = gpu[K]["C"][p] - Cprev, want.C - Cprev
    if "pick" in rec and rec["armijo"] and np.abs(dC_dev).max() > 0:
        a = rec["pick"] + int(round(np.log2(np.abs(dC_ref).max() / np.abs(dC_dev).max())))
        if a != rec["pick"]:
            return f"step index {a} against {rec['pick']} (margin {rec['margin']:.1e})"
        return f"d (C_K - C_K-1 off by {np.abs(dC_dev - dC_ref).max():.2e}) or the projection"
    if "pick" in rec and rec["armijo"] != bool(np.abs(dC_dev).max() > 0):
        return f"acceptance: the reference {'took' if rec['armijo'] else 'rejected'} the step (d or the search)"
    return (f"status / iters (device {gpu[K]['status'][p]}/{gpu[K]['iters'][p]}, "
            f"reference {want.status}/{want.iters})")


@pytest.mark.parametrize("name", nl.SETUPS)
def test_iterations_match_the_reference_bit_for_bit(lib, port, name):
    """C, f, iters and status after every K equal the reference's bits; the device's structure (K, w, perm)
    is the host's; a finished problem keeps its outputs bit for bit at every later K"""
    from ntg_b200 import Problem
    spec, X, bounds, rejected, Kmax = nl.setup(name)
    nw = nl.Newton(lib, port, spec)
    pb = Problem(spec, 0)
    assert not pb.fast
    K_, w_, perm = pb.newton_structure()
    assert (K_, w_) == (nw.s.K, nw.s.w) and np.array_equal(perm, nw.s.perm), (name, K_, w_)
    gpu = {K: _gpu(pb, X, K, bounds) for K in range(1, Kmax + 1)}
    refs = nl.references(nw, X, bounds, rejected, Kmax)
    drops, failures = 0, []
    for p, ref in enumerate(refs):
        Cp = None if bounds is None or p in rejected else nw.problem_cpart(bounds[0][p], bounds[1][p])
        for K in range(1, Kmax + 1):
            s = ref["snaps"][K]
            g = {k: v[p] for k, v in gpu[K].items()}
            same = (np.array_equal(_bits(g["C"]), _bits(s["C"])) and _bits(g["f"]) == _bits(s["f"])
                    and g["iters"] == s["iters"] and g["status"] == s["status"])
            if same:
                continue
            why = _diagnose(nw, pb, gpu, ref, p, K, Cp)
            close = min((r["margin"] for r in ref["recs"][:K] if "margin" in r), default=1.0)
            if why.startswith("step index") and close < MARGIN:
                drops += 1
            else:
                failures.append(f"{name} p={p} K={K}: {why}")
            break
    assert not failures, failures[:8]
    assert drops * 20 <= max(len(refs), 20), (name, drops)
    # finished problems stay put
    for K in range(2, Kmax + 1):
        done = gpu[K - 1]["status"] != 0
        for k in ("C", "f", "iters", "status"):
            a, b = gpu[K - 1][k][done], gpu[K][k][done]
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (name, K, k)
    if rejected:
        assert (gpu[Kmax]["status"][rejected] == 5).all()
        assert np.array_equal(_bits(gpu[Kmax]["C"][rejected]), _bits(X[rejected]))
    print(f"{name}: nC {spec.nC} K {nw.s.K} w {nw.s.w} r {nw.r} P {X.shape[0]} Kmax {Kmax}: bit for bit, "
          f"{drops} problems compared only up to a search decision within {MARGIN:g}; status at Kmax "
          f"{np.bincount(gpu[Kmax]['status']).tolist()}")
    pb.close()


def test_shapes_above_the_band_limit_are_refused(port):
    """w = 65 (syn6, order 7, mult 1, five cost outputs) and w = 67 (CFG-5's shape without its nonlinear rows):
    NTGB_ELIMIT with the half-bandwidth message, C untouched bit for bit"""
    import dataclasses
    from ntg_b200 import Problem, configs
    from ntg_b200.problem import NtgError
    cfg5 = dataclasses.replace(configs.syn6(200), callbacks={"ucf": "syn6_ucf", "nltcf": ""}, nnltc=0,
                               trajectoryconstrav=[], name="nl_cfg5_eq")
    for spec, w in ((nl.syn6_eq(7, 1, 4, range(5), "nl_syn6_w65"), 65), (cfg5, 67)):
        pb = Problem(spec, 0)
        X = np.random.default_rng(3).uniform(-1.0, 1.0, (3, spec.nC))
        Cd = _cuda(X)
        with pytest.raises(NtgError, match=f"half-bandwidth {w} is above the limit of 64"):
            pb.solve_eq_newton(Cd)
        assert np.array_equal(_bits(Cd.cpu().numpy()), _bits(X))
        pb.close()
