"""GPU tests of the banded Newton solver (ntgb_solve_eq_newton): the problems of ntgb_solve_eq_lbfgs with a Hessian
from coloured gradient differences, factored per problem in band form.  Convex instances are checked against the
solution of their KKT system, the nonconvex van der Pol against the projected gradient and scipy's SLSQP.  The host
structure and the per-problem algebra are checked on the CPU in tests/test_newton_host.py.

"Finished" is status 1 or 2: on the long lane changes the cost stops resolving a decrease (rounding at about 1e-13
of |f|) before |P g| reaches gtol, and the solver then stops with status 2."""
import dataclasses

import numpy as np
import pytest

from ntg_b200 import configs
from test_gpu_solve_lbfgs import _cuda, _finished, _hi_eq, _kkt, _lane_bounds, _long_kincar, _same

pytestmark = pytest.mark.gpu


def _run(pb, X, **kw):
    Cd = _cuda(X)
    f, it, st = pb.solve_eq_newton(Cd, **kw)
    return Cd.cpu().numpy(), f.cpu().numpy(), it.cpu().numpy(), st.cpu().numpy()


def test_structure_of_the_lane_change():
    """K and w do not depend on the horizon; perm is a permutation"""
    from ntg_b200 import Problem
    for ni, nbps in ((8, 25), (64, 193), (256, 769)):
        pb = Problem(_long_kincar(ni, nbps, f"newton_struct{ni}"), 0)
        K, w, perm = pb.newton_structure()
        assert (K, w) == (18, 13)
        assert np.array_equal(np.sort(perm), np.arange(pb.spec.nC))
        pb.close()


@pytest.mark.parametrize("ninterv,nbps,P", [(64, 193, 512), (256, 769, 256)])
def test_long_lane_change_reaches_the_kkt_point(port, ninterv, nbps, P):
    """2 x 64 intervals (nC = 262) and 2 x 256 (nC = 1030): every start reaches the KKT cost to 1e-9 relative and
    C to 1e-6 of max |C|, on A C = b; at 64 intervals within a mean of 30 iterations"""
    from ntg_b200 import Problem
    spec = _long_kincar(ninterv, nbps, f"newton_kincar{ninterv}")
    A, b, H, Cref, fref = _kkt(port, spec)
    pb = Problem(spec, 0)
    Cd = _cuda(configs.coefficients("cfg3", P, spec, seed=11))
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_newton(Cd))
    Cs = Cd.cpu().numpy()
    assert _finished(st).all(), (np.bincount(st), it.max())
    assert np.abs(Cs @ A.T - b).max() <= 1e-10 * (1 + np.abs(b).max())
    ferr = np.abs(f - fref) / max(1.0, abs(fref))
    assert ferr.max() <= 1e-9, ferr.max()
    if ninterv == 64:
        cerr = np.abs(Cs - Cref).max(axis=1) / max(1.0, np.abs(Cref).max())
        assert cerr.max() <= 1e-6, cerr.max()
        assert it.mean() <= 30, (it.mean(), it.max())
    print(f"newton lane change 2 x {ninterv}: P {P} iters mean {it.mean():.2f} max {it.max()} status "
          f"{np.bincount(st).tolist()} max cost gap {ferr.max():.2e}")
    pb.close()


def test_nonconvex_van_der_pol(port):
    """van der Pol without its nonlinear row over 40 intervals (nC = 83): a stationary point from every start, and
    SLSQP's cost from the same starts on a handful"""
    from scipy.optimize import minimize
    from ntg_b200 import Problem
    spec = dataclasses.replace(configs.vanderpol(121, constraints=False, name="newton_vdp40"), ninterv=[40], knots=None)
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    Nb = np.linalg.svd(A)[2][np.linalg.matrix_rank(A):]
    P = 64
    X = np.random.default_rng(7).uniform(-2.0, 2.0, (P, nC))
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_newton(Cd))
    Cs = Cd.cpu().numpy()
    ok = _finished(st)
    assert ok.all(), (np.bincount(st), it.max())
    assert np.abs(Cs @ A.T - b).max() <= 1e-10 * (1 + np.abs(b).max())
    r = port.eval(spec, Cs, mode_obj=2, mode_con=-1, dense=False, band=False)
    pg = np.abs((r["g"] @ Nb.T) @ Nb).max(axis=1) / np.maximum(1.0, np.abs(r["f"]))
    assert pg.max() <= 1e-5, np.quantile(pg, [0.5, 0.99, 1.0])

    def fun(x):
        q = port.eval(spec, x[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        return float(q["f"][0]), q["g"][0]

    for p in range(4):
        res = minimize(fun, X[p], jac=True, method="SLSQP",
                       constraints=[{"type": "eq", "fun": lambda x: A @ x - b, "jac": lambda x: A}],
                       options={"maxiter": 2000, "ftol": 1e-14})
        assert res.success, res.message
        assert abs(res.fun - f[p]) <= 1e-6 * max(1.0, abs(f[p])), (p, res.fun, f[p])
    print(f"newton van der Pol 40: iters mean {it.mean():.2f} max {it.max()} status {np.bincount(st).tolist()}")
    pb.close()


def test_per_problem_bounds(port):
    """lane changes with their own x0 / xf against one Problem per set of bounds; replicated bounds against the
    shared ones; rejected bounds leave C untouched and the other problems exactly as without them"""
    from ntg_b200 import Problem
    spec = _long_kincar(16, 49, "newton_kincar16")
    P = 256
    lo, up = _lane_bounds(spec, P, 3)
    X = configs.coefficients("cfg3", P, spec, seed=13)
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_newton(Cd, lowerb=_cuda(lo), upperb=_cuda(up)))
    Cs = Cd.cpu().numpy()
    assert _finished(st).all(), np.bincount(st)
    for p in (0, 1, 117, 255):
        one = Problem(dataclasses.replace(spec, lowerb=lo[p], upperb=up[p], name=f"newton_one{p}"), 0)
        Cp = _cuda(X[p:p + 1])
        f1, _, st1 = (t.cpu().numpy() for t in one.solve_eq_newton(Cp))
        A, b, H, Cref, fref = _kkt(port, one.spec)
        assert _finished(st1).all()
        assert abs(f1[0] - f[p]) <= 1e-9 * max(1.0, abs(f1[0])), (p, f1[0], f[p])
        for Cx in (Cp.cpu().numpy()[0], Cs[p]):
            assert np.abs(Cx - Cref).max() <= 1e-6 * max(1.0, np.abs(Cref).max()), (p, np.abs(Cx - Cref).max())
        one.close()
    rep_lo = np.ascontiguousarray(np.tile(spec.lowerb, (8, 1)))
    C1, C2 = _cuda(X[:8]), _cuda(X[:8])
    f1, _, s1 = (t.cpu().numpy() for t in pb.solve_eq_newton(C1))
    f2, _, s2 = (t.cpu().numpy() for t in pb.solve_eq_newton(C2, lowerb=_cuda(rep_lo), upperb=_cuda(rep_lo)))
    assert _finished(s1).all() and _finished(s2).all()
    assert np.abs(f1 - f2).max() <= 1e-9 * max(1.0, np.abs(f1).max())
    lo2, up2 = lo[:64].copy(), up[:64].copy()
    lo2[5, 2] = np.nan
    lo2[17, 4] = up2[17, 4] + 1.0
    up2[40, 7] += 0.5
    Ca, Cb = _cuda(X[:64]), _cuda(X[:64])
    fa, ia, sa = (t.cpu().numpy() for t in pb.solve_eq_newton(Ca, lowerb=_cuda(lo[:64]), upperb=_cuda(up[:64])))
    fb, ib, sb = (t.cpu().numpy() for t in pb.solve_eq_newton(Cb, lowerb=_cuda(lo2), upperb=_cuda(up2)))
    bad = np.zeros(64, bool)
    bad[[5, 17, 40]] = True
    assert (sb[bad] == 5).all() and (ib[bad] == 0).all()
    Ca, Cb = Ca.cpu().numpy(), Cb.cpu().numpy()
    assert np.array_equal(Cb[bad].view(np.int64), X[:64][bad].view(np.int64))
    assert np.array_equal(Cb[~bad].view(np.int64), Ca[~bad].view(np.int64))
    assert np.array_equal(fb[~bad].view(np.int64), fa[~bad].view(np.int64))
    assert np.array_equal(ib[~bad], ia[~bad]) and np.array_equal(sb[~bad], sa[~bad])
    pb.close()


def test_deterministic_across_calls_batches_and_problems():
    """two calls are bit-identical; permuting the batch permutes every output bit for bit; P = 3, 300, 3 on one
    Problem equals fresh Problems"""
    from ntg_b200 import Problem
    spec = _long_kincar(32, 97, "newton_kincar32")
    X = configs.coefficients("cfg3", 300, spec, seed=17)
    pb = Problem(spec, 0)
    r1, r2 = _run(pb, X), _run(pb, X)
    assert _same(r1, r2)
    perm = np.random.default_rng(1).permutation(300)
    assert _same(_run(pb, X[perm]), tuple(a[perm] for a in r1))
    pb.close()
    pb = Problem(spec, 0)
    seq = [_run(pb, X[:3]), _run(pb, X), _run(pb, X[3:6])]
    pb.close()
    for Xi, got in zip((X[:3], X, X[3:6]), seq):
        fresh = Problem(spec, 0)
        assert _same(got, _run(fresh, Xi))
        fresh.close()


def test_long_single_output_without_a_dense_matrix():
    """one output, 2000 intervals of order 4 (nC = 4002), 64 problems: less device memory than nC^2 doubles, on
    A C = b, and the minimiser of the quadratic cost"""
    import torch
    from ntg_b200 import Problem
    spec = dataclasses.replace(_hi_eq(4, 2, 2000, "newton_hi4002"), nbps=4001, bps=None)
    nC, P = spec.nC, 64
    assert nC == 4002
    pb = Problem(spec, 0)
    X = np.random.default_rng(19).uniform(-0.5, 0.5, (P, nC))
    Cd = _cuda(X)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    f, it, st = pb.solve_eq_newton(Cd)
    torch.cuda.synchronize()
    used = free0 - torch.cuda.mem_get_info()[0]
    st, f, it = st.cpu().numpy(), f.cpu().numpy(), it.cpu().numpy()
    assert used < nC * nC * 8, used
    A = pb.linear()
    Cs = Cd.cpu().numpy()
    assert np.abs(Cs @ A.T - np.array([1.0, 0.5])).max() <= 1e-10
    print(f"newton hi4002: P {P} used {used / 2**20:.1f} MiB (nC^2 doubles: {nC * nC * 8 / 2**20:.1f} MiB) status "
          f"{np.bincount(st).tolist()} iters mean {it.mean():.2f} max {it.max()} f range {f.min():.6e} {f.max():.6e}")
    assert _finished(st).all(), np.bincount(st)
    assert np.abs(f - f[0]).max() <= 1e-9 * max(1.0, abs(f[0]))
    pb.close()


def _many_trajectory_rows(nbps=193):
    """the lane change with x'' = 0 at every breakpoint (x = 8 t is its one solution): about 130 independent
    equality rows on x, y still free"""
    spec = _long_kincar(64, nbps, "newton_rows")
    lo = np.concatenate([spec.lowerb[:6], [0.0], spec.lowerb[6:12]])
    return dataclasses.replace(spec, ltc=np.array([[0.0, 0.0, 1.0, 0.0, 0.0, 0.0]]), lowerb=lo, upperb=lo.copy())


def test_refusals_and_sharing_the_reduced_form(port):
    """refusals as ntgb_solve_eq's; r above 128 is NTGB_ELIMIT; solve_eq_newton, solve_eq_lbfgs, solve_eq and
    solve_sqp on one Problem equal the same calls on fresh Problems"""
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    from test_gpu_next import _kincar_active_constraints
    ineq = configs.kincar(20, constraints=False, name="newton_ineq")
    ineq = dataclasses.replace(ineq, lowerb=ineq.lowerb - np.eye(12)[4], upperb=ineq.upperb + np.eye(12)[4])
    for spec, why in ((configs.kincar(20, constraints=True, name="newton_nl"), "nonlinear constraints"),
                      (_kincar_active_constraints(), "nonlinear constraints"),
                      (ineq, "linear constraint 4 is not an equality")):
        pb = Problem(spec, 0)
        C = _cuda(np.zeros((2, spec.nC)))
        msgs = []
        for fn in (pb.solve_eq, pb.solve_eq_newton):
            with pytest.raises(NtgError) as e:
                fn(C)
            msgs.append(str(e.value))
        assert why in msgs[0]
        assert msgs[1] == msgs[0].replace("ntgb_solve_eq:", "ntgb_solve_eq_newton:")
        pb.close()
    spec = _many_trajectory_rows()
    pb = Problem(spec, 0)
    A = pb.linear()
    r = np.linalg.matrix_rank(A)
    assert 128 < r < spec.nC, r
    X = np.zeros((2, spec.nC))
    Cd = _cuda(X)
    with pytest.raises(NtgError, match=f"span {r} dimensions, above the limit of 128"):
        pb.solve_eq_newton(Cd)
    assert np.array_equal(Cd.cpu().numpy(), X)
    pb.close()
    spec = configs.kincar(64, constraints=False, name="newton_share")
    X = configs.coefficients("cfg4", 40, spec, seed=23)
    calls = (lambda pb, C: pb.solve_eq_newton(C), lambda pb, C: pb.solve_eq_lbfgs(C), lambda pb, C: pb.solve_eq(C),
             lambda pb, C: pb.solve_sqp(C))
    shared = Problem(spec, 0)
    for call in calls:
        Cs, Cf = _cuda(X), _cuda(X)
        a = [t.cpu().numpy() for t in call(shared, Cs)] + [Cs.cpu().numpy()]
        fresh = Problem(spec, 0)
        b = [t.cpu().numpy() for t in call(fresh, Cf)] + [Cf.cpu().numpy()]
        fresh.close()
        assert _same(a, b)
    shared.close()


def test_no_free_direction():
    """equalities that pin every coefficient: C = C_part, status 1 and iters 0, bit for bit what ntgb_solve_eq
    returns, with shared and with per-problem bounds"""
    from ntg_b200 import Problem
    base = configs.high_order(4, 2, 2, 9, name="newton_pinned")
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(callbacks={"ucf": "hi20_ucf", "nltcf": ""}, nnltc=0, trajectoryconstrav=[],
              ltc=np.array([[1.0, 0.0, 0.0]]), lowerb=np.array([0.3]), upperb=np.array([0.3]))
    spec = type(base)(**kw)
    pb = Problem(spec, 0)
    X = np.random.default_rng(29).uniform(-1.0, 1.0, (4, spec.nC))
    lo = np.array([[0.3], [0.5], [np.nan], [-0.2]])
    for bounds in ({}, {"lowerb": lo, "upperb": lo.copy()}):
        b = {k: _cuda(v) for k, v in bounds.items()}
        got = _run(pb, X, **b)
        Ce = _cuda(X)
        want = (Ce,) + tuple(pb.solve_eq(Ce, **b))
        want = tuple(t.cpu().numpy() for t in want)
        assert _same(got, want)
        st = got[3]
        assert (st[np.arange(4) != 2] == 1).all() and (got[2] == 0).all()
        if bounds:
            assert st[2] == 5 and np.array_equal(got[0][2].view(np.int64), X[2].view(np.int64))
    pb.close()
