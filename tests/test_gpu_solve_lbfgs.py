"""GPU tests of the projected L-BFGS solver (ntgb_solve_eq_lbfgs): the problems of ntgb_solve_eq with any number of
free directions.  Convex instances are checked against the solution of their KKT system (H from the oracle's
gradient at the identity columns, then [H A'; A 0]), the nonconvex van der Pol against the projected gradient
and scipy's SLSQP.  The per-iteration core is checked on the CPU in tests/test_lbfgs_host.py.

The spline costs' Hessians in the coefficients have condition numbers that grow like the fourth power of the
intervals per output (3e4 at 24, 2e6 at 64 for the lane change), and their evaluation rounds at about 1e-13 of
|f| (positions up to 40 against second derivatives near 1).  Near the solution no Armijo step of any length
then decreases the cost measurably, and the solver stops with status 2 before |P g| reaches gtol: "finished"
below is status 1 or 2, and the checks are on the point reached (the KKT solution, the projected gradient)."""
import dataclasses

import numpy as np
import pytest

from ntg_b200 import configs

pytestmark = pytest.mark.gpu

LANE_GTOL = 1e-6


def _finished(st):
    return (st == 1) | (st == 2)


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _long_kincar(ninterv=64, nbps=193, name="lbfgs_kincar64"):
    """the lane change of configs.kincar over ninterv intervals per output (64: nC = 262, nr = 250)"""
    return dataclasses.replace(configs.kincar(nbps, constraints=False, name=name), ninterv=[ninterv, ninterv],
                               knots=None)


def _kkt(port, spec, b=None):
    """-> (A, b, H, the KKT solution of the quadratic cost, its cost); asserts H > 0 on null(A)"""
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    A = o["A"]
    if b is None:
        b = o["bl"][nC:nC + spec.nclin]
    H = port.eval(spec, np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]   # g(C) = H C
    H = 0.5 * (H + H.T)
    Nb = np.linalg.svd(A)[2][np.linalg.matrix_rank(A):]
    assert np.linalg.eigvalsh(Nb @ H @ Nb.T).min() > 0.0
    K = np.block([[H, A.T], [A, np.zeros((A.shape[0], A.shape[0]))]])
    Cref = np.linalg.solve(K, np.concatenate([np.zeros(nC), b]))[:nC]
    fref = float(port.eval(spec, Cref[None, :], mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0])
    return A, b, H, Cref, fref


def _hi_eq(order, mult, ninterv, name):
    from test_gpu_sqp_lockstep import _hi_eq as h
    return h(order, mult, ninterv, name)


def test_at_the_old_limit_and_past_it(port):
    """nr = 32, the most ntgb_solve_eq takes: both solvers reach numpy's minimiser; nr = 33, which ntgb_solve_eq
    refuses, reaches its KKT point"""
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    spec = _hi_eq(4, 2, 16, "lbfgs_eq32")
    A, b, H, Cref, fref = _kkt(port, spec)
    assert spec.nC - np.linalg.matrix_rank(A) == 32
    X = np.random.default_rng(4).uniform(-0.5, 0.5, (5, spec.nC))
    pb = Problem(spec, 0)
    Cl, Ce = _cuda(X), _cuda(X)
    fl, itl, stl = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Cl, max_iter=5000))
    fe, ite, ste = (t.cpu().numpy() for t in pb.solve_eq(Ce, max_iter=500))
    assert _finished(stl).all(), (stl, itl)
    for f, Cs in ((fl, Cl.cpu().numpy()), (fe, Ce.cpu().numpy())):
        assert np.abs(Cs @ A.T - b).max() <= 1e-10
        assert (np.abs(f - fref) <= 1e-9 * max(1.0, abs(fref))).all(), (f, fref)
        assert np.abs(Cs - Cref).max() <= 1e-4 * max(1.0, np.abs(Cref).max())
    assert np.abs(fl - fe).max() <= 1e-9 * max(1.0, abs(fref))
    pb.close()

    spec = _hi_eq(5, 2, 11, "lbfgs_eq33")
    A, b, H, Cref, fref = _kkt(port, spec)
    assert spec.nC - np.linalg.matrix_rank(A) == 33
    pb = Problem(spec, 0)
    with pytest.raises(NtgError, match="33 free directions"):
        pb.solve_eq(_cuda(np.zeros((2, spec.nC))))
    Cd = _cuda(np.random.default_rng(5).uniform(-0.5, 0.5, (5, spec.nC)))
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Cd, max_iter=5000))
    Cs = Cd.cpu().numpy()
    assert _finished(st).all(), (st, it)
    assert np.abs(Cs @ A.T - b).max() <= 1e-10
    assert (np.abs(f - fref) <= 1e-9 * max(1.0, abs(fref))).all()
    assert np.abs(Cs - Cref).max() <= 1e-4 * max(1.0, np.abs(Cref).max())
    pb.close()


def test_long_lane_change_reaches_the_kkt_point(port):
    """2 x 64 intervals (nC = 262, 250 free directions), 512 random starts"""
    from ntg_b200 import Problem
    spec = _long_kincar()
    A, b, H, Cref, fref = _kkt(port, spec)
    assert spec.nC == 262 and spec.nC - np.linalg.matrix_rank(A) == 250
    P = 512
    pb = Problem(spec, 0)
    Cd = _cuda(configs.coefficients("cfg3", P, spec, seed=11))
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Cd, max_iter=40000, gtol=LANE_GTOL, memory=16))
    Cs = Cd.cpu().numpy()
    ok = _finished(st)
    assert ok.mean() >= 0.99, (np.bincount(st), it.max())
    assert np.abs(Cs @ A.T - b).max() <= 1e-10 * (1 + np.abs(b).max())
    ferr = np.abs(f - fref) / max(1.0, abs(fref))
    assert ferr[ok].max() <= 1e-9, ferr.max()
    cerr = np.abs(Cs - Cref).max(axis=1) / max(1.0, np.abs(Cref).max())
    assert cerr[ok].max() <= 1e-6, cerr.max()
    pb.close()


def test_nonconvex_van_der_pol(port):
    """van der Pol without its nonlinear row over 40 intervals (nC = 83, 80 free directions): a stationary point
    from every start, and SLSQP's cost from the same starts on a handful"""
    from scipy.optimize import minimize
    from ntg_b200 import Problem
    spec = dataclasses.replace(configs.vanderpol(121, constraints=False, name="lbfgs_vdp40"), ninterv=[40], knots=None)
    nC = spec.nC
    assert nC == 83
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    assert nC - np.linalg.matrix_rank(A) == 80
    Nb = np.linalg.svd(A)[2][np.linalg.matrix_rank(A):]
    P, gtol = 256, 1e-9
    pg_bar = 1e-5
    X = np.random.default_rng(7).uniform(-2.0, 2.0, (P, nC))
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Cd, max_iter=5000, gtol=gtol))
    Cs = Cd.cpu().numpy()
    ok = _finished(st)
    assert ok.mean() >= 0.99, (np.bincount(st), it.max())
    assert np.abs(Cs @ A.T - b).max() <= 1e-10 * (1 + np.abs(b).max())
    r = port.eval(spec, Cs, mode_obj=2, mode_con=-1, dense=False, band=False)
    pg = np.abs((r["g"] @ Nb.T) @ Nb).max(axis=1)
    pgr = pg / np.maximum(1.0, np.abs(r["f"]))
    assert pgr[ok].max() <= pg_bar, np.quantile(pgr[ok], [0.5, 0.99, 1.0])

    def fun(x):
        q = port.eval(spec, x[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        return float(q["f"][0]), q["g"][0]

    for p in np.flatnonzero(ok)[:4]:
        res = minimize(fun, X[p], jac=True, method="SLSQP",
                       constraints=[{"type": "eq", "fun": lambda x: A @ x - b, "jac": lambda x: A}],
                       options={"maxiter": 2000, "ftol": 1e-14})
        assert res.success, res.message
        assert abs(res.fun - f[p]) <= 1e-6 * max(1.0, abs(f[p])), (p, res.fun, f[p])
    pb.close()


def _lane_bounds(spec, P, seed):
    """per-problem lane changes: x0 / xf of configs.kincar moved per problem, lower == upper"""
    rng = np.random.default_rng(seed)
    lo = np.tile(spec.lowerb, (P, 1))
    lo[:, 0] += rng.uniform(-2.0, 2.0, P)       # x(0)
    lo[:, 3] += rng.uniform(-1.0, 1.0, P)       # y(0)
    lo[:, 6] += rng.uniform(-5.0, 5.0, P)       # x(T)
    lo[:, 9] += rng.uniform(-1.0, 1.0, P)       # y(T)
    return np.ascontiguousarray(lo), np.ascontiguousarray(lo.copy())


def test_per_problem_bounds(port):
    """1024 lane changes with their own x0 / xf against one Problem per set of bounds; replicated bounds against
    the shared ones; rejected bounds leave C untouched and the other problems exactly as without them"""
    from ntg_b200 import Problem
    spec = _long_kincar(16, 49, "lbfgs_kincar16")
    P = 1024
    lo, up = _lane_bounds(spec, P, 3)
    X = configs.coefficients("cfg3", P, spec, seed=13)
    kw = dict(max_iter=20000, gtol=LANE_GTOL)
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    f, it, st = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Cd, lowerb=_cuda(lo), upperb=_cuda(up), **kw))
    Cs = Cd.cpu().numpy()
    assert _finished(st).mean() >= 0.99, np.bincount(st)
    for p in (0, 1, 517, 1023):
        one = Problem(dataclasses.replace(spec, lowerb=lo[p], upperb=up[p], name=f"lbfgs_one{p}"), 0)
        Cp = _cuda(X[p:p + 1])
        f1, _, st1 = (t.cpu().numpy() for t in one.solve_eq_lbfgs(Cp, **kw))
        A, b, H, Cref, fref = _kkt(port, one.spec)
        assert _finished(st1).all()
        assert abs(f1[0] - f[p]) <= 1e-8 * max(1.0, abs(f1[0])), (p, f1[0], f[p])
        for Cx in (Cp.cpu().numpy()[0], Cs[p]):
            assert np.abs(Cx - Cref).max() <= 1e-6 * max(1.0, np.abs(Cref).max()), (p, np.abs(Cx - Cref).max())
        one.close()
    # replicated setup bounds = the shared-bounds call
    rep_lo = np.ascontiguousarray(np.tile(spec.lowerb, (8, 1)))
    C1, C2 = _cuda(X[:8]), _cuda(X[:8])
    f1, _, s1 = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(C1, **kw))
    f2, _, s2 = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(C2, lowerb=_cuda(rep_lo), upperb=_cuda(rep_lo), **kw))
    assert _finished(s1).all() and _finished(s2).all()
    assert np.abs(f1 - f2).max() <= 1e-8 * max(1.0, np.abs(f1).max())
    # rejected bounds: NaN, lower > upper, an eliminated row with lower != upper
    lo2, up2 = lo[:64].copy(), up[:64].copy()
    lo2[5, 2] = np.nan
    lo2[17, 4] = up2[17, 4] + 1.0
    up2[40, 7] += 0.5
    Ca, Cb = _cuda(X[:64]), _cuda(X[:64])
    fa, ia, sa = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Ca, lowerb=_cuda(lo[:64]), upperb=_cuda(up[:64]), **kw))
    fb, ib, sb = (t.cpu().numpy() for t in pb.solve_eq_lbfgs(Cb, lowerb=_cuda(lo2), upperb=_cuda(up2), **kw))
    bad = np.zeros(64, bool)
    bad[[5, 17, 40]] = True
    assert (sb[bad] == 5).all() and (ib[bad] == 0).all()
    Ca, Cb = Ca.cpu().numpy(), Cb.cpu().numpy()
    assert np.array_equal(Cb[bad].view(np.int64), X[:64][bad].view(np.int64))
    assert np.array_equal(Cb[~bad].view(np.int64), Ca[~bad].view(np.int64))
    assert np.array_equal(fb[~bad].view(np.int64), fa[~bad].view(np.int64))
    assert np.array_equal(ib[~bad], ia[~bad]) and np.array_equal(sb[~bad], sa[~bad])
    pb.close()


def _run(pb, X, **kw):
    Cd = _cuda(X)
    f, it, st = pb.solve_eq_lbfgs(Cd, **kw)
    return Cd.cpu().numpy(), f.cpu().numpy(), it.cpu().numpy(), st.cpu().numpy()


def _same(a, b):
    return all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(a, b))


def test_deterministic_across_calls_batches_and_problems():
    """two calls are bit-identical; permuting the batch permutes every output bit for bit; P = 3, 300, 3 on one
    Problem equals fresh Problems"""
    from ntg_b200 import Problem
    spec = _long_kincar(32, 97, "lbfgs_kincar32")
    kw = dict(max_iter=300, gtol=LANE_GTOL)
    X = configs.coefficients("cfg3", 300, spec, seed=17)
    pb = Problem(spec, 0)
    r1, r2 = _run(pb, X, **kw), _run(pb, X, **kw)
    assert _same(r1, r2)
    perm = np.random.default_rng(1).permutation(300)
    rp = _run(pb, X[perm], **kw)
    assert _same(rp, tuple(a[perm] for a in r1))
    pb.close()
    pb = Problem(spec, 0)
    seq = [_run(pb, X[:3], **kw), _run(pb, X, **kw), _run(pb, X[3:6], **kw)]
    pb.close()
    for Xi, got in zip((X[:3], X, X[3:6]), seq):
        fresh = Problem(spec, 0)
        assert _same(got, _run(fresh, Xi, **kw))
        fresh.close()


def test_cfg5_scale_without_a_dense_basis():
    """one output, 2000 intervals of order 4 (nC = 4002, 4000 free directions), 64 problems: the first call takes
    less device memory than a dense nC x nC basis would, stays on A C = b and lowers every cost by orders of
    magnitude.  The Hessian's condition number at 2000 intervals keeps plain L-BFGS from reaching gtol within
    the 3000 iterations run here (status 0)."""
    import torch
    from ntg_b200 import Problem
    spec = dataclasses.replace(_hi_eq(4, 2, 2000, "lbfgs_hi4002"), nbps=4001, bps=None)
    nC, P = spec.nC, 64
    assert nC == 4002
    pb = Problem(spec, 0)
    X = np.random.default_rng(19).uniform(-0.5, 0.5, (P, nC))
    Cd = _cuda(X)
    f0 = pb.eval(Cd, mode_obj=0, mode_con=-1, jac=0)["f"].cpu().numpy()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    f, it, st = pb.solve_eq_lbfgs(Cd, max_iter=3000, gtol=1e-6)
    torch.cuda.synchronize()
    used = free0 - torch.cuda.mem_get_info()[0]
    st, f = st.cpu().numpy(), f.cpu().numpy()
    assert used < nC * nC * 8, used
    assert np.isin(st, (0, 1, 2)).all(), np.bincount(st)
    assert (f < 1e-3 * f0).all(), (f / f0).max()
    A = pb.linear()
    Cs = Cd.cpu().numpy()
    assert np.abs(Cs @ A.T - np.array([1.0, 0.5])).max() <= 1e-10
    pb.close()


def test_refusals_and_sharing_the_reduced_form():
    """refusals as ntgb_solve_eq's; solve_eq_lbfgs, then solve_eq, then solve_sqp on one Problem equal the same
    calls on fresh Problems (they share the reduced form, and the L-BFGS call builds it without N)"""
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    from test_gpu_next import _kincar_active_constraints
    ineq = configs.kincar(20, constraints=False, name="lbfgs_ineq")
    ineq = dataclasses.replace(ineq, lowerb=ineq.lowerb - np.eye(12)[4], upperb=ineq.upperb + np.eye(12)[4])
    for spec, why in ((configs.kincar(20, constraints=True, name="lbfgs_nl"), "nonlinear constraints"),
                      (_kincar_active_constraints(), "nonlinear constraints"),
                      (ineq, "linear constraint 4 is not an equality")):
        pb = Problem(spec, 0)
        C = _cuda(np.zeros((2, spec.nC)))
        msgs = []
        for fn in (pb.solve_eq, pb.solve_eq_lbfgs):
            with pytest.raises(NtgError) as e:
                fn(C)
            msgs.append(str(e.value))
        assert why in msgs[0]
        assert msgs[1] == msgs[0].replace("ntgb_solve_eq:", "ntgb_solve_eq_lbfgs:")
        pb.close()
    spec = configs.kincar(64, constraints=False, name="lbfgs_share")
    X = configs.coefficients("cfg4", 40, spec, seed=23)
    calls = (lambda pb, C: pb.solve_eq_lbfgs(C, gtol=LANE_GTOL), lambda pb, C: pb.solve_eq(C),
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
    """equalities that pin every coefficient (z = 0.3 at 9 breakpoints of a 6-coefficient spline): C = C_part,
    status 1 and iters 0, bit for bit what ntgb_solve_eq returns, with shared and with per-problem bounds"""
    from ntg_b200 import Problem
    base = configs.high_order(4, 2, 2, 9, name="lbfgs_pinned")
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(callbacks={"ucf": "hi20_ucf", "nltcf": ""}, nnltc=0, trajectoryconstrav=[],
              ltc=np.array([[1.0, 0.0, 0.0]]), lowerb=np.array([0.3]), upperb=np.array([0.3]))
    spec = type(base)(**kw)
    pb = Problem(spec, 0)
    A = pb.linear()
    assert spec.nC == 6 and np.linalg.matrix_rank(A) == 6
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
        else:
            assert np.abs(got[0] - 0.3 * np.linalg.lstsq(A, np.ones(A.shape[0]), rcond=None)[0]).max() < 1e-12
    pb.close()
