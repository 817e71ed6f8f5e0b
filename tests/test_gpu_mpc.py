"""GPU tests of the per-problem bounds of the batched solvers (ntgb_solve_eq_bounds,
ntgb_solve_sqp_bounds): a batch of MPC problems that share the setup but each start from their own
state.  Replicated bounds give the shared-bounds answer; distinct states and limits give each problem
its own solution (checked by the oracle and against one Problem per set of bounds); rejected bounds
leave their problem untouched and the others unchanged; and the receding-horizon loop runs with the
bounds kept on the device."""
import dataclasses

import numpy as np
import pytest

from ntg_b200 import configs
from ntg_b200.abi import STATUS_BAD_BOUNDS

pytestmark = pytest.mark.gpu


def _with_bounds(spec, lo, up, name=None):
    kw = {f.name: getattr(spec, f.name) for f in dataclasses.fields(spec)}
    kw.update(lowerb=np.asarray(lo, dtype=np.float64).copy(), upperb=np.asarray(up, dtype=np.float64).copy())
    if name:
        kw["name"] = name
    return type(spec)(**kw)


def _lane_changes(P, seed):
    """per-problem compact bounds of the kinematic-car lane change (configs.kincar, no nonlinear rows):
    initial / final flat state [x, x', x'', y, y', y''], seeded speeds and lateral offsets"""
    rng = np.random.default_rng(seed)
    v0, vf = rng.uniform(6.0, 10.0, P), rng.uniform(6.0, 10.0, P)
    y0, yf = rng.uniform(-3.0, -1.0, P), rng.uniform(1.0, 3.0, P)
    z = np.zeros(P)
    xf = 5.0 * 0.5 * (v0 + vf) + rng.uniform(-2.0, 2.0, P)
    b = np.stack([z, v0, z, y0, z, z, xf, vf, z, yf, z, z], axis=1)
    return np.ascontiguousarray(b)


def _expand_lin(spec, b):
    """compact [P][nb] -> the expanded linear rows [P][nclin]"""
    nl = spec.nlic + spec.nltc + spec.nlfc
    rep = [1] * spec.nlic + [spec.nbps] * spec.nltc + [1] * spec.nlfc
    return np.repeat(b[:, :nl], rep, axis=1)


def _expand_nl(spec, b):
    nl = spec.nlic + spec.nltc + spec.nlfc
    rep = [1] * spec.nnlic + [spec.nbps] * spec.nnltc + [1] * spec.nnlfc
    return np.repeat(b[:, nl:], rep, axis=1)


def _active_specs(P, seed):
    """_kincar_active_constraints with per-problem bounds: its lane change scaled by s (x and y), so that
    with the speed^2 limit 66.2 s^2 drawn in [60, 66.2] and the curvature limit 7.2 s^2 every problem
    stays feasible with its bounds active; lateral start perturbed a little on top"""
    from test_gpu_next import _kincar_active_constraints
    spec = _kincar_active_constraints()
    rng = np.random.default_rng(seed)
    L = rng.uniform(60.0, 66.2, P)
    s2 = L / 66.2
    s = np.sqrt(s2)
    lo = np.tile(spec.lowerb, (P, 1))
    up = np.tile(spec.upperb, (P, 1))
    lo[:, :12] *= s[:, None]
    lo[:, 3] += rng.uniform(-0.05, 0.05, P)
    up[:, :12] = lo[:, :12]
    up[:, 12] = L
    lo[:, 13], up[:, 13] = -7.2 * s2, 7.2 * s2
    return spec, np.ascontiguousarray(lo), np.ascontiguousarray(up)


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---- 1. replicated bounds give the shared-bounds answer ---------------------------------------------

def test_replicated_bounds_eq_match_shared():
    from ntg_b200 import Problem
    spec = configs.kincar(64, constraints=False, name="mpc_rep_eq")
    P = 4096
    X = configs.coefficients("cfg4", P, spec, seed=21)
    pb = Problem(spec, 0)
    Ca, Cb = _cuda(X), _cuda(X)
    fa, ia, sa = pb.solve_eq(Ca)
    lo, up = _cuda(np.tile(spec.lowerb, (P, 1))), _cuda(np.tile(spec.upperb, (P, 1)))
    fb, ib, sb = pb.solve_eq(Cb, lowerb=lo, upperb=up)
    Ca, Cb = Ca.cpu().numpy(), Cb.cpu().numpy()
    assert np.array_equal(sa.cpu().numpy(), sb.cpu().numpy())
    assert (np.abs(Ca - Cb).max(axis=1) <= 1e-9 * (1 + np.abs(Ca).max(axis=1))).all()
    fa, fb = fa.cpu().numpy(), fb.cpu().numpy()
    assert (np.abs(fa - fb) <= 1e-10 * np.abs(fa)).all()
    pb.close()


def test_replicated_bounds_sqp_match_shared():
    from ntg_b200 import Problem
    from test_gpu_next import _kincar_active_constraints
    spec = _kincar_active_constraints()
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=5)
    pb = Problem(spec, 0)
    Ca, Cb = _cuda(X), _cuda(X)
    fa, va, ia, sa, la, ista = pb.solve_sqp(Ca, multipliers=True)
    lo, up = _cuda(np.tile(spec.lowerb, (P, 1))), _cuda(np.tile(spec.upperb, (P, 1)))
    fb, vb, ib, sb, lb, istb = pb.solve_sqp(Cb, multipliers=True, lowerb=lo, upperb=up)
    assert np.array_equal(sa.cpu().numpy(), sb.cpu().numpy())
    fa, fb = fa.cpu().numpy(), fb.cpu().numpy()
    assert (np.abs(fa - fb) <= 1e-7 * np.maximum(1.0, np.abs(fa))).all()
    ok = sa.cpu().numpy() == 1
    assert np.array_equal(ista.cpu().numpy()[ok], istb.cpu().numpy()[ok])
    pb.close()


def test_null_bounds_are_refused():
    import torch
    from ntg_b200 import Problem
    from ntg_b200.problem import core
    spec = configs.kincar(20, constraints=False, name="mpc_null")
    pb = Problem(spec, 0)
    Cd = torch.zeros((4, spec.nC), dtype=torch.float64, device="cuda")
    lo = _cuda(np.tile(spec.lowerb, (4, 1)))
    assert core().ntgb_solve_eq_bounds(pb._h, 4, Cd.data_ptr(), None, lo.data_ptr(), None, None, None, None, None) == -1
    assert core().ntgb_solve_sqp_bounds(pb._h, 4, Cd.data_ptr(), lo.data_ptr(), None,
                                        *([None] * 8)) == -1
    with pytest.raises(ValueError):
        pb.solve_eq(Cd, lowerb=lo)
    pb.close()


# ---- 2. distinct initial and final states (eq) ------------------------------------------------------

def test_distinct_states_eq(port):
    from ntg_b200 import Problem
    spec = configs.kincar(64, constraints=False, name="mpc_eq")
    nC, P = spec.nC, 4096
    b = _lane_changes(P, seed=7)
    X = configs.coefficients("cfg4", P, spec, seed=8)
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    lo, up = _cuda(b), _cuda(b)
    f, it, st = pb.solve_eq(Cd, lowerb=lo, upperb=up)
    Cs, f, it, st = Cd.cpu().numpy(), f.cpu().numpy(), it.cpu().numpy(), st.cpu().numpy()
    assert (st == 1).all(), np.bincount(st)
    o = port.eval(spec, Cs, mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    be = _expand_lin(spec, b)
    res = np.abs(Cs @ o["A"].T - be).max(axis=1)
    assert (res <= 1e-8 * (1 + np.abs(be).max(axis=1))).all(), res.max()
    np.testing.assert_allclose(f, o["f"], rtol=1e-12)
    # one Problem per set of bounds, the shared-bounds solver: the same minimiser (convex quadratic)
    for p in np.random.default_rng(1).choice(P, 8, replace=False):
        q = Problem(_with_bounds(spec, b[p], b[p], name=f"mpc_eq_{p}"), 0)
        C1 = _cuda(X[p:p + 1])
        f1, _, s1 = q.solve_eq(C1)
        assert int(s1[0]) == 1
        assert np.abs(C1.cpu().numpy()[0] - Cs[p]).max() <= 1e-8 * (1 + np.abs(Cs[p]).max())
        q.close()
    # permuting the batch permutes every output bit for bit
    perm = np.random.default_rng(2).permutation(P)
    Cp = _cuda(X[perm])
    fp, itp, stp = pb.solve_eq(Cp, lowerb=_cuda(b[perm]), upperb=_cuda(b[perm]))
    assert np.array_equal(Cp.cpu().numpy().view(np.int64), Cs[perm].view(np.int64))
    assert np.array_equal(fp.cpu().numpy().view(np.int64), f[perm].view(np.int64))
    assert np.array_equal(itp.cpu().numpy(), it[perm]) and np.array_equal(stp.cpu().numpy(), st[perm])
    pb.close()


# ---- 3. distinct bounds with active nonlinear rows (SQP) -------------------------------------------

def test_distinct_bounds_sqp(port):
    from ntg_b200 import Problem
    from test_gpu_sqp import _kkt_residual
    spec, blo, bup = _active_specs(512, seed=3)
    nC, P, nclin = spec.nC, 512, spec.nclin
    X = configs.coefficients("cfg3", P, spec, seed=5)
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    f, v, it, st, lam, ist = pb.solve_sqp(Cd, multipliers=True, lowerb=_cuda(blo), upperb=_cuda(bup))
    Cs, f, v, it, st, lam, ist = (t.cpu().numpy() for t in (Cd, f, v, it, st, lam, ist))
    ok = st == 1
    assert ok.mean() >= 0.99, np.bincount(st)
    o = port.eval(spec, Cs, mode_obj=0, mode_con=0, dense=False, band=False, linear=True)
    bl, bu = _expand_lin(spec, blo), _expand_lin(spec, bup)
    nl_lo, nl_up = _expand_nl(spec, blo), _expand_nl(spec, bup)
    lin = Cs @ o["A"].T
    assert (np.abs(lin - bl).max(axis=1)[ok] <= 1e-8 * (1 + np.abs(bl).max(axis=1)[ok])).all()
    viol = np.maximum(np.maximum(nl_lo - o["c"], o["c"] - nl_up), 0).max(axis=1)
    assert (viol[ok] <= 1e-6).all(), viol[ok].max()
    assert (o["c"][ok][:, spec.nbps:].max(axis=1) > 0.99 * nl_up[ok][:, -1]).all(), "curvature bounds active"
    for p in np.flatnonzero(ok)[:6]:
        sp = _with_bounds(spec, blo[p], bup[p])
        r, e = _kkt_residual(port, sp, Cs[p], lam[p])
        assert np.abs(r).max() <= 1e-4 * max(1.0, np.abs(e["g"][0]).max()), (p, np.abs(r).max())
        ln, sn, cn = lam[p][nclin:], ist[p][nclin:], e["c"][0]
        assert (ist[p][:nclin] == 3).all()
        assert (np.abs(cn - nl_lo[p])[sn == 1] <= 1e-6).all() and (np.abs(cn - nl_up[p])[sn == 2] <= 1e-6).all()
        assert (ln[sn == 1] >= 0).all() and (ln[sn == 2] <= 0).all() and (ln[sn == 0] == 0).all()
        assert (sn != 0).sum() >= 1
    # one Problem per set of bounds, the shared-bounds solver
    for p in np.flatnonzero(ok)[[0, 7, 31, 101]]:
        q = Problem(_with_bounds(spec, blo[p], bup[p], name=f"mpc_sqp_{p}"), 0)
        C1 = _cuda(X[p:p + 1])
        f1, v1, i1, s1, l1, is1 = q.solve_sqp(C1, multipliers=True)
        assert int(s1[0]) == 1
        assert abs(float(f1[0]) - f[p]) <= 1e-7 * max(1.0, abs(f[p]))
        assert np.array_equal(is1.cpu().numpy()[0], ist[p])
        q.close()
    pb.close()


# ---- 4. rejected bounds -----------------------------------------------------------------------------

def _outputs(res, Cd):
    return [Cd.cpu().numpy()] + [t.cpu().numpy() for t in res]


def test_rejected_bounds_sqp():
    from ntg_b200 import Problem
    spec, blo, bup = _active_specs(256, seed=9)
    P = 256
    X = configs.coefficients("cfg3", P, spec, seed=10)
    pb = Problem(spec, 0)
    good = _outputs(pb.solve_sqp(Cg := _cuda(X), multipliers=True, lowerb=_cuda(blo), upperb=_cuda(bup)), Cg)
    lo, up = blo.copy(), bup.copy()
    lo[3, 12], up[3, 12] = 70.0, 60.0        # lower > upper on the speed row (an inequality)
    up[17, 4] = lo[17, 4] + 1e-9             # an eliminated row with lower != upper
    lo[40, 13] = np.nan                      # a NaN
    bad = [3, 17, 40]
    out = _outputs(pb.solve_sqp(Cb := _cuda(X), multipliers=True, lowerb=_cuda(lo), upperb=_cuda(up)), Cb)
    C_, f, v, it, st, lam, ist = out
    assert (st[bad] == STATUS_BAD_BOUNDS).all() and (it[bad] == 0).all() and np.isnan(v[bad]).all()
    assert (lam[bad] == 0).all() and (ist[bad] == 0).all()
    assert np.array_equal(C_[bad].view(np.int64), X[bad].view(np.int64))
    keep = np.setdiff1d(np.arange(P), bad)
    for a, g in zip(out, good):
        assert np.array_equal(a[keep].view(np.uint8), g[keep].view(np.uint8))
    pb.close()


def test_rejected_bounds_eq_dependent_rows():
    """a setup with a duplicated initial row: a problem whose duplicate right-hand sides disagree is
    rejected; the other problems are unchanged"""
    from ntg_b200 import Problem
    base = configs.kincar(64, constraints=False, name="mpc_dup")
    lic = np.vstack([base.lic, base.lic[3:4]])
    b0 = np.concatenate([base.lowerb[:6], base.lowerb[3:4], base.lowerb[6:]])
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(lic=lic, lowerb=b0.copy(), upperb=b0.copy())
    spec = type(base)(**kw)
    P = 512
    lc = _lane_changes(P, seed=12)
    b = np.concatenate([lc[:, :6], lc[:, 3:4], lc[:, 6:]], axis=1)
    X = configs.coefficients("cfg4", P, spec, seed=13)
    pb = Problem(spec, 0)
    good = _outputs(pb.solve_eq(Cg := _cuda(X), lowerb=_cuda(b), upperb=_cuda(b)), Cg)
    assert (good[3] == 1).all()
    b2 = b.copy()
    b2[[5, 300], 6] += 0.5                   # duplicate disagrees
    b2[9, 3] = np.inf                        # |b| = inf on an eliminated row: residual inf, rejected
    b2[9, 6] = np.inf
    bad = [5, 9, 300]
    out = _outputs(pb.solve_eq(Cb := _cuda(X), lowerb=_cuda(b2), upperb=_cuda(b2)), Cb)
    C_, f, it, st = out
    assert (st[bad] == STATUS_BAD_BOUNDS).all() and (it[bad] == 0).all()
    assert np.array_equal(C_[bad].view(np.int64), X[bad].view(np.int64))
    keep = np.setdiff1d(np.arange(P), bad)
    for a, g in zip(out, good):
        assert np.array_equal(a[keep].view(np.uint8), g[keep].view(np.uint8))
    pb.close()


# ---- 5. receding horizon on the device --------------------------------------------------------------

def test_receding_horizon_on_device(port):
    import torch
    from ntg_b200 import Problem
    spec = configs.kincar(64, constraints=False, name="mpc_rh")
    P, steps, dt = 1024, 5, 0.1
    b = _lane_changes(P, seed=31)
    X = configs.coefficients("cfg4", P, spec, seed=32)
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    lo, up = _cuda(b), _cuda(b)
    tq = torch.tensor([dt], dtype=torch.float64, device="cuda")
    A = port.eval(spec, np.zeros((1, spec.nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)["A"]
    prev_state = None
    for k in range(steps):
        f, it, st = pb.solve_eq(Cd, lowerb=lo, upperb=up)
        assert bool((st == 1).all()), np.bincount(st.cpu().numpy())
        Cs = Cd.cpu().numpy()
        bh = lo.cpu().numpy()
        be = _expand_lin(spec, bh)
        assert (np.abs(Cs @ A.T - be).max(axis=1) <= 1e-8 * (1 + np.abs(be).max(axis=1))).all()
        if prev_state is not None:
            # the initial rows of this solution are the previous solution's state at dt
            got = Cs @ A[:6].T
            assert (np.abs(got - prev_state).max(axis=1) <= 1e-9 * (1 + np.abs(prev_state).max(axis=1))).all()
        # previous state at dt by the oracle's SplineInterp, for the next step's check
        prev_state = np.empty((P, 6))
        for p in range(P):
            for j in range(2):
                c = Cs[p, j * 7:(j + 1) * 7]
                prev_state[p, 3 * j:3 * j + 3] = port.spline_interp(dt, spec.knots[j], c, 5, 3, 3)
        # the device-resident update: flat state at dt -> rows 0..5 of the bounds, no host round trip
        z = pb.spline_interp(Cd, tq)[:, 0, :]
        lo[:, :6] = z
        up[:, :6] = z
        assert np.allclose(z.cpu().numpy(), prev_state, rtol=1e-12, atol=1e-12)
    pb.close()
