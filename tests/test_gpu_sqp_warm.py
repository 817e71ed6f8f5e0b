"""GPU tests of the SQP warm start (ntgb_solve_sqp_warm): solver state carried between calls in a
device array, one row per problem.  Rows that do not match the setup give exactly today's solver;
a re-solve at a solution stops at once, on this Problem or another one of the same setup; a receding-
horizon loop with active bounds reaches the cold loop's answers in fewer iterations; a real-time-
iteration loop (two SQP iterations per call) reaches the full solve; rows travel with their problems;
rejected problems keep their rows; bad arguments are refused."""
import dataclasses

import numpy as np
import pytest

from ntg_b200 import configs
from ntg_b200.abi import STATUS_BAD_BOUNDS

pytestmark = pytest.mark.gpu

HEADER = 6


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(ts):
    return [t.cpu().numpy() for t in ts]


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8)


def _same_bits(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _solve(pb, X, warm=None, lo=None, up=None, **kw):
    """-> [C, f, viol, iters, status, lambda, istate] as numpy; warm (device) is updated in place"""
    Cd = _cuda(X)
    b = {} if lo is None else {"lowerb": _cuda(lo), "upperb": _cuda(up)}
    res = pb.solve_sqp(Cd, multipliers=True, warm=warm, **b, **kw)
    return [Cd.cpu().numpy()] + _np(res)


def _spec_other_final_time():
    """_kincar_active_constraints over a shorter horizon: the same nr and m, another A (and N)"""
    from test_gpu_next import _kincar_active_constraints
    base = _kincar_active_constraints()
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(t1=0.9 * base.t1, knots=None, bps=None, name="warm_other_tf")
    return type(base)(**kw)


def _assert_filled(W, nr, m, rows):
    W = W[rows]
    assert (W[:, 0] == float(0x4E545731)).all() and (W[:, 1] == nr).all() and (W[:, 2] == m).all()
    assert (W[:, 3] == W[0, 3]).all() and (W[:, 4] == W[0, 4]).all()
    assert (W[:, 5] >= 0).all() and np.isfinite(W[:, HEADER:]).all()
    B = W[:, HEADER:].reshape(-1, nr, nr)
    assert np.array_equal(B, B.transpose(0, 2, 1))


# ---- 1. cold rows are today's solver -------------------------------------------------------------------

def test_cold_rows_are_todays_solver():
    from ntg_b200 import Problem
    from test_gpu_mpc import _active_specs
    spec, blo, bup = _active_specs(512, seed=3)
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=5)
    pb = Problem(spec, 0)
    n = pb.sqp_warm_doubles()
    nr, m = int(round(np.sqrt(n - HEADER))), pb.dims.ncnln   # every linear row of this setup is eliminated
    other = Problem(_spec_other_final_time(), 0)
    assert other.sqp_warm_doubles() == n
    Wo = other.sqp_warm_state(P)
    _solve(other, X, warm=Wo)
    foreign = Wo.cpu().numpy()
    garbage = np.random.default_rng(4).normal(size=(P, n))
    for lo, up in ((None, None), (blo, bup)):
        if lo is None:
            ref = _solve(pb, X)
        else:
            ref = _solve(pb, X, lo=lo, up=up)
        assert (ref[4] == 1).mean() >= 0.99
        for name, rows in (("zeros", np.zeros((P, n))), ("garbage", garbage), ("other setup", foreign)):
            W = _cuda(rows)
            got = _solve(pb, X, warm=W, lo=lo, up=up)
            for a, b in zip(got, ref):
                assert _same_bits(a, b), name
            Wn = W.cpu().numpy()
            _assert_filled(Wn, nr, m, np.arange(P))
            if name == "other setup":
                assert not (Wn[0, 3] == foreign[0, 3] and Wn[0, 4] == foreign[0, 4]), "digests differ"
    other.close()
    pb.close()


# ---- 2. re-solve at the solution ---------------------------------------------------------------------

def test_resolve_at_the_solution_stops_at_once():
    from ntg_b200 import Problem
    from test_gpu_mpc import _active_specs
    spec, blo, bup = _active_specs(512, seed=6)
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=7)
    pb = Problem(spec, 0)
    W = pb.sqp_warm_state(P)
    first = _solve(pb, X, warm=W, lo=blo, up=bup)
    Cs = first[0]
    rows = W.cpu().numpy()
    pb2 = Problem(spec, 0)
    for q in (pb, pb2):
        Wq = _cuda(rows)
        C2, f2, v2, it2, st2, _, _ = _solve(q, Cs, warm=Wq, lo=blo, up=bup)
        done = (st2 == 1) & (it2 == 0)
        assert done.mean() >= 0.99, (np.bincount(st2), np.bincount(it2))
        move = np.abs(C2 - Cs).max(axis=1) / np.maximum(1.0, np.abs(Cs).max(axis=1))
        assert (move[done] <= 1e-8).all(), move[done].max()
    pb2.close()
    pb.close()


# ---- 3. receding horizon with active bounds -----------------------------------------------------------

def test_receding_horizon_warm_vs_cold(port):
    import torch
    from ntg_b200 import Problem
    from test_gpu_mpc import _active_specs, _expand_lin, _expand_nl, _with_bounds
    from test_gpu_sqp import _kkt_residual
    spec, blo, bup = _active_specs(512, seed=11)
    P, steps, dt = 512, 5, 0.1
    X = configs.coefficients("cfg3", P, spec, seed=12)
    pb = Problem(spec, 0)
    tq = torch.tensor([dt], dtype=torch.float64, device="cuda")
    loops = {}
    for mode in ("cold", "warm"):
        Cd, lo, up = _cuda(X), _cuda(blo), _cuda(bup)
        W = pb.sqp_warm_state(P) if mode == "warm" else None
        per_step = []
        for k in range(steps):
            f, v, it, st, lam, ist = pb.solve_sqp(Cd, multipliers=True, lowerb=lo, upperb=up, warm=W)
            per_step.append(dict(C=Cd.cpu().numpy(), f=f.cpu().numpy(), it=it.cpu().numpy(), st=st.cpu().numpy(),
                                 lam=lam.cpu().numpy(), lo=lo.cpu().numpy(), up=up.cpu().numpy()))
            z = pb.spline_interp(Cd, tq)[:, 0, :]
            lo[:, :6] = z
            up[:, :6] = z
        loops[mode] = per_step
    its = {m: [int(s["it"].sum()) for s in loops[m]] for m in loops}
    for k in range(steps):
        for mode in loops:
            s = loops[mode][k]
            ok = s["st"] == 1
            assert ok.mean() >= 0.99, (mode, k, np.bincount(s["st"]))
            # KKT by the oracle against this loop's own bounds
            o = port.eval(spec, s["C"], mode_obj=0, mode_con=0, dense=False, band=False, linear=True)
            bl, nl_lo, nl_up = _expand_lin(spec, s["lo"]), _expand_nl(spec, s["lo"]), _expand_nl(spec, s["up"])
            lin = s["C"] @ o["A"].T
            assert (np.abs(lin - bl).max(axis=1)[ok] <= 1e-8 * (1 + np.abs(bl).max(axis=1)[ok])).all(), (mode, k)
            viol = np.maximum(np.maximum(nl_lo - o["c"], o["c"] - nl_up), 0).max(axis=1)
            assert (viol[ok] <= 1e-6).all(), (mode, k, viol[ok].max())
            for p in np.flatnonzero(ok)[[0, 9, 99]]:
                r, e = _kkt_residual(port, _with_bounds(spec, s["lo"][p], s["up"][p]), s["C"][p], s["lam"][p])
                assert np.abs(r).max() <= 1e-4 * max(1.0, np.abs(e["g"][0]).max()), (mode, k, p)
        c, w = loops["cold"][k], loops["warm"][k]
        agree = np.abs(w["f"] - c["f"]) <= 1e-6 * np.maximum(1.0, np.abs(c["f"]))
        assert agree.mean() >= 0.99, (k, np.abs(w["f"] - c["f"]).max())
    cold, warm = sum(its["cold"][1:]), sum(its["warm"][1:])
    print(f"receding horizon, {P} problems, iterations per step: cold {its['cold']}, warm {its['warm']}; "
          f"steps 2..{steps}: warm / cold = {warm / cold:.3f}")
    assert warm < cold
    pb.close()


# ---- 4. real-time iteration ------------------------------------------------------------------------

def test_real_time_iteration_reaches_the_full_solve():
    from ntg_b200 import Problem
    from test_gpu_mpc import _active_specs
    spec, blo, bup = _active_specs(512, seed=13)
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=14)
    pb = Problem(spec, 0)
    full = _solve(pb, X, lo=blo, up=bup)
    Cd, lo, up = _cuda(X), _cuda(blo), _cuda(bup)
    W = pb.sqp_warm_state(P)
    for calls in range(1, 21):
        f, v, it, st = _np(pb.solve_sqp(Cd, max_iter=2, lowerb=lo, upperb=up, warm=W))
        assert (it <= 2).all()
        if (st == 1).mean() >= 0.99:
            break
    print(f"real-time iteration (max_iter = 2): {calls} calls to reach status 1 on {(st == 1).mean():.3f}")
    assert (st == 1).mean() >= 0.99, np.bincount(st)
    both = (st == 1) & (full[4] == 1)
    assert both.mean() >= 0.98
    assert (np.abs(f - full[1])[both] <= 1e-7 * np.maximum(1.0, np.abs(full[1][both]))).all()
    pb.close()


# ---- 5. batch management -----------------------------------------------------------------------------

def test_rows_travel_with_their_problems():
    from ntg_b200 import Problem
    from test_gpu_mpc import _active_specs
    spec, blo, bup = _active_specs(512, seed=15)
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=16)
    pb = Problem(spec, 0)
    W = pb.sqp_warm_state(P)
    first = _solve(pb, X, warm=W, lo=blo, up=bup)
    # the next step: the initial states move, the carried rows go with their problems
    lo2, up2 = blo.copy(), bup.copy()
    z = pb.spline_interp(_cuda(first[0]), _cuda(np.array([0.1])))[:, 0, :].cpu().numpy()
    lo2[:, :6] = up2[:, :6] = z
    rows = W.cpu().numpy()
    Wa = _cuda(rows)
    a = _solve(pb, first[0], warm=Wa, lo=lo2, up=up2)
    perm = np.random.default_rng(17).permutation(P)
    Wp = _cuda(rows[perm])
    b = _solve(pb, first[0][perm], warm=Wp, lo=lo2[perm], up=up2[perm])
    for x, y in zip(b, a):
        assert _same_bits(x, y[perm])
    assert _same_bits(Wp.cpu().numpy(), Wa.cpu().numpy()[perm])
    # fresh zero rows among carried ones: the fresh problems get a cold solve of them alone
    fresh = np.zeros(P, dtype=bool)
    fresh[np.random.default_rng(18).choice(P, 64, replace=False)] = True
    mixed = rows.copy()
    mixed[fresh] = 0.0
    got = _solve(pb, first[0], warm=_cuda(mixed), lo=lo2, up=up2)
    alone = _solve(pb, first[0][fresh], lo=lo2[fresh], up=up2[fresh])
    for x, y in zip(got, alone):
        assert _same_bits(x[fresh], y)
    carried = _solve(pb, first[0][~fresh], warm=_cuda(rows[~fresh]), lo=lo2[~fresh], up=up2[~fresh])
    for x, y in zip(got, carried):
        assert _same_bits(x[~fresh], y)
    pb.close()


# ---- 6. rejected problems ----------------------------------------------------------------------------

def test_rejected_problems_keep_their_rows():
    from ntg_b200 import Problem
    from test_gpu_mpc import _active_specs
    spec, blo, bup = _active_specs(256, seed=19)
    P = 256
    X = configs.coefficients("cfg3", P, spec, seed=20)
    pb = Problem(spec, 0)
    W0 = pb.sqp_warm_state(P)
    start = _solve(pb, X, warm=W0, lo=blo, up=bup)[0]
    rows = W0.cpu().numpy()
    rows[5] = np.random.default_rng(21).normal(size=rows.shape[1])   # a row of garbage on a rejected problem
    Wg = _cuda(rows)
    good = _solve(pb, start, warm=Wg, lo=blo, up=bup)
    lo, up = blo.copy(), bup.copy()
    lo[3, 12], up[3, 12] = 70.0, 60.0        # lower > upper
    lo[5, 13] = np.nan                       # a NaN
    up[40, 4] = lo[40, 4] + 1e-9             # an eliminated row with lower != upper
    bad = [3, 5, 40]
    Wb = _cuda(rows)
    out = _solve(pb, start, warm=Wb, lo=lo, up=up)
    C_, f, v, it, st, lam, ist = out
    assert (st[bad] == STATUS_BAD_BOUNDS).all() and (it[bad] == 0).all()
    assert _same_bits(C_[bad], start[bad])
    Wb, Wg = Wb.cpu().numpy(), Wg.cpu().numpy()
    assert _same_bits(Wb[bad], rows[bad])
    keep = np.setdiff1d(np.arange(P), bad)
    for a, g in zip(out, good):
        assert _same_bits(a[keep], g[keep])
    assert _same_bits(Wb[keep], Wg[keep])
    pb.close()


# ---- 7. refusals -------------------------------------------------------------------------------------

def test_bad_arguments_are_refused():
    import torch
    from ntg_b200 import Problem
    from ntg_b200.problem import core
    from test_gpu_next import _kincar_active_constraints
    spec = _kincar_active_constraints()
    pb = Problem(spec, 0)
    P = 4
    Cd = _cuda(configs.coefficients("cfg3", P, spec, seed=22))
    C0 = Cd.clone()
    W = pb.sqp_warm_state(P)
    lo = _cuda(np.tile(spec.lowerb, (P, 1)))
    h, out = pb._h, [None] * 6 + [None]
    assert core().ntgb_solve_sqp_warm(h, P, Cd.data_ptr(), None, None, None, *out, None) == -1
    assert core().ntgb_solve_sqp_warm(h, P, Cd.data_ptr(), lo.data_ptr(), None, W.data_ptr(), *out, None) == -1
    assert core().ntgb_solve_sqp_warm(h, P, Cd.data_ptr(), None, lo.data_ptr(), W.data_ptr(), *out, None) == -1
    assert torch.equal(Cd, C0) and not W.any()
    n = pb.sqp_warm_doubles()
    for bad in (torch.zeros((P, n + 1), dtype=torch.float64, device="cuda"),
                torch.zeros((P + 1, n), dtype=torch.float64, device="cuda"),
                torch.zeros((P, n), dtype=torch.float32, device="cuda"),
                torch.zeros((n, P), dtype=torch.float64, device="cuda").t(),
                torch.zeros((P, n), dtype=torch.float64)):
        with pytest.raises(ValueError):
            pb.solve_sqp(Cd, warm=bad)
    pb.close()
