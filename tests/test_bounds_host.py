"""CPU checks of the per-problem bounds of ntgb_solve_eq_bounds / ntgb_solve_sqp_bounds
(ntg_b200/csrc/ntg_bounds.h, compiled with g++ through tests/tools/bounds_host.cpp -- the same text
k_bounds_prep runs with one warp per problem): the expansion of each problem's compact bounds into the
rows the solvers use equals, bit for bit, the oracle's bounds() for a setup carrying that problem's
bounds, and each rejection rule flags exactly the problem that breaks it.  The device half (the warp
split, Cpart on the GPU, the solvers) is checked in tests/test_gpu_mpc.py."""
import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np
import pytest

from ntg_b200 import configs

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

NAN_BIT, CROSSED_BIT, NOT_EQUAL_BIT, INCONSISTENT_BIT = 1, 2, 4, 8


@pytest.fixture(scope="module")
def bounds_bin(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("bounds") / "bounds_host")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "ntg_b200", "csrc"), "-o", exe,
                           os.path.join(HERE, "tools", "bounds_host.cpp")])
    return exe


def _with_bounds(spec, lo, up):
    kw = {f.name: getattr(spec, f.name) for f in dataclasses.fields(spec)}
    kw.update(lowerb=np.asarray(lo, dtype=np.float64).copy(), upperb=np.asarray(up, dtype=np.float64).copy())
    return type(spec)(**kw)


def _structure(spec):
    """the solvers' split of the expanded linear rows, from the SETUP's bounds (ntg_core.cu alm_prepare)"""
    nl = spec.nlic + spec.nltc + spec.nlfc
    rep = [1] * spec.nlic + [spec.nbps] * spec.nltc + [1] * spec.nlfc
    lo, up = np.repeat(spec.lowerb[:nl], rep), np.repeat(spec.upperb[:nl], rep)
    eq = np.flatnonzero(lo == up)
    li = np.flatnonzero(lo != up)
    return li, eq


def _min_norm_operator(Ae):
    """Cpart = M b on the independent rows (first occurrence), zero columns for the dependent ones"""
    me, nC = Ae.shape
    keep = []
    for r in range(me):
        if np.linalg.matrix_rank(Ae[keep + [r]], tol=1e-10) == len(keep) + 1:
            keep.append(r)
    M = np.zeros((nC, me))
    if keep:
        M[:, keep] = np.linalg.pinv(Ae[keep])
    return M


def run_bounds(exe, spec, li, eq, M, Ae, lo, up):
    """-> list of (bad, hl, hu, be, Cpart) per problem"""
    h = float.hex
    words = [spec.nlic, spec.nltc, spec.nlfc, spec.nnlic, spec.nnltc, spec.nnlfc, spec.nbps, spec.nC,
             len(li), *li, len(eq), *eq]
    txt = " ".join(str(int(w)) for w in words) + "\n"
    txt += " ".join(h(float(v)) for v in M.ravel()) + "\n" + " ".join(h(float(v)) for v in Ae.ravel()) + "\n"
    txt += f"{lo.shape[0]}\n"
    for p in range(lo.shape[0]):
        txt += " ".join(h(float(v)) for v in np.concatenate([lo[p], up[p]])) + "\n"
    out = subprocess.run([exe], input=txt, capture_output=True, text=True, check=True).stdout.split("\n")
    m, me, nC = len(li) + spec.ncnln, len(eq), spec.nC
    rows = []
    for line in out:
        if not line.strip():
            continue
        w = line.split()
        v = np.array([float.fromhex(x) for x in w[1:]])
        assert v.shape[0] == 2 * m + me + nC
        rows.append((int(w[0]), v[:m], v[m:2 * m], v[2 * m:2 * m + me], v[2 * m + me:]))
    assert len(rows) == lo.shape[0]
    return rows


def _endpoint_with_equalities():
    """configs.endpoint() (every row kind: linear and nonlinear initial / trajectory / final rows) with
    its second initial and its final linear rows turned into equalities, so that the setup both
    eliminates rows and keeps linear inequality rows"""
    spec = configs.endpoint()
    lo, up = spec.lowerb.copy(), spec.upperb.copy()
    for k in (1, 3, 4):           # lic[1], lfc[0], lfc[1]
        lo[k] = up[k] = 0.25 * k
    return _with_bounds(spec, lo, up)


def _random_bounds(spec, li, eq, P, seed):
    rng = np.random.default_rng(seed)
    nb = spec.nbounds
    nl = spec.nlic + spec.nltc + spec.nlfc
    eq_compact = set()
    rep = [1] * spec.nlic + [spec.nbps] * spec.nltc + [1] * spec.nlfc
    src = np.repeat(np.arange(nl), rep)
    for r in eq:
        eq_compact.add(int(src[r]))
    lo = rng.uniform(-5, 5, (P, nb))
    up = lo + rng.uniform(0.0, 3.0, (P, nb))
    for k in eq_compact:
        up[:, k] = lo[:, k]
    free = [k for k in range(nb) if k not in eq_compact]
    # some rows without a bound on one side (|b| >= 1e19)
    for p in range(P):
        k = free[p % len(free)]
        if p % 3 == 0:
            lo[p, k] = -1e20
        elif p % 3 == 1:
            up[p, k] = 1e20
    return lo, up


def test_expansion_matches_the_oracle_bounds_bit_for_bit(port, bounds_bin):
    spec = _endpoint_with_equalities()
    nC, nclin = spec.nC, spec.nclin
    li, eq = _structure(spec)
    assert len(li) > 0 and len(eq) > 0 and spec.nnlic and spec.nnltc and spec.nnlfc
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=0, dense=False, band=False, linear=True)
    Ae = o["A"][eq]
    M = _min_norm_operator(Ae)
    P = 24
    lo, up = _random_bounds(spec, li, eq, P, seed=11)
    rows = run_bounds(bounds_bin, spec, li, eq, M, Ae, lo, up)
    for p, (bad, hl, hu, be, Cp) in enumerate(rows):
        assert bad == 0, (p, bad)
        r = port.eval(_with_bounds(spec, lo[p], up[p]), np.zeros((1, nC)), mode_obj=0, mode_con=0, dense=False,
                      band=False, linear=True)
        bl, bu = r["bl"], r["bu"]
        want_hl = np.concatenate([bl[nC:nC + nclin][li], bl[nC + nclin:]])
        want_hu = np.concatenate([bu[nC:nC + nclin][li], bu[nC + nclin:]])
        assert np.array_equal(hl.view(np.int64), want_hl.view(np.int64)), p
        assert np.array_equal(hu.view(np.int64), want_hu.view(np.int64)), p
        assert np.array_equal(be.view(np.int64), bl[nC:nC + nclin][eq].view(np.int64)), p
        assert np.array_equal(be, bu[nC:nC + nclin][eq]), p
        # Cpart = M be solves the eliminated rows
        np.testing.assert_allclose(Cp, M @ be, rtol=1e-13, atol=1e-13)
        assert np.abs(Ae @ Cp - be).max() <= 1e-10 * (1 + np.abs(be).max())


def test_each_rejection_rule_flags_exactly_its_problem(port, bounds_bin):
    spec = _endpoint_with_equalities()
    nC = spec.nC
    li, eq = _structure(spec)
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=0, dense=False, band=False, linear=True)
    Ae = o["A"][eq]
    M = _min_norm_operator(Ae)
    P = 12
    lo, up = _random_bounds(spec, li, eq, P, seed=4)
    lin_ineq_compact = 0                                    # lic[0] is an inequality in this setup
    eq_compact = 1                                          # lic[1] is eliminated
    nl_compact = spec.nlic + spec.nltc + spec.nlfc + 2      # a nonlinear trajectory row
    lo[2, lin_ineq_compact], up[2, lin_ineq_compact] = 1.0, 0.5        # lower > upper
    lo[5, eq_compact], up[5, eq_compact] = 0.0, 1e-12                  # eliminated row, lower != upper
    lo[7, nl_compact] = np.nan                                         # NaN
    up[9, lin_ineq_compact] = np.nan                                   # NaN on the other side
    lo[10, nl_compact], up[10, nl_compact] = 3.0, 3.0                  # equal bounds on a kept row: fine
    rows = run_bounds(bounds_bin, spec, li, eq, M, Ae, lo, up)
    bad = [r[0] for r in rows]
    want = [0] * P
    want[2], want[5], want[7], want[9] = CROSSED_BIT, NOT_EQUAL_BIT, NAN_BIT, NAN_BIT
    assert bad == want


def test_inconsistent_equalities_of_dependent_rows(port, bounds_bin):
    """a setup whose initial rows contain a duplicate: per-problem right-hand sides that agree are
    fine, ones that disagree (beyond reduce_linear's 1e-8 (1 + |b|_inf)) are rejected"""
    base = configs.kincar(20, constraints=False, name="dup_kincar")
    lic = np.vstack([base.lic, base.lic[2:3]])
    lo = np.concatenate([base.lowerb[:6], base.lowerb[2:3], base.lowerb[6:]])
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(lic=lic, lowerb=lo.copy(), upperb=lo.copy())
    spec = type(base)(**kw)
    nC = spec.nC
    li, eq = _structure(spec)
    assert len(li) == 0 and len(eq) == spec.nclin == 13
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    Ae = o["A"][eq]
    M = _min_norm_operator(Ae)
    assert np.count_nonzero(np.abs(M).sum(axis=0) == 0) == 1, "the duplicate row is dependent"
    P = 6
    rng = np.random.default_rng(2)
    los = np.tile(lo, (P, 1))
    los[:, :6] += rng.uniform(-1, 1, (P, 6))
    los[:, 6] = los[:, 2]                                   # duplicate agrees ...
    los[1, 6] += 1e-3                                       # ... except in problem 1
    los[3, 6] += 1e-10 * (1 + np.abs(los[3]).max())         # within the tolerance: accepted
    los[4, 2] = -los[4, 2] - 7.0                            # both sides moved together: accepted
    los[4, 6] = los[4, 2]
    los[5, 2] = los[5, 6] = np.inf                          # "no bound" on an eliminated row: no solution
    rows = run_bounds(bounds_bin, spec, li, eq, M, Ae, los, los.copy())
    assert [r[0] for r in rows] == [0, INCONSISTENT_BIT, 0, 0, 0, INCONSISTENT_BIT]


def test_null_arguments_are_refused_before_cuda(built_libs):
    """without a device: a NULL problem / bounds pointer is NTGB_EINVAL, not a CUDA error"""
    from ntg_b200 import problem
    lib = problem.core()
    C_ = (C.c_double * 4)()
    for fn, extra in ((lib.ntgb_solve_eq_bounds, 5), (lib.ntgb_solve_sqp_bounds, 8)):
        assert fn(None, 4, C_, None, None, *([None] * extra)) == -1
        assert "null argument" in lib.ntgb_last_error().decode()
        assert fn(None, 4, None, C_, C_, *([None] * extra)) == -1
