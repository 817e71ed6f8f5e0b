"""CPU checks of the lock-step reference of the banded Newton solver (tests/tools/newton_lockstep.py), which
tests/test_gpu_newton_lockstep.py compares ntgb_solve_eq_newton with bit for bit: its row-space basis, its
agreement with the restated solve of test_newton_host.py, its numpy assemble against the header's, the KKT point on
the convex setups, the shape of every setup (so that the GPU test is known to reach the band and row limits before
it runs) and the paths the setups take between them."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools"))
import newton_lockstep as nl  # noqa: E402
from sqp_lockstep import reduce_linear  # noqa: E402


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    return nl.load_host(tmp_path_factory.mktemp("newton_lockstep"))


@pytest.fixture(scope="module")
def refs(lib, port):
    """every setup's reference, to its Kmax"""
    out = {}
    for name in nl.SETUPS:
        spec, X, bounds, rejected, K = nl.setup(name)
        nw = nl.Newton(lib, port, spec)
        out[name] = (nw, nl.references(nw, X, bounds, rejected, K))
    return out


@pytest.mark.parametrize("name", ["lane64", "rows128", "syn6_w63"])
def test_row_space_basis(port, name):
    """Q1 is orthonormal and spans the equality rows, Q1 and N make one orthonormal Q, and A Cpart = b.  (That
    these are the library's bits is checked on the device, through the bit-equal projections.)"""
    spec = nl.setup(name)[0]
    A, b, _ = nl.eq_rows(port, spec)
    N, Cpart, _, r, Q1 = reduce_linear(A, b, q1=True)
    assert r == np.linalg.matrix_rank(A) and Q1.shape == (r, spec.nC)
    assert np.abs(Q1 @ Q1.T - np.eye(r)).max() <= 1e-14
    assert np.abs(A - (A @ Q1.T) @ Q1).max() <= 1e-14 * np.abs(A).max() * A.shape[1]
    Q = np.vstack([Q1, N])
    assert Q.shape == (spec.nC, spec.nC)
    assert np.abs(Q @ Q.T - np.eye(spec.nC)).max() <= 1e-14
    assert np.abs(A @ Cpart - b).max() <= 1e-14 * np.abs(A).sum(axis=1).max() * max(1.0, np.abs(Cpart).max())


@pytest.mark.parametrize("name", nl.SETUPS)
def test_setup_shapes(lib, port, name):
    """nC, colours, half-bandwidth and row rank of every setup; the limits are reached: w = 64 (kMaxHalfBand, a
    window of 65^2 doubles), r = 128 (kMaxRows: 129 right-hand sides on 128 threads) and r = 0"""
    spec = nl.setup(name)[0]
    nw = nl.Newton(lib, port, spec)
    assert (spec.nC, nw.s.K, nw.s.w, nw.r) == nl.SHAPES[name]
    assert nw.r == (np.linalg.matrix_rank(nw.A) if nw.A.shape[0] else 0)
    assert max(s[2] for s in nl.SHAPES.values()) == 64 and max(s[3] for s in nl.SHAPES.values()) == 128


@pytest.mark.parametrize("name", ["lane64", "syn6_w64", "free", "vdp40"])
def test_assemble_restatement_equals_the_header(lib, port, name):
    """the driver's numpy assemble gives the bits of ntg_newton.h's assemble (g++), with and without a shift,
    so a fault in the header's text cannot hide in a reference built from the same text"""
    spec, X, _, _, _ = nl.setup(name)
    nw = nl.Newton(lib, port, spec)
    s, n = nw.s, spec.nC
    for p in range(2):
        x = nw.init(X[p]).C
        G = np.ascontiguousarray(nw.fg(nw.points(x))[1])
        for tau in (0.0, 0.37):
            band, dmax = nl.assemble(s, x, G, tau)
            hb = np.zeros(n * (s.w + 1))
            hd = lib.newton_host_assemble(n, s.w, s.K, nw.r, nl._p(s.perm, nl.ip), nl._p(s.color, nl.ip),
                                          nl._p(s.hmask, nl.bp), nl._p(s.ata), s.ata_max, nl._p(x), nl._p(G), tau,
                                          nl._p(hb))
            assert np.array_equal(band.view(np.int64), hb.view(np.int64)) and dmax == hd, (name, p, tau)


def test_refused_shapes_are_above_the_band_limit(lib, port):
    """syn6 at order 7, mult 1 with five cost outputs, and CFG-5's shape without its nonlinear rows, have
    w = 65 and 67 > 64: ntgb_solve_eq_newton refuses them (tests/test_gpu_newton_lockstep.py)"""
    import dataclasses
    from ntg_b200 import configs
    spec = nl.syn6_eq(7, 1, 4, range(5), "nl_syn6_w65")
    assert nl.structure(lib, port, spec, nl.eq_rows(port, spec)[0]).w == 65
    cfg5 = dataclasses.replace(configs.syn6(200), callbacks={"ucf": "syn6_ucf", "nltcf": ""}, nnltc=0,
                               trajectoryconstrav=[], name="nl_cfg5_eq")
    assert nl.structure(lib, port, cfg5, nl.eq_rows(port, cfg5)[0]).w == 67


def test_sequential_order_reproduces_the_restated_solve(lib, port):
    """with its reductions in one thread's order (nt = 1), the driver reproduces test_newton_host.py's
    newton_restated bit for bit, iteration by iteration to the end of the solve, when that restatement is given
    the same Q1 and Cpart and sums in the same order.  The 128-thread order gives other bits: the comparison
    sees the order of the sums."""
    from test_newton_host import Struct, _kincar, newton_restated
    spec = _kincar(24)
    s = Struct(lib, spec, port)
    x0 = np.random.default_rng(3).uniform(-2.0, 2.0, spec.nC)
    nw = nl.Newton(lib, port, spec, nt=1)
    ref = nl.lockstep(nw, x0, 12)
    kw = dict(Q1=nw.Q1, Cpart=nw.Cpart, proj=nw.project, dot=lambda a, b: nl.coop_sum(a * b, 1))
    for k in range(1, 13):
        Cr, st, it = newton_restated(lib, port, spec, s, x0, max_iter=k, **kw)
        snap = ref["snaps"][k]
        assert (snap["status"], snap["iters"]) == (st, it), (k, snap["status"], st, snap["iters"], it)
        assert np.array_equal(snap["C"].view(np.int64), Cr.view(np.int64)), (k, np.abs(snap["C"] - Cr).max())
        if st != 0:
            break
    assert st in (1, 2) and k >= 3, (st, k)
    wide = nl.lockstep(nl.Newton(lib, port, spec), x0, 2)
    assert not np.array_equal(wide["snaps"][2]["C"].view(np.int64), ref["snaps"][2]["C"].view(np.int64))


def test_coop_sum_orders():
    """coop_sum at one thread is the sequential sum; at 128 it is a sum of the same terms in another order"""
    v = np.random.default_rng(1).normal(size=1030) * 10.0 ** np.random.default_rng(2).integers(-8, 8, 1030)
    seq = 0.0
    for x in v:
        seq += x
    assert nl.coop_sum(v, 1) == seq
    assert abs(nl.coop_sum(v) - np.sum(v, dtype=np.longdouble)) <= 1e-13 * np.abs(v).sum()
    assert nl.coop_sum(np.ones(129)) == 129.0 and nl.coop_sum(np.zeros(0)) == 0.0


@pytest.mark.parametrize("name", nl.CONVEX)
def test_reference_reaches_the_kkt_point(lib, port, name):
    """run on, the reference ends with status 1 or 2 at the KKT solution (cost to 1e-9, C to 1e-6 of max |C|),
    on A C = b, for two starts of every convex setup"""
    from test_gpu_solve_lbfgs import _kkt
    spec, X, bounds, rejected, _ = nl.setup(name)
    nw = nl.Newton(lib, port, spec)
    for p in [q for q in range(X.shape[0]) if q not in rejected][:2]:
        Cp, b = None, None
        if bounds is not None:
            Cp = nw.problem_cpart(bounds[0][p], bounds[1][p])
            b = nl.eq_rows(port, nl.with_bounds(spec, bounds[0][p], bounds[1][p]))[1]
        A, b, _, Cref, fref = _kkt(port, spec, b)
        ref = nl.lockstep(nw, X[p], 40, Cpart=Cp)
        last = ref["snaps"][-1]
        assert last["status"] in (1, 2), (name, p, last["status"])
        assert np.abs(A @ last["C"] - b).max() <= 1e-10 * (1 + np.abs(b).max())
        assert abs(last["f"] - fref) <= 1e-9 * max(1.0, abs(fref)), (name, p, last["f"], fref)
        assert np.abs(last["C"] - Cref).max() <= 1e-6 * max(1.0, np.abs(Cref).max())


def test_setups_cover_every_path(refs):
    """between them, the GPU setups' references take a shifted refactorization, the -P g fallback (a slope
    d'g >= 0), a search without an Armijo step, and end problems with status 1 and with status 2, within their
    Kmax.  A factorization that fails after all kMaxShift shifts, and an S that is not positive definite, are
    not reached: M + tau I is positive definite long before tau = 4^8 beta, and S = Q1 M^-1 Q1' is then too."""
    recs = [r for _, rs in refs.values() for ref in rs for r in ref["recs"]]
    status = [ref["snaps"][-1]["status"] for _, rs in refs.values() for ref in rs]
    assert sum(r.get("shifts", 0) > 0 for r in recs) > 0
    assert sum(r.get("fallback") == "slope" for r in recs) > 0
    assert sum(not r["armijo"] for r in recs if "armijo" in r) > 0
    assert 1 in status and 2 in status
    for name, (nw, rs) in refs.items():
        print(name, "shifted", sum(r.get("shifts", 0) > 0 for ref in rs for r in ref["recs"]),
              "fallbacks", sum(r.get("fallback") is not None for ref in rs for r in ref["recs"]),
              "no Armijo step", sum(not r.get("armijo", True) for ref in rs for r in ref["recs"]),
              "status", np.bincount([ref["snaps"][-1]["status"] for ref in rs]).tolist())
