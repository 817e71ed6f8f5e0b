"""CPU checks of the projected L-BFGS solver (ntgb_solve_eq_lbfgs).  Its per-problem core (ntg_b200/csrc/ntg_lbfgs.h,
compiled with g++ through tests/tools/lbfgs_host.cpp -- the same text the CTA kernels run) against the numpy
restatement tests/tools/lbfgs_reference.py: the two-loop direction, the pair and reset rules, the projection
and the step back onto the affine set.  A whole solve of the restatement with the CPU oracle's evaluations on
a long-horizon lane change reaches the KKT point.  The argument refusals need no device.  The device half is
tests/test_gpu_solve_lbfgs.py."""
import ctypes as C
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "tools"))
import lbfgs_reference as ref  # noqa: E402

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("lbfgs") / "lbfgs_host.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "ntg_b200", "csrc"),
                           "-o", so, os.path.join(HERE, "tools", "lbfgs_host.cpp")])
    L = C.CDLL(so)
    L.lbfgs_host_project.argtypes = [dp, C.c_int, C.c_int, dp]
    L.lbfgs_host_direction.restype = C.c_int
    L.lbfgs_host_direction.argtypes = [dp, C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, ip, dp, C.c_double, dp,
                                       C.c_double, dp, dp]
    L.lbfgs_host_accept.restype = C.c_int
    L.lbfgs_host_accept.argtypes = [dp, C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, ip, dp, dp, dp, dp, C.c_double,
                                    C.c_double, C.c_double]
    return L


def _p(a):
    return a.ctypes.data_as(dp)


class Core:
    """one problem's state as the header keeps it, driven through the g++ build"""

    def __init__(self, lib, Q1, mem):
        self.lib, self.Q1, self.mem = lib, np.ascontiguousarray(Q1), mem
        self.r, self.n = Q1.shape
        self.ring = np.zeros((mem, 2, self.n))
        self.rho = np.zeros(mem)
        self.sv, self.gp = np.zeros(self.n), np.zeros(self.n)
        self.st = np.zeros(3, dtype=np.int32)   # head, npair, pend
        self.gamma = np.ones(1)

    @property
    def npair(self):
        return int(self.st[1])

    def direction(self, f, g, gtol=1e-12):
        d, dg = np.zeros(self.n), np.zeros(1)
        rc = self.lib.lbfgs_host_direction(_p(self.Q1), self.r, self.n, self.mem, _p(self.ring), _p(self.rho),
                                           _p(self.sv), _p(self.gp), self.st.ctypes.data_as(ip), _p(self.gamma), f,
                                           _p(np.ascontiguousarray(g)), gtol, _p(d), _p(dg))
        return rc, d, float(dg[0])

    def accept(self, Cpart, Cv, d, a, phi0, phib):
        rc = self.lib.lbfgs_host_accept(_p(self.Q1), self.r, self.n, self.mem, _p(self.ring), _p(self.rho), _p(self.sv),
                                        _p(self.gp), self.st.ctypes.data_as(ip), _p(self.gamma), _p(Cpart), _p(Cv),
                                        _p(d), a, phi0, phib)
        return rc


def _instance(seed, n=48, m=6):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(m, n))
    Q1 = ref.row_basis(A)
    X = rng.normal(size=(n, n))
    M = X @ X.T / n + np.diag(rng.uniform(0.1, 3.0, n))   # SPD: a convex quadratic 1/2 C'MC + q'C
    q = rng.normal(size=n)
    b = rng.normal(size=m)
    Cpart = np.linalg.lstsq(A, b, rcond=None)[0]
    return rng, A, b, Q1, M, q, Cpart


def test_projection_and_direction_stay_in_null_space(lib):
    rng, A, b, Q1, M, q, Cpart = _instance(1)
    v = rng.normal(size=A.shape[1]) * 10
    w = v.copy()
    lib.lbfgs_host_project(_p(Q1), Q1.shape[0], Q1.shape[1], _p(w))
    assert np.abs(A @ w).max() <= 1e-13 * np.abs(v).max() * np.abs(A).max() * A.shape[1]
    np.testing.assert_allclose(w, ref.project(Q1, v), rtol=0, atol=1e-13 * np.abs(v).max())
    # every direction of a run with pairs in the ring is in null(A), and every accepted C is on A C = b
    core = Core(lib, Q1, 4)
    Cv = Cpart + rng.normal(size=A.shape[1])
    for k in range(10):
        g = M @ Cv + q
        rc, d, dg = core.direction(0.5 * Cv @ M @ Cv + q @ Cv, g)
        assert rc == 0 and dg < 0
        assert np.abs(A @ d).max() <= 1e-12 * max(1.0, np.abs(d).max())
        assert core.accept(Cpart, Cv, d, 0.5, 1.0, 0.0) == 0
        assert np.abs(A @ Cv - b).max() <= 1e-12 * (1 + np.abs(b).max())
    assert core.npair == 4


@pytest.mark.parametrize("mem", [1, 3, 8])
def test_two_loop_direction_matches_the_restatement(lib, mem):
    """the header's ring (wrapping after mem pairs) against the textbook two-loop, fed the same C at each step"""
    rng, A, b, Q1, M, q, Cpart = _instance(2 + mem)
    core, h = Core(lib, Q1, mem), ref.History(mem)
    Cv = Cpart + ref.project(Q1, rng.normal(size=A.shape[1]))
    for k in range(2 * mem + 2):     # past a wrap of the ring, before the run converges to rounding level
        f, g = 0.5 * Cv @ M @ Cv + q @ Cv, M @ Cv + q
        rc, d, dg = core.direction(f, g)
        st, dr, dgr = ref.direction(Q1, h, f, g, 1e-12)
        assert rc == st == 0
        assert core.npair == len(h.S)
        assert np.abs(d - dr).max() <= 1e-12 * np.abs(dr).max(), (k, np.abs(d - dr).max())
        assert abs(dg - dgr) <= 1e-12 * abs(dgr)
        C0 = Cv.copy()
        a = 0.25 + 0.5 * rng.uniform()
        core.accept(Cpart, Cv, d, a, 1.0, 0.0)
        h.sv = Cv - C0          # the restatement pairs exactly the step the core took
    assert core.npair == mem


def test_pair_skip_rule(lib):
    """a pair with s'u <= kSkipEps |s| |u| is not kept; one just above it is, with rho = 1/s'u and gamma = s'u/u'u"""
    n = 6
    Q1 = np.zeros((0, n))
    e = np.eye(n)
    for su, kept in ((-1.0, False), (0.0, False), (0.5e-10, False), (2e-10, True), (0.3, True)):
        core = Core(lib, Q1, 4)
        core.sv[:] = e[0]                        # s
        u = su * e[0] + e[1]                     # s'u = su, |s| = 1, |u| ~ 1
        core.gp[:] = 0.0
        core.st[2] = 1                           # pending pair
        g = u.copy()
        rc, d, dg = core.direction(1.0, g)
        assert rc == 0
        uu = float(u @ u)
        kept_here = core.npair == 1
        # the rule is on s'u against 1e-10 |s| |u|: |u| is a little above 1
        assert kept_here == (su > 1e-10 * np.sqrt(uu)), su
        assert kept_here == kept
        if kept:
            np.testing.assert_array_equal(core.ring[0, 0], e[0])
            np.testing.assert_array_equal(core.ring[0, 1], u)
            assert core.rho[0] == 1.0 / su and core.gamma[0] == su / uu
            assert core.st[0] == 1
        else:
            assert core.st[0] == 0 and core.gamma[0] == 1.0
        np.testing.assert_array_equal(core.gp, g)   # the projected gradient of this point, for the next pair


def test_reset_rule_and_steepest_scaling(lib):
    """a history whose H is not positive definite gives d'g >= 0: it is dropped and d = -P g, scaled to length 1"""
    rng, A, b, Q1, M, q, Cpart = _instance(5)
    n = A.shape[1]
    core = Core(lib, Q1, 3)
    s = ref.project(Q1, rng.normal(size=n))
    core.ring[0, 0], core.ring[0, 1] = s, s
    core.rho[0] = 1.0 / float(s @ s)
    core.st[:] = (1, 1, 0)
    core.gamma[0] = -1.0                          # H = -I on the complement of s: an ascent direction
    g = 5.0 * rng.normal(size=n)
    rc, d, dg = core.direction(1.0, g)
    pg = ref.project(Q1, g)
    assert rc == 0 and core.npair == 0
    np.testing.assert_allclose(d, -pg / np.linalg.norm(pg), rtol=0, atol=1e-13)
    assert dg == pytest.approx(-np.linalg.norm(pg), rel=1e-13)
    # a short steepest-descent direction is not lengthened
    rc, d, dg = core.direction(1.0, 1e-3 * g)
    np.testing.assert_allclose(d, -1e-3 * pg, rtol=0, atol=1e-15)


def test_convergence_test_and_failed_searches(lib):
    rng, A, b, Q1, M, q, Cpart = _instance(6)
    n = A.shape[1]
    core = Core(lib, Q1, 3)
    g = A.T @ rng.normal(size=A.shape[0])          # in the row space: P g = 0 up to rounding
    assert core.direction(10.0, g, gtol=1e-12)[0] == 1
    g[0] = np.nan
    assert core.direction(10.0, g)[0] == 2
    Cv = Cpart.copy()
    C0 = Cv.copy()
    d = ref.project(Q1, rng.normal(size=n))
    assert core.accept(Cpart, Cv, d, 1.0, 1.0, 1.0) == 2      # no decrease from steepest descent: done
    np.testing.assert_array_equal(Cv, C0)
    core.st[:] = (2, 2, 1)
    assert core.accept(Cpart, Cv, d, 1.0, 1.0, 2.0) == 0      # no decrease along an L-BFGS direction: retry
    assert tuple(core.st) == (2, 0, 0)
    np.testing.assert_array_equal(Cv, C0)


def _long_kincar(ninterv, nbps):
    from ntg_b200 import configs
    return dataclasses.replace(configs.kincar(nbps, constraints=False, name=f"lbfgs_kincar{ninterv}"),
                               ninterv=[ninterv, ninterv], knots=None)


def test_whole_solve_reaches_the_kkt_point_on_a_long_lane_change(port):
    """the restated solver with the oracle's evaluations: a lane change over 2 x 24 intervals (nC = 102, 90 free
    directions), from a random start, reaches the solution of its KKT system in under 1000 iterations"""
    spec = _long_kincar(24, 97)
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    H = port.eval(spec, np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]
    H = 0.5 * (H + H.T)
    K = np.block([[H, A.T], [A, np.zeros((A.shape[0], A.shape[0]))]])
    Cref = np.linalg.solve(K, np.concatenate([np.zeros(nC), b]))[:nC]
    fref = float(port.eval(spec, Cref[None, :], mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0])

    def fg(Cv):
        r = port.eval(spec, Cv[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        return float(r["f"][0]), r["g"][0]

    Q1 = ref.row_basis(A)
    Cpart = np.linalg.lstsq(A, b, rcond=None)[0]
    X0 = np.random.default_rng(3).uniform(-2.0, 2.0, nC)
    Cs, st, it = ref.solve(fg, Q1, Cpart, X0, max_iter=2000)
    assert st in (1, 2) and it < 1000, (st, it)     # 2: no Armijo step decreases the cost measurably any more (rounding level)
    assert np.abs(A @ Cs - b).max() <= 1e-10 * (1 + np.abs(b).max())
    assert abs(fg(Cs)[0] - fref) <= 1e-9 * max(1.0, abs(fref))
    assert np.abs(Cs - Cref).max() <= 1e-6 * max(1.0, np.abs(Cref).max())


def test_arguments_are_refused_before_cuda(built_libs):
    """bad memory and exactly one bound array NULL are NTGB_EINVAL before the handle is read, so a handle that
    was never created is enough"""
    from ntg_b200 import problem
    from ntg_b200.abi import LbfgsOpts
    lib = problem.core()
    C_ = (C.c_double * 4)()
    fake = C.create_string_buffer(64)
    pb = C.c_void_p(C.addressof(fake))
    assert lib.ntgb_solve_eq_lbfgs(None, 1, C_, None, None, None, None, None, None, None) == -1
    assert "null argument" in lib.ntgb_last_error().decode()
    for mem in (0, 33, -1):
        opts = LbfgsOpts(0, 0.0, 0.0, mem, 0)
        assert lib.ntgb_solve_eq_lbfgs(pb, 1, C_, None, None, None, None, None, C.addressof(opts), None) == -1
        assert f"memory = {mem} outside [1,32]" in lib.ntgb_last_error().decode()
    lo = (C.c_double * 4)()
    for lb, ub in ((lo, None), (None, lo)):
        assert lib.ntgb_solve_eq_lbfgs(pb, 1, C_, lb, ub, None, None, None, None, None) == -1
        assert "exactly one of lowerb / upperb is NULL" in lib.ntgb_last_error().decode()
