"""CPU checks of the banded Newton solver (ntgb_solve_eq_newton).  Its host structure and per-problem algebra
(ntg_b200/csrc/ntg_newton.h, compiled with g++ through tests/tools/newton_host.cpp -- the same text the CTA kernels
run) against the CPU oracle and numpy: the pattern, permutation, bandwidth and colouring on long horizons, the
band recovered from coloured gradient differences, the banded Cholesky and the range-space step, and a whole
restated solve with the oracle's evaluations.  The argument refusals need no device.  The device half is
tests/test_gpu_solve_newton.py."""
import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)
up = C.POINTER(C.c_uint)
bp_ = C.POINTER(C.c_ubyte)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("newton") / "newton_host.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "ntg_b200", "csrc"),
                           "-o", so, os.path.join(HERE, "tools", "newton_host.cpp")])
    L = C.CDLL(so)
    L.newton_host_structure.restype = C.c_int
    L.newton_host_structure.argtypes = [C.c_int, C.c_int, ip, ip, ip, up, dp, C.c_int, ip, ip]
    L.newton_host_fetch.argtypes = [ip, ip, bp_, dp]
    L.newton_host_step_of.restype = C.c_double
    L.newton_host_step_of.argtypes = [C.c_double]
    L.newton_host_assemble.restype = C.c_double
    L.newton_host_assemble.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, bp_, dp, C.c_double, dp, dp,
                                       C.c_double, dp]
    L.newton_host_factor.restype = C.c_int
    L.newton_host_factor.argtypes = [C.c_int, C.c_int, dp]
    L.newton_host_solve.argtypes = [C.c_int, C.c_int, dp, ip, dp]
    L.newton_host_range_step.restype = C.c_int
    L.newton_host_range_step.argtypes = [C.c_int, C.c_int, C.c_int, ip, dp, dp, dp, dp]
    L.newton_host_after_search.restype = C.c_int
    L.newton_host_after_search.argtypes = [dp, C.c_int, C.c_double, C.c_double, C.c_double]
    return L


def _p(a, t=dp):
    return a.ctypes.data_as(t)


class Struct:
    """what build_structure derives for one setup"""

    def __init__(self, lib, spec, port):
        _, off, _ = port.tables(spec)
        nC = spec.nC
        o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
        A = o["A"]
        eq = o["bl"][nC:nC + spec.nclin] == o["bu"][nC:nC + spec.nclin]
        self.A, self.b = np.ascontiguousarray(A[eq]), o["bl"][nC:nC + spec.nclin][eq]
        mask = np.zeros(3, dtype=np.uint32)
        for k, (cnt, av) in enumerate(((spec.nicf, spec.initialcostav), (spec.nucf, spec.trajectorycostav),
                                       (spec.nfcf, spec.finalcostav))):
            if cnt:
                for j, _d in av:
                    mask[k] |= 1 << j
        order = np.array(spec.order, dtype=np.int32)
        ncoef = np.array(spec.ncoef, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int32)
        K, w = C.c_int(), C.c_int()
        assert lib.newton_host_structure(spec.nout, spec.nbps, _p(order, ip), _p(ncoef, ip), _p(off, ip),
                                         _p(mask, up), _p(self.A), self.A.shape[0], C.byref(K), C.byref(w)) == 0
        self.nC, self.K, self.w = nC, K.value, w.value
        W = self.w + 1
        self.perm = np.zeros(nC, dtype=np.int32)
        self.color = np.zeros(nC, dtype=np.int32)
        self.hmask = np.zeros(nC * W, dtype=np.uint8)
        self.ata = np.zeros(nC * W)
        lib.newton_host_fetch(_p(self.perm, ip), _p(self.color, ip), _p(self.hmask, bp_), _p(self.ata))
        self.pos = np.argsort(self.perm)

    def pattern(self):
        """dense boolean H pattern from the band mask (original order)"""
        W = self.w + 1
        P = np.zeros((self.nC, self.nC), bool)
        i, d = np.nonzero(self.hmask.reshape(self.nC, W))
        a, b = self.perm[i], self.perm[i - d]
        P[a, b] = P[b, a] = True
        return P


def _kincar(ninterv):
    from ntg_b200 import configs
    return dataclasses.replace(configs.kincar(3 * ninterv + 1, constraints=False, name=f"newton_kincar{ninterv}"),
                               ninterv=[ninterv, ninterv], knots=None)


def _vdp40():
    from ntg_b200 import configs
    return dataclasses.replace(configs.vanderpol(121, constraints=False, name="newton_vdp40"), ninterv=[40], knots=None)


def _syn6():
    from ntg_b200 import configs
    return configs.syn6(8, name="newton_syn6")


def _dense_hessian(port, spec, x, h=1e-4):
    nC = spec.nC
    gp = port.eval(spec, x + h * np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]
    gm = port.eval(spec, x - h * np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]
    H = (gp - gm) / (2 * h)     # row c: column c of H
    return 0.5 * (H + H.T)


SHAPES = {"kincar8": lambda: _kincar(8), "kincar64": lambda: _kincar(64), "kincar256": lambda: _kincar(256),
          "vdp40": _vdp40, "syn6": _syn6}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_structure(lib, port, shape):
    spec = SHAPES[shape]()
    s = Struct(lib, spec, port)
    nC = spec.nC
    assert np.array_equal(np.sort(s.perm), np.arange(nC))
    P = s.pattern()
    ata = s.A.T @ s.A
    i, j = np.nonzero(P | (ata != 0))
    assert np.abs(s.pos[i] - s.pos[j]).max() == s.w
    # the pattern holds every nonzero of the oracle's dense difference Hessian and of A'A
    if nC <= 300:
        x = np.random.default_rng(1).uniform(-2, 2, nC)
        H = _dense_hessian(port, spec, x)
        big = np.abs(H) > 1e-7 * np.abs(H).max()
        assert not (big & ~P).any(), np.argwhere(big & ~P)[:5]
    ri, rj = np.nonzero(ata)
    assert (np.abs(s.pos[ri] - s.pos[rj]) <= s.w).all()
    # no two columns of one colour share a row of the H pattern
    for k in range(s.K):
        cols = np.flatnonzero(s.color == k)
        assert (P[:, cols].sum(axis=1) <= 1).all(), k
    assert s.K <= 2 * s.w + 1
    if shape.startswith("kincar"):
        # the structural pattern couples both outputs at every breakpoint (the cost's active variables); the
        # same colours and bandwidth at every horizon
        assert (s.K, s.w) == (18, 13)


def _colored_gradients(port, spec, s, x):
    """G [2K][nC]: point 2k = x + h on colour k, 2k + 1 = x - h (the device's k_newton_points)"""
    h = np.array([s.lib.newton_host_step_of(float(v)) for v in x])
    X = []
    for k in range(s.K):
        e = np.where(s.color == k, h, 0.0)
        X += [x + e, x - e]
    return np.ascontiguousarray(port.eval(spec, np.array(X), mode_obj=2, mode_con=-1, dense=False, band=False)["g"])


def _assemble(lib, s, x, G, tau=0.0, ata_max=0.0):
    band = np.zeros(s.nC * (s.w + 1))
    dmax = lib.newton_host_assemble(s.nC, s.w, s.K, 0, _p(s.perm, ip), _p(s.color, ip), _p(s.hmask, bp_), _p(s.ata),
                                    ata_max, _p(np.ascontiguousarray(x)), _p(G), tau, _p(band))
    return band, dmax


def _band_to_dense(s, band):
    W = s.w + 1
    B = band.reshape(s.nC, W)
    M = np.zeros((s.nC, s.nC))
    for i in range(s.nC):
        for d in range(min(i, s.w) + 1):
            a, b = s.perm[i], s.perm[i - d]
            M[a, b] = M[b, a] = B[i, d]
    return M


@pytest.mark.parametrize("shape", ["kincar8", "vdp40"])
def test_band_recovery(lib, port, shape):
    spec = SHAPES[shape]()
    s = Struct(lib, spec, port)
    s.lib = lib
    x = np.random.default_rng(2).uniform(-2, 2, spec.nC)
    band, _ = _assemble(lib, s, x, _colored_gradients(port, spec, s, x))
    H = _dense_hessian(port, spec, x)
    Hb = _band_to_dense(s, band)
    assert np.abs(Hb - H).max() <= 1e-6 * np.abs(H).max(), np.abs(Hb - H).max() / np.abs(H).max()


def _random_band(rng, n, w, spd=True):
    """a symmetric band matrix in a random order: (M dense, perm, band [n][w+1])"""
    perm = rng.permutation(n).astype(np.int32)
    B = np.zeros((n, w + 1))
    for i in range(n):
        for d in range(min(i, w) + 1):
            B[i, d] = rng.normal()
    Mp = np.zeros((n, n))
    for i in range(n):
        for d in range(min(i, w) + 1):
            Mp[i, i - d] = Mp[i - d, i] = B[i, d]
    if spd:
        Mp += np.diag(np.abs(Mp).sum(axis=1) + 0.5)
    else:
        Mp[np.diag_indices(n)] = rng.normal(size=n)
    for i in range(n):
        B[i, 0] = Mp[i, i]
    M = np.zeros((n, n))
    M[np.ix_(perm, perm)] = Mp
    return M, perm, B.ravel().copy()


@pytest.mark.parametrize("n,w,r", [(40, 3, 5), (120, 8, 12), (64, 17, 1), (30, 5, 0)])
def test_banded_cholesky_and_range_space_step(lib, n, w, r):
    rng = np.random.default_rng(n + w + r)
    M, perm, band = _random_band(rng, n, w)
    L = band.copy()
    assert lib.newton_host_factor(n, w, _p(L)) == 1
    x = rng.normal(size=n)
    y = x.copy()
    lib.newton_host_solve(n, w, _p(L), _p(perm, ip), _p(y))
    assert np.abs(M @ y - x).max() <= 1e-10 * np.abs(x).max()
    A = rng.normal(size=(max(r, 1), n))[:r]
    Q1 = np.ascontiguousarray(np.linalg.qr(A.T)[0].T) if r else np.zeros((1, n))
    g = rng.normal(size=n)
    d = np.zeros(n)
    assert lib.newton_host_range_step(n, w, r, _p(perm, ip), _p(Q1), _p(L), _p(g), _p(d)) == 1
    K = np.block([[M, Q1[:r].T], [Q1[:r], np.zeros((r, r))]])
    want = np.linalg.solve(K, np.concatenate([-g, np.zeros(r)]))[:n]
    assert np.abs(d - want).max() <= 1e-10 * max(1.0, np.abs(want).max())
    if r:
        assert np.abs(Q1[:r] @ d).max() <= 1e-12 * np.abs(d).max()


def test_shifted_factorization_of_an_indefinite_band(lib):
    rng = np.random.default_rng(9)
    n, w = 50, 4
    M, perm, band = _random_band(rng, n, w, spd=False)
    assert np.linalg.eigvalsh(M).min() < 0
    assert lib.newton_host_factor(n, w, _p(band.copy())) == 0
    tau = 1.1 * -np.linalg.eigvalsh(M).min()
    shifted = band.reshape(n, w + 1).copy()
    shifted[:, 0] += tau
    L = shifted.ravel().copy()
    assert lib.newton_host_factor(n, w, _p(L)) == 1
    x = rng.normal(size=n)
    y = x.copy()
    lib.newton_host_solve(n, w, _p(L), _p(perm, ip), _p(y))
    assert np.abs((M + tau * np.eye(n)) @ y - x).max() <= 1e-9 * np.abs(x).max()


def test_shift_and_stopping_rule(lib):
    st = np.array([0.0, 2.0, 0.0])
    assert lib.newton_host_after_search(_p(st), 1, 1.0, 0.5, 1.0) == 0 and tuple(st) == (0.0, 2.0, 0.0)
    assert lib.newton_host_after_search(_p(st), 1, 0.125, 0.5, 1.0) == 0 and tuple(st) == (2.0, 2.0, 0.0)
    assert lib.newton_host_after_search(_p(st), 1, 0.5, 0.5, 1.0) == 0 and tuple(st) == (2.0, 2.0, 0.0)
    assert lib.newton_host_after_search(_p(st), 1, 1.0, 0.5, 1.0) == 0 and tuple(st) == (0.5, 2.0, 0.0)
    assert lib.newton_host_after_search(_p(st), 0, 1.0, 1.0, 1.0) == 0 and tuple(st) == (2.0, 2.0, 1.0)
    assert lib.newton_host_after_search(_p(st), 1, 1.0, 0.5, 1.0) == 0 and tuple(st) == (0.5, 2.0, 0.0)
    # two iterations in a row without a strict decrease: the rounding floor, status 2
    assert lib.newton_host_after_search(_p(st), 1, 1.0, 1.0, 1.0) == 0 and tuple(st) == (0.125, 2.0, 1.0)
    assert lib.newton_host_after_search(_p(st), 0, 1.0, 1.0, 1.0) == 2 and tuple(st) == (2.0, 2.0, 2.0)


def newton_restated(lib, port, spec, s, x0, gtol=1e-9, c1=1e-4, max_iter=50, Q1=None, Cpart=None, proj=None,
                    dot=np.dot):
    """the device loop restated with the g++ build and the oracle's evaluations: -> (C, status, iters).  By default
    Q1 from numpy's QR, Cpart from lstsq, P v = v - Q1' (Q1 v) and BLAS dot products; Q1, Cpart, proj and dot may
    be given instead (the library's basis and a fixed summation order make the result exact)."""
    nC = spec.nC
    A, b = s.A, s.b
    Q1 = np.ascontiguousarray(np.linalg.qr(A.T)[0].T) if Q1 is None else Q1
    Cpart = np.linalg.lstsq(A, b, rcond=None)[0] if Cpart is None else Cpart
    proj = (lambda v: v - Q1.T @ (Q1 @ v)) if proj is None else proj
    x = Cpart + proj(x0 - Cpart)
    ata_max = float(s.ata.reshape(nC, -1)[:, 0].max())
    st = np.array([0.0, 0.0, 0.0])
    s.lib = lib
    eps = np.finfo(float).eps
    for it in range(max_iter):
        r = port.eval(spec, x[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        f, g = float(r["f"][0]), r["g"][0]
        pg = proj(g)
        if np.abs(pg).max() <= gtol * max(1.0, abs(f)):
            return x, 1, it
        G = _colored_gradients(port, spec, s, x)
        ok = False
        for _ in range(8):
            band, dmax = _assemble(lib, s, x, G, st[0], ata_max)
            st[1] = 1e-3 * (dmax if dmax > 0 else 1.0)
            if lib.newton_host_factor(nC, s.w, _p(band)):
                ok = True
                break
            st[0] = max(4 * st[0], st[1])
        d = np.zeros(nC)
        dg = 0.0
        if ok and lib.newton_host_range_step(nC, s.w, Q1.shape[0], _p(s.perm, ip), _p(Q1), _p(band), _p(g), _p(d)):
            dg = dot(d, g)
        if not dg < 0:
            d = -pg
            dg = -dot(pg, pg)
        phi0 = f + 8 * eps * abs(f)
        alphas = 2.0 ** -np.arange(16)
        ft = port.eval(spec, x[None, :] + alphas[:, None] * d[None, :], mode_obj=0, mode_con=-1, dense=False,
                       band=False)["f"]
        arm = np.flatnonzero(ft <= phi0 + c1 * alphas * dg)
        a = alphas[arm[0]] if arm.size else 1.0
        if arm.size:
            x = Cpart + proj(x + a * d - Cpart)
        done = lib.newton_host_after_search(_p(st), int(arm.size > 0), a, float(ft[arm[0]]) if arm.size else f, f)
        if done:
            return x, 2, it + 1
    return x, 0, max_iter


def test_whole_solve_reaches_the_kkt_point_on_a_long_lane_change(lib, port):
    """2 x 24 intervals (nC = 102, 90 free directions) from a random start: the KKT point within 10 iterations"""
    spec = _kincar(24)
    s = Struct(lib, spec, port)
    nC = spec.nC
    A, b = s.A, s.b
    H = port.eval(spec, np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]
    H = 0.5 * (H + H.T)
    K = np.block([[H, A.T], [A, np.zeros((A.shape[0], A.shape[0]))]])
    Cref = np.linalg.solve(K, np.concatenate([np.zeros(nC), b]))[:nC]
    fref = float(port.eval(spec, Cref[None, :], mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0])
    x0 = np.random.default_rng(3).uniform(-2.0, 2.0, nC)
    Cs, st, it = newton_restated(lib, port, spec, s, x0)
    assert st in (1, 2) and it <= 10, (st, it)
    assert np.abs(A @ Cs - b).max() <= 1e-10 * (1 + np.abs(b).max())
    f = float(port.eval(spec, Cs[None, :], mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0])
    assert abs(f - fref) <= 1e-9 * max(1.0, abs(fref))
    assert np.abs(Cs - Cref).max() <= 1e-6 * max(1.0, np.abs(Cref).max())


def test_arguments_are_refused_before_cuda(built_libs):
    """exactly one bound array NULL is NTGB_EINVAL before the handle is read, so a handle that was never created
    is enough"""
    from ntg_b200 import problem
    lib = problem.core()
    C_ = (C.c_double * 4)()
    fake = C.create_string_buffer(64)
    pb = C.c_void_p(C.addressof(fake))
    assert lib.ntgb_solve_eq_newton(None, 1, C_, None, None, None, None, None, None, None) == -1
    assert "null argument" in lib.ntgb_last_error().decode()
    lo = (C.c_double * 4)()
    for lb, ub in ((lo, None), (None, lo)):
        assert lib.ntgb_solve_eq_newton(pb, 1, C_, lb, ub, None, None, None, None, None) == -1
        assert "exactly one of lowerb / upperb is NULL" in lib.ntgb_last_error().decode()
