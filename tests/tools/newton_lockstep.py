"""tests/tools/newton_lockstep.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The banded Newton solver (ntgb_solve_eq_newton) followed iteration by iteration on the host, so that a GPU solve
stopped after K iterations can be compared with the same K iterations here, bit for bit.  Every input of one
device iteration is reproduced exactly:

  * the evaluations at C, at the 2K difference points and at the trial points: the CPU oracle, which the exact
    build matches bit for bit on the libm-free packs (kincar, vanderpol, syn6);
  * the difference points C +- fd_step(C) and the trial points C + alpha d: numpy, the same IEEE operations as
    ntg_core.cu (always built with -fmad=false);
  * assemble: numpy, entry by entry the header's operations (elementwise, so exact), checked against the
    header's g++ build; a fault in the header's assemble then shows up against the device;
  * band_cholesky, range_step and after_search: the g++ build of ntg_newton.h (tests/tools/newton_host.cpp),
    whose every dot product and triangular solve one thread walks in a fixed order, so a group of one thread
    gives the bits of a CTA of 128.  A fault in this text that does not depend on the number of threads is on
    both sides; test_newton_host.py holds these functions to dense numpy solves;
  * Q1, Cpart and M: sqp_lockstep.reduce_linear, bit-identical to the library's reduce_linear;
  * project, dot, affine_step and the |P g| test of k_newton_check: numpy restated at the CTA's reduction order
    (coop_sum: per-thread strided sums, the xor butterfly 16, 8, 4, 2, 1 in each warp, then the warps in order);
  * the two-stage search's pick (k_alm_pick1 / k_alm_pick2) and the Armijo test of k_newton_update.

A run with max_iter = K is the first K iterations of a longer run, so lockstep() records the snapshot of every
K at once.  iterate() is also the teacher-forced mode: one iteration from a given C, tau, beta and stall.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np

from sqp_lockstep import reduce_linear, with_bounds

NT = 128                      # kNewtonThreads
KMAX_SHIFT = 8                # ntg_newton.h kMaxShift
BETA_REL = 1e-3               # kBetaRel
NALPHA1, NALPHA = 4, 16       # two_stage_search: kN1 coarse steps, kNalpha in all
EPS = float(np.finfo(np.float64).eps)
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "ntg_b200", "csrc")

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)
up = C.POINTER(C.c_uint)
bp = C.POINTER(C.c_ubyte)


def _p(a, t=dp):
    return a.ctypes.data_as(t)


def load_host(directory):
    """compile tests/tools/newton_host.cpp into `directory` and declare its functions"""
    so = os.path.join(str(directory), "newton_host.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I", CSRC, "-o", so,
                           os.path.join(os.path.dirname(os.path.abspath(__file__)), "newton_host.cpp")])
    L = C.CDLL(so)
    L.newton_host_structure.restype = C.c_int
    L.newton_host_structure.argtypes = [C.c_int, C.c_int, ip, ip, ip, up, dp, C.c_int, ip, ip]
    L.newton_host_fetch.argtypes = [ip, ip, bp, dp]
    L.newton_host_step_of.restype = C.c_double
    L.newton_host_step_of.argtypes = [C.c_double]
    L.newton_host_assemble.restype = C.c_double
    L.newton_host_assemble.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, bp, dp, C.c_double, dp, dp,
                                       C.c_double, dp]
    L.newton_host_factor.restype = C.c_int
    L.newton_host_factor.argtypes = [C.c_int, C.c_int, dp]
    L.newton_host_range_step.restype = C.c_int
    L.newton_host_range_step.argtypes = [C.c_int, C.c_int, C.c_int, ip, dp, dp, dp, dp]
    L.newton_host_after_search.restype = C.c_int
    L.newton_host_after_search.argtypes = [dp, C.c_int, C.c_double, C.c_double, C.c_double]
    return L


def coop_sum(v, nt=NT):
    """sqp::Coop::reduce<false> of the terms v [n] over a group of nt threads (ntg_sqp.cuh): thread t sums
    e = t, t + nt, ... in order from 0.0; then (nt >= 32) the xor butterfly 16, 8, 4, 2, 1 in each warp and the
    warps' sums in order.  nt = 1 is the host build's group of one thread: one sequential sum."""
    v = np.asarray(v, dtype=np.float64).ravel()
    acc = np.zeros(nt)
    for s in range(0, v.size, nt):
        c = v[s:s + nt]
        acc[:c.size] = acc[:c.size] + c
    if nt == 1:
        return float(acc[0])
    lanes = acc.reshape(nt // 32, 32)
    idx = np.arange(32)
    for d in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, idx ^ d]
    s = lanes[0, 0]
    for k in range(1, nt // 32):
        s = s + lanes[k, 0]
    return float(s)


def coop_max(v):
    """reduce<true> of per-thread fmax from 0.0: the largest entry, order-free"""
    return float(np.fmax.reduce(np.concatenate([[0.0], np.asarray(v, dtype=np.float64).ravel()])))


def fd_step(x):
    """ntg_newton.h fd_step, elementwise"""
    return 6.0554544523933395e-06 * np.maximum(np.abs(x), 1.0)


def eq_rows(port, spec):
    """the equality rows A [m][nC] and right-hand side b of a setup (alm's order: row index)"""
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False, linear=True)
    lb, ub = o["bl"][nC:nC + spec.nclin], o["bu"][nC:nC + spec.nclin]
    eq = lb == ub
    return np.ascontiguousarray(o["A"][eq]).reshape(int(eq.sum()), nC), lb[eq], eq


@dataclasses.dataclass
class Structure:
    K: int
    w: int
    perm: np.ndarray
    color: np.ndarray
    hmask: np.ndarray
    ata: np.ndarray

    @property
    def ata_max(self):
        return float(self.ata.reshape(-1, self.w + 1)[:, 0].max(initial=0.0))


def structure(lib, port, spec, A):
    """newton_prepare's build_structure for the setup, through the g++ build"""
    _, off, _ = port.tables(spec)
    mask = np.zeros(3, dtype=np.uint32)
    for k, (cnt, av) in enumerate(((spec.nicf, spec.initialcostav), (spec.nucf, spec.trajectorycostav),
                                   (spec.nfcf, spec.finalcostav))):
        if cnt:
            for j, _d in av:
                mask[k] |= 1 << j
    order = np.array(spec.order, dtype=np.int32)
    ncoef = np.array(spec.ncoef, dtype=np.int32)
    off = np.ascontiguousarray(off, dtype=np.int32)
    Am = np.ascontiguousarray(A if A.shape[0] else np.zeros((1, spec.nC)))
    K, w = C.c_int(), C.c_int()
    assert lib.newton_host_structure(spec.nout, spec.nbps, _p(order, ip), _p(ncoef, ip), _p(off, ip), _p(mask, up),
                                     _p(Am), A.shape[0], C.byref(K), C.byref(w)) == 0
    nC, W = spec.nC, w.value + 1
    s = Structure(K.value, w.value, np.zeros(nC, dtype=np.int32), np.zeros(nC, dtype=np.int32),
                  np.zeros(nC * W, dtype=np.uint8), np.zeros(nC * W))
    lib.newton_host_fetch(_p(s.perm, ip), _p(s.color, ip), _p(s.hmask, bp), _p(s.ata))
    return s


def assemble(s, C0, G, tau):
    """ntg_newton.h assemble restated in numpy, entry by entry the same IEEE operations: -> (band [nC][w+1] of
    H + rho A'A + tau I, max diag (H + rho A'A)).  The g++ build is checked against it bit for bit, so a fault in
    the header's text cannot hide in a reference built from that same text."""
    n, W = s.perm.size, s.w + 1
    i, d = np.divmod(np.arange(n * W), W)
    on = (d <= i) & (s.hmask != 0)
    ci, cj = s.perm[i[on]], s.perm[i[on] - d[on]]
    xi, xj = C0[ci], C0[cj]
    hi, hj = fd_step(xi), fd_step(xj)
    vj = (G[2 * s.color[cj], ci] - G[2 * s.color[cj] + 1, ci]) / ((xj + hj) - (xj - hj))
    vi = (G[2 * s.color[ci], cj] - G[2 * s.color[ci] + 1, cj]) / ((xi + hi) - (xi - hi))
    band = np.zeros(n * W)
    band[on] = 0.5 * (vj + vi)
    hm = coop_max(band[::W])
    am = s.ata_max
    rho = hm / am if am > 0.0 and hm > 0.0 else (1.0 if am > 0.0 else 0.0)
    band = band + rho * s.ata
    dmax = coop_max(band[::W])
    band[::W] = band[::W] + tau
    return band, dmax


@dataclasses.dataclass
class State:
    """one problem between iterations: what the device carries (C, tau, beta, stall, status, iters)"""
    C: np.ndarray
    tau: float = 0.0
    beta: float = 0.0
    stall: int = 0
    status: int = 0
    iters: int = 0

    def copy(self):
        return dataclasses.replace(self, C=self.C.copy())


class Newton:
    """one setup's solve restated.  nt: the CTA size the reductions of project / dot / check are ordered for
    (128, the device's; 1 for the sequential order of test_newton_host.py's restatement)."""

    def __init__(self, lib, port, spec, nt=NT, gtol=1e-9, c1=1e-4):
        self.lib, self.port, self.spec, self.nt, self.gtol, self.c1 = lib, port, spec, nt, gtol, c1
        self.A, self.b, self.eq = eq_rows(port, spec)
        _N, self.Cpart, self.Mop, self.r, self.Q1 = reduce_linear(self.A, self.b, q1=True)
        self.nC = spec.nC
        self.s = structure(lib, port, spec, self.A)
        self.Q1p = self.Q1 if self.r else np.zeros((1, self.nC))

    # ---- the reductions of ntg_lbfgs.h at the CTA's order ----
    def project(self, v):
        v = np.array(v, dtype=np.float64)
        for k in range(self.r):
            q = self.Q1[k]
            w = coop_sum(q * v, self.nt)
            v = v - w * q
        return v

    def affine_step(self, Cpart, C0, d=None, a=0.0):
        """ntg_lbfgs.h affine_step: Cpart + P (C0 + a d - Cpart)"""
        sv = ((C0 + a * d) if d is not None else C0) - Cpart
        return Cpart + self.project(sv)

    def problem_cpart(self, lo, up):
        """Cpart = M b for one problem's own bounds, summed in ntg_bounds.h's order (Reduced.problem_bounds)"""
        nC = self.nC
        o = self.port.eval(with_bounds(self.spec, lo, up), np.zeros((1, nC)), mode_obj=0, mode_con=-1, dense=False,
                           band=False, linear=True)
        be = o["bl"][nC:nC + self.spec.nclin][self.eq]
        Cp = np.zeros(nC)
        for j in range(len(be)):
            Cp = Cp + self.Mop[:, j] * float(be[j])
        return Cp

    # ---- evaluations (the oracle) ----
    def fg(self, X):
        e = self.port.eval(self.spec, np.atleast_2d(X), mode_obj=2, mode_con=-1, dense=False, band=False)
        return e["f"], e["g"]

    def f(self, X):
        return self.port.eval(self.spec, np.atleast_2d(X), mode_obj=0, mode_con=-1, dense=False, band=False)["f"]

    def points(self, x):
        """k_newton_points: [2K][nC], point 2k = x + h on colour k, 2k + 1 = x - h"""
        h = fd_step(x)
        X = np.empty((2 * self.s.K, self.nC))
        for k in range(self.s.K):
            on = self.s.color == k
            X[2 * k] = np.where(on, x + h, x)
            X[2 * k + 1] = np.where(on, x - h, x)
        return X

    def init(self, C0, Cpart=None):
        """k_newton_init"""
        Cpart = self.Cpart if Cpart is None else Cpart
        if self.r == self.nC:
            return State(Cpart.copy(), status=1)
        return State(self.affine_step(Cpart, np.asarray(C0, dtype=np.float64)))

    def iterate(self, st, Cpart=None, rec=None):
        """one pass of solve_newton_impl's loop for one problem; returns the new State.  rec (a dict) receives
        what the iteration decided: f, g, G, shifts, fallback, d, dg, phi0, pick, armijo, margin, tau, beta"""
        rec = {} if rec is None else rec
        if st.status != 0:
            return st
        Cpart = self.Cpart if Cpart is None else Cpart
        s, n, x = self.s, self.nC, st.C
        st = st.copy()
        f, g = (a[0] for a in self.fg(x))
        f = float(f)
        rec.update(f=f, g=g)
        # k_newton_check
        pg = self.project(g)
        gmax, gg = coop_max(np.abs(pg)), coop_sum(pg * pg, self.nt)
        if gg != gg:
            st.status = 2
        elif not gmax > self.gtol * max(abs(f), 1.0):
            st.status = 1
        if st.status:
            rec["checked"] = st.status
            return st
        # k_newton_points, the evaluation, k_newton_factor
        Xp = self.points(x)
        G = np.ascontiguousarray(self.fg(Xp)[1])
        rec["G"] = G
        tau, beta, ok = st.tau, 0.0, False
        for a in range(KMAX_SHIFT + 1):
            if a > 0:
                tau = max(4.0 * tau, beta)
            band, dmax = assemble(s, x, G, tau)
            beta = BETA_REL * (dmax if dmax > 0.0 else 1.0)
            ok = bool(self.lib.newton_host_factor(n, s.w, _p(band)))
            if ok:
                break
        rec.update(shifts=a, factored=ok, tau=tau, beta=beta)
        st.tau, st.beta = tau, beta
        # k_newton_dir
        d = np.zeros(n)
        fallback = None
        if not ok:
            fallback = "factor"
        elif not self.lib.newton_host_range_step(n, s.w, self.r, _p(s.perm, ip), _p(self.Q1p), _p(band),
                                                 _p(np.ascontiguousarray(g)), _p(d)):
            fallback = "S"
        else:
            dg = coop_sum(d * g, self.nt)
            if not dg < 0.0:
                fallback = "slope"
        if fallback is not None:
            d = -pg
            dg = -coop_sum(pg * pg, self.nt)
        phi0 = f + 8.0 * EPS * abs(f)
        rec.update(fallback=fallback, d=d, dg=dg, phi0=phi0)
        # two_stage_search on the cost: k_alm_pick1, then k_alm_pick2 when stage 1 has no Armijo step
        alphas = np.ldexp(1.0, -np.arange(NALPHA))
        scale = max(1.0, abs(phi0))
        thr = phi0 + self.c1 * alphas * dg
        phi = self.f(x[None, :] + alphas[:NALPHA1, None] * d[None, :])
        margins = list(np.abs(phi - thr[:NALPHA1]) / scale)
        best, phib, chosen = 0, phi[0], -1
        for a in range(NALPHA1):
            if a == 0 or phi[a] < phib:
                best, phib = a, phi[a]
            if chosen < 0 and phi[a] <= thr[a]:
                chosen = a
        pick = chosen if chosen >= 0 else best
        stage2 = chosen < 0
        if stage2:
            phi2 = self.f(x[None, :] + alphas[NALPHA1:, None] * d[None, :])
            margins += list(np.abs(phi2 - thr[NALPHA1:]) / scale)
            best2, chosen2 = -1, -1
            for a in range(NALPHA - NALPHA1):
                if phi2[a] < phib:
                    best2, phib = a, phi2[a]
                if chosen2 < 0 and phi2[a] <= thr[NALPHA1 + a]:
                    chosen2 = a
            p2 = chosen2 if chosen2 >= 0 else best2
            if p2 >= 0:
                pick = NALPHA1 + p2
            phi = np.concatenate([phi, phi2])
        a_best, phi_best = float(alphas[pick]), float(phi[pick])
        # k_newton_update
        armijo = bool(phi_best <= phi0 + self.c1 * a_best * dg)
        rec.update(pick=pick, armijo=armijo, stage2=stage2, margin=float(min(margins[:pick + 1])),
                   fnew=phi_best, decrease=phi_best < f)
        if armijo:
            st.C = self.affine_step(Cpart, x, d, a_best)
        sv = np.array([st.tau, st.beta, float(st.stall)])
        done = self.lib.newton_host_after_search(_p(sv), int(armijo), a_best, phi_best, f)
        st.tau, st.stall = float(sv[0]), int(sv[2])
        st.iters += 1
        if done:
            st.status = done
        return st


def lockstep(nw, C0, K, Cpart=None, rejected=False):
    """one problem from C0 as solve_eq_newton(max_iter = k) leaves it for every k = 1..K.  Returns
    dict(snaps=[k = 0..K: C, f, iters, status, tau, beta, stall], recs=[per iteration run: the iterate() record])
    (snaps[0] is the state after k_newton_init).  rejected: per-problem bounds the device refused (status 5,
    C untouched)."""
    if rejected:
        st = State(np.asarray(C0, dtype=np.float64).copy(), status=5)
    else:
        st = nw.init(C0, Cpart)
    snaps, recs = [], []
    for k in range(K + 1):
        if k > 0:
            rec = {}
            st = nw.iterate(st, Cpart, rec)
            recs.append(rec)
        snaps.append(dict(state=st.copy(), C=st.C.copy(), iters=st.iters, status=st.status))
    fk = nw.f(np.array([s["C"] for s in snaps]))
    for s, fv in zip(snaps, fk):
        s["f"] = float(fv)
    return dict(snaps=snaps, recs=recs)


# ---- the setups of tests/test_newton_lockstep_host.py and tests/test_gpu_newton_lockstep.py ----------------------

def long_kincar(ninterv, nbps, name):
    """the lane change of configs.kincar over ninterv intervals per output"""
    from ntg_b200 import configs
    return dataclasses.replace(configs.kincar(nbps, constraints=False, name=name), ninterv=[ninterv, ninterv],
                               knots=None)


def kincar_rows(nbps, name):
    """the 2 x 64 lane change with x'' = 0 at every breakpoint as well: one equality row per breakpoint on x"""
    spec = long_kincar(64, nbps, name)
    lo = np.concatenate([spec.lowerb[:6], [0.0], spec.lowerb[6:12]])
    return dataclasses.replace(spec, ltc=np.array([[0.0, 0.0, 1.0, 0.0, 0.0, 0.0]]), lowerb=lo, upperb=lo.copy())


def kincar_free(name):
    """the 2 x 64 lane change without its end conditions: no linear row at all (r = 0); straight lines cost
    nothing, so the Hessian is singular"""
    return dataclasses.replace(long_kincar(64, 193, name), lic=None, lfc=None, lowerb=np.zeros(0), upperb=np.zeros(0))


def syn6_eq(order, mult, ninterv, cost_outputs, name):
    """syn6 without its nonlinear rows: the trajectory cost on cost_outputs (every derivative), each output's
    value pinned at t0 (lic) and t1 (lfc)"""
    from ntg_b200 import configs
    base = configs.syn6(ninterv, name=name)
    pin = np.zeros((6, 24))
    pin[np.arange(6), 4 * np.arange(6)] = 1.0
    v = np.concatenate([0.25 * np.arange(1, 7), -0.125 * np.arange(1, 7)])
    return dataclasses.replace(base, order=[order] * 6, mult=[mult] * 6, callbacks={"ucf": "syn6_ucf", "nltcf": ""},
                               nnltc=0, trajectoryconstrav=[],
                               trajectorycostav=[(j, d) for j in cost_outputs for d in range(4)],
                               lic=pin, lfc=pin.copy(), lowerb=v, upperb=v.copy())


def lane_bounds(spec, P, seed):
    """per-problem lane changes: x0 / xf of configs.kincar moved per problem, lower == upper"""
    rng = np.random.default_rng(seed)
    lo = np.tile(spec.lowerb, (P, 1))
    lo[:, 0] += rng.uniform(-2.0, 2.0, P)
    lo[:, 3] += rng.uniform(-1.0, 1.0, P)
    lo[:, 6] += rng.uniform(-5.0, 5.0, P)
    lo[:, 9] += rng.uniform(-1.0, 1.0, P)
    return np.ascontiguousarray(lo), np.ascontiguousarray(lo.copy())


def vdp40(name):
    from ntg_b200 import configs
    return dataclasses.replace(configs.vanderpol(121, constraints=False, name=name), ninterv=[40], knots=None)


def setup(name):
    """-> (spec, starts [P][nC], per-problem (lowerb, upperb) or None, indices of problems whose bounds are
    rejected, Kmax).  SHAPES holds each setup's (nC, K, w, r), computed with the host structure."""
    from ntg_b200 import configs

    def cfg3(spec, P, seed=11):
        return configs.coefficients("cfg3", P, spec, seed=seed)

    def uni(spec, P, r, seed):
        return np.random.default_rng(seed).uniform(-r, r, (P, spec.nC))

    if name == "lane16_bounds":
        spec = long_kincar(16, 49, "nl_lane16")
        lo, up = lane_bounds(spec, 129, 3)
        lo[5, 2] = np.nan                        # rejected: a NaN bound, lower above upper, an inconsistent pin
        lo[17, 4] = up[17, 4] + 1.0
        up[40, 7] += 0.5
        return spec, cfg3(spec, 129, 13), (lo, up), [5, 17, 40], 6
    spec, X, K = {
        "lane64": lambda: (lambda s: (s, cfg3(s, 129), 8))(long_kincar(64, 193, "nl_lane64")),
        "lane256": lambda: (lambda s: (s, cfg3(s, 3), 4))(long_kincar(256, 769, "nl_lane256")),
        "syn6_w63": lambda: (lambda s: (s, uni(s, 16, 1.0, 5), 6))(syn6_eq(8, 4, 4, range(5), "nl_syn6_w63")),
        "syn6_w64": lambda: (lambda s: (s, uni(s, 16, 1.0, 8), 6))(syn6_eq(7, 6, 6, range(4), "nl_syn6_w64")),
        "syn6_one": lambda: (lambda s: (s, uni(s, 8, 1.0, 6), 4))(syn6_eq(8, 4, 1, range(6), "nl_syn6_one")),
        "rows128": lambda: (lambda s: (s, cfg3(s, 5), 4))(kincar_rows(118, "nl_rows128")),
        "rows127": lambda: (lambda s: (s, cfg3(s, 5), 4))(kincar_rows(117, "nl_rows127")),
        "free": lambda: (lambda s: (s, cfg3(s, 16), 6))(kincar_free("nl_free")),
        "vdp40": lambda: (lambda s: (s, uni(s, 64, 2.0, 7), 8))(vdp40("nl_vdp40")),
    }[name]()
    return spec, X, None, [], K


SETUPS = ["lane64", "lane256", "syn6_w63", "syn6_w64", "syn6_one", "rows128", "rows127", "free", "lane16_bounds",
          "vdp40"]
SHAPES = {"lane64": (262, 18, 13, 12), "lane256": (1030, 18, 13, 12), "syn6_w63": (120, 60, 63, 12),
          "syn6_w64": (72, 48, 64, 12),
          "syn6_one": (48, 48, 47, 12), "rows128": (262, 18, 13, 128), "rows127": (262, 18, 13, 127),
          "free": (262, 18, 13, 0), "lane16_bounds": (70, 18, 13, 12), "vdp40": (83, 9, 4, 3)}
CONVEX = ["lane64", "lane256", "lane16_bounds"]   # rows12x: x is pinned, H is singular on null(A) to rounding


def references(nw, X, bounds, rejected, K):
    """lockstep() of every problem of a setup"""
    refs = []
    for p in range(X.shape[0]):
        Cp = None if bounds is None or p in rejected else nw.problem_cpart(bounds[0][p], bounds[1][p])
        refs.append(lockstep(nw, X[p], K, Cpart=Cp, rejected=p in rejected))
    return refs
