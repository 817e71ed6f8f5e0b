"""tests/tools/sqp_lockstep.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The batched SQP solver (ntgb_solve_sqp, ntgb_solve_sqp_bounds, ntgb_solve_sqp_warm) followed iteration by
iteration on the host, so that a GPU solve stopped after K iterations can be compared with the same K
iterations here.  It restates what ntg_core.cu does around the per-problem core:

  * the reduced space: reduce_linear (Householder QR of A_eq' with column pivoting) written with plain
    float loops in the C++ loop order, so that N, Cpart and Mop come out bit for bit as the library's --
    the warm-row digest proves it on the GPU.  An SVD basis would not do: the row scales of the QP and the
    gtol test use infinity norms in reduced coordinates, which are not rotation-invariant;
  * the general rows in alm_prepare's order [linear inequality rows in index order; nonlinear rows];
  * k_sqp_init (y = N (C - Cpart), C = Cpart + N' y, B and nu from a matching warm row);
  * the K line-searched steps of solve_sqp_impl plus its final direction() pass, which applies the BFGS
    update at the final point and solves the QP whose multipliers and active set are reported;
  * the two-stage Armijo search (k_alm_pick1 over alpha = 2^-a, a = 0..3; k_alm_pick2 over a = 4..15 only
    when stage 1 found no Armijo point) and k_sqp_update;
  * the multipliers of the eliminated equality rows (k_alm_grad, then k_sqp_outputs: the least-squares
    solution of Ae' le = g - A_in' l_in - J' l_nl).

Each direction comes from the g++-compiled core of ntg_sqp.cuh (tests/tools/sqp_host.cpp, a group of one
thread); every evaluation is the CPU oracle's, in float64, with the dense Jacobian.  The driver records the
step index each line search chose and how far each decision sat from the Armijo threshold, so that a test
can tell a real disagreement from a decision within rounding of it.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math

import numpy as np

KBIG = 1e19
NALPHA1, NALPHA = 4, 16


def fnv1a(data: bytes) -> int:
    h = 14695981039346656037
    for b in data:
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def reduce_linear(Ae, b, q1=False):
    """reduce_linear (ntg_core.cu) for the rows Ae [m][n] and right-hand side b [m]: N [nr][n], Cpart [n],
    Mop [n][m] (Cpart = Mop b for any b; zero columns for rows found dependent), rank r, and with q1=True
    also Q1 [r][n] (the first r columns of Q, the row-space basis of ntgb_solve_eq_lbfgs / _newton).  Same
    operations in the same order as the C++ (no FMA contraction on the host), so the results are
    bit-identical: every sequential sum of the C++ stays sequential here, numpy only runs the independent
    sums of different columns side by side, one elementwise IEEE operation at a time."""
    m, n = int(Ae.shape[0]), int(Ae.shape[1])
    M = np.array(Ae, dtype=np.float64).reshape(m, n).copy()      # M[j] = column j of A'
    Q = np.eye(n)
    perm = list(range(m))
    r, norm0 = 0, 0.0
    for k in range(min(n, m)):
        a = np.zeros(m - k)
        for i in range(k, n):
            a = a + M[k:, i] * M[k:, i]
        jb = k + int(np.argmax(a))                               # the first largest, as `if (a > nb)`
        norm = math.sqrt(a[jb - k])
        if k == 0:
            norm0 = norm
        if not (norm > 1e-11 * max(norm0, 1e-300)):
            break
        if jb != k:
            M[[k, jb]] = M[[jb, k]]
            perm[k], perm[jb] = perm[jb], perm[k]
        alpha = -norm if M[k, k] > 0.0 else norm
        v = np.zeros(n)
        v[k:] = M[k, k:]
        v[k] -= alpha
        vv = 0.0
        for x in v[k:].tolist():
            vv += x * x
        if vv > 0.0:
            t = np.zeros(m - k)
            for i in range(k, n):
                t = t + v[i] * M[k:, i]
            t = 2.0 * t / vv
            M[k:, k:] = M[k:, k:] - t[:, None] * v[None, k:]
            t = np.zeros(n)
            for l in range(k, n):
                t = t + Q[:, l] * v[l]
            t = 2.0 * t / vv
            Q[:, k:] = Q[:, k:] - t[:, None] * v[None, k:]
        r += 1

    def back(R):
        """the back substitution for the right-hand sides R [m][q] at once, then Q1 w"""
        w = np.zeros((r, R.shape[1]))
        for i in range(r):
            a = R[perm[i]].copy()
            for l in range(i):
                a = a - M[i, l] * w[l]
            w[i] = a / M[i, i]
        out = np.zeros((n, R.shape[1]))
        for l in range(r):
            out = out + Q[:, l:l + 1] * w[l][None, :]
        return out

    Cpart = back(np.asarray(b, dtype=np.float64).reshape(m, 1))[:, 0].copy()
    Mop = back(np.eye(m)) if m else np.zeros((n, 0))
    N = np.ascontiguousarray(Q[:, r:].T)
    if q1:
        return N, Cpart, Mop, r, np.ascontiguousarray(Q[:, :r].T)
    return N, Cpart, Mop, r


def with_bounds(spec, lo, up):
    kw = {f.name: getattr(spec, f.name) for f in dataclasses.fields(spec)}
    kw.update(lowerb=np.asarray(lo, dtype=np.float64).copy(), upperb=np.asarray(up, dtype=np.float64).copy())
    return type(spec)(**kw)


class Reduced:
    """the reduced form alm_prepare / solve_sqp_impl build for a setup, restated on the host"""

    def __init__(self, port, spec):
        self.port, self.spec = port, spec
        nC, nclin = spec.nC, spec.nclin
        o = port.eval(spec, np.zeros((1, nC)), mode_obj=0, mode_con=0, dense=False, band=False, linear=True)
        self.A = o["A"]                                   # [nclin][nC]
        lb, ub = o["bl"][nC:nC + nclin], o["bu"][nC:nC + nclin]
        self.eq = [i for i in range(nclin) if lb[i] == ub[i]]
        self.li = [i for i in range(nclin) if lb[i] != ub[i]]
        self.Ae = self.A[self.eq].reshape(len(self.eq), nC)
        self.N, self.Cpart, self.Mop, _ = reduce_linear(self.Ae, lb[self.eq])
        self.nC, self.nr, self.n_li = nC, self.N.shape[0], len(self.li)
        self.m = self.n_li + spec.ncnln
        # reduced gradients of the linear inequality rows, summed in solve_sqp_impl's order
        self.ArN = np.zeros((self.n_li, self.nr))
        for i, row in enumerate(self.li):
            for k in range(self.nr):
                a = 0.0
                for e in range(nC):
                    a += float(self.A[row, e]) * float(self.N[k, e])
                self.ArN[i, k] = a
        self.hl, self.hu = self._rows(o["bl"], o["bu"])

    def digest(self) -> int:
        """what ntgb_solve_sqp_warm writes into a row's header: FNV-1a of (nC, nr, m, n_li, li, N)"""
        head = np.array([self.nC, self.nr, self.m, self.n_li], dtype="<i4").tobytes()
        return fnv1a(head + np.array(self.li, dtype="<i4").tobytes() + np.ascontiguousarray(self.N, dtype="<f8").tobytes())

    def _rows(self, bl, bu):
        nC, nclin = self.nC, self.spec.nclin
        hl = np.concatenate([bl[nC:nC + nclin][self.li], bl[nC + nclin:]])
        hu = np.concatenate([bu[nC:nC + nclin][self.li], bu[nC + nclin:]])
        return hl, hu

    def problem_bounds(self, lo, up):
        """per-problem compact bounds -> (hl, hu, Cpart): the rows' bounds and Cpart = Mop be, summed in
        ntg_bounds.h's order"""
        nC = self.nC
        o = self.port.eval(with_bounds(self.spec, lo, up), np.zeros((1, nC)), mode_obj=0, mode_con=0, dense=False,
                           band=False, linear=True)
        be = o["bl"][nC:nC + self.spec.nclin][self.eq]
        Cp = np.zeros(nC)
        for e in range(nC):
            a = 0.0
            for j in range(len(self.eq)):
                a += float(self.Mop[e, j]) * float(be[j])
            Cp[e] = a
        hl, hu = self._rows(o["bl"], o["bu"])
        return hl, hu, Cp

    def evaluate(self, X, deriv):
        """f, g, h = [A_in C; c(C)], J [ncnln][nC] (dense, zeros where the pattern has no entry) at the rows of X"""
        spec = self.spec
        if deriv:
            e = self.port.eval(spec, X, mode_obj=2, mode_con=2 if spec.ncnln else -1, dense=True, band=False)
        else:
            e = self.port.eval(spec, X, mode_obj=0, mode_con=0 if spec.ncnln else -1, dense=False, band=False)
        h = np.concatenate([X @ self.A[self.li].T if self.n_li else np.zeros((X.shape[0], 0)),
                            e["c"] if spec.ncnln else np.zeros((X.shape[0], 0))], axis=1)
        J = None
        if deriv:
            J = (np.nan_to_num(e["Jdense"], nan=0.0).transpose(0, 2, 1) if spec.ncnln
                 else np.zeros((X.shape[0], 0, self.nC)))
        return e["f"], e["g"], h, J


def row_violation(h, hl, hu):
    v = np.zeros_like(h)
    lo = (hl > -KBIG) & (hl - h > v)
    v = np.where(lo, hl - h, v)
    hi = (hu < KBIG) & (h - hu > v)
    return np.where(hi, h - hu, v)


def warm_row_state(row, nr):
    """what k_sqp_init takes from a matching warm row (ntg_warm.h warm_load / warm_nu): B from the lower
    triangle, nu clamped to a finite value >= 0"""
    Br = np.asarray(row[6:6 + nr * nr], dtype=np.float64).reshape(nr, nr)
    B = np.tril(Br) + np.tril(Br, -1).T
    nu = float(row[5])
    return B, (nu if 0.0 <= nu <= 1.7976931348623157e308 else 0.0)


class Core:
    """the g++-compiled sqp_step (tests/tools/sqp_host.cpp).  noise (a numpy Generator): every entry of the
    reduced gradient and of the row gradients is moved by one unit in the last place, up or down at random
    -- what a different summation order does to them on the GPU"""

    def __init__(self, lib, noise=None):
        self.lib, self.noise = lib, noise
        lib.sqp_host_step.argtypes = ([C.c_int, C.c_int, C.c_double] + [C.POINTER(C.c_double)] * 12
                                      + [C.POINTER(C.c_int)] * 2 + [C.c_double] * 3)
        lib.sqp_host_step.restype = None

    def step(self, s, f, gr, h, hl, hu, Ar, gtol, ctol, rho_pen):
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
        gr, h, Ar = (np.ascontiguousarray(a, dtype=np.float64) for a in (gr, h, Ar))
        if self.noise is not None:
            gr, Ar = (a * (1.0 + 2.0 ** -52 * self.noise.choice([-1.0, 1.0], a.shape)) for a in (gr, Ar))
        self.lib.sqp_host_step(s["nr"], s["m"], float(f), dp(gr), dp(h), dp(hl), dp(hu), dp(Ar), dp(s["B"]), dp(s["lam"]),
                               dp(s["sprev"]), dp(s["grLold"]), dp(s["grold"]), dp(s["d"]), dp(s["scal"]), ip(s["flag"]),
                               ip(s["istate"]), gtol, ctol, rho_pen)


def lockstep(core, red, C0, K, hl=None, hu=None, Cpart=None, B0=None, nu0=0.0, gtol=1e-6, ctol=1e-8, rho_pen=1e4,
             c1=1e-4):
    """One problem from C0, as solve_sqp_impl runs it with max_iter = k for every k = 1..K at once (a run
    with max_iter = k is a prefix of the run with max_iter = K: its final pass is the (k+1)-th direction).
    hl / hu / Cpart: per-problem bounds (default: the setup's).  B0 / nu0: start from a warm row's state.

    Returns dict(C0=C after k_sqp_init, snaps=[snapshot for max_iter = k, k = 0..K], steps=[per line search:
    dict(a=chosen index, accepted, margin, stage2=whether stage 2 ran)]).  A snapshot holds what the solve reports: C, f, viol, status,
    iters, lam / istate (NPSOL order over [linear rows; nonlinear rows], eliminated rows included), and the
    warm row's B and nu."""
    nr, m, nC, n_li = red.nr, red.m, red.nC, red.n_li
    hl = np.ascontiguousarray(red.hl if hl is None else hl, dtype=np.float64)
    hu = np.ascontiguousarray(red.hu if hu is None else hu, dtype=np.float64)
    Cpart = red.Cpart if Cpart is None else np.asarray(Cpart, dtype=np.float64)
    N = red.N
    s = dict(nr=nr, m=m, B=np.eye(nr).ravel().copy(), lam=np.zeros(max(m, 1)), sprev=np.zeros(nr), grLold=np.zeros(nr),
             grold=np.zeros(nr), d=np.zeros(nr), scal=np.zeros(8), flag=np.zeros(8, dtype=np.int32),
             istate=np.zeros(max(m, 1), dtype=np.int32))
    if B0 is None:
        s["flag"][3] = 1
    else:
        s["B"][:] = np.asarray(B0, dtype=np.float64).ravel()
        s["scal"][0] = nu0
    y = N @ (np.asarray(C0, dtype=np.float64) - Cpart)
    C = Cpart + N.T @ y
    out = dict(C0=C.copy(), snaps=[], steps=[])
    status, iters = 0, 0
    f = g = J = None
    nclin = red.spec.nclin
    for it in range(K + 1):
        f, g, h, J = (a[0] for a in red.evaluate(C[None, :], True))
        if status == 0:
            Ar = np.vstack([red.ArN, J @ N.T]) if m else np.zeros((0, nr))
            core.step(s, f, N @ g, h, hl, hu, Ar, gtol, ctol, rho_pen)
            if s["flag"][5] != 0:
                status = int(s["flag"][5])
        # what a solve with max_iter = it reports
        lam_full = np.zeros(nclin + red.spec.ncnln)
        ist_full = np.zeros(nclin + red.spec.ncnln, dtype=np.int32)
        rows = list(red.li) + list(range(nclin, nclin + red.spec.ncnln))
        lam_full[rows] = s["lam"][:m]
        ist_full[rows] = s["istate"][:m]
        if red.eq:
            gL = g - red.A[red.li].T @ s["lam"][:n_li] - J.T @ s["lam"][n_li:m]
            lam_full[red.eq] = np.linalg.lstsq(red.Ae.T, gL, rcond=None)[0]
            ist_full[red.eq] = 3
        out["snaps"].append(dict(C=C.copy(), f=float(f), viol=float(s["scal"][3]), status=status, iters=iters,
                                 lam=lam_full, istate=ist_full, B=s["B"].reshape(nr, nr).copy(), nu=float(s["scal"][0])))
        if it == K:
            break
        if status != 0:
            continue
        # ---- two-stage Armijo search on the L1 merit (k_sqp_merit, k_alm_pick1, k_alm_pick2) ----
        nu, phi0, D = s["scal"][0], s["scal"][1], s["scal"][2]
        dC = N.T @ s["d"]
        scale = max(1.0, abs(phi0))

        def merit(a0, a1):
            al = np.ldexp(1.0, -np.arange(a0, a1))
            ft, _, ht, _ = red.evaluate(C[None, :] + al[:, None] * dC[None, :], False)
            return al, ft + nu * row_violation(ht, hl[None, :], hu[None, :]).sum(axis=1)

        al, phi = merit(0, NALPHA1)
        armijo = phi <= phi0 + c1 * al * D
        margins = list(np.abs(phi - (phi0 + c1 * al * D)) / scale)
        best, phib = 0, phi[0]
        for a in range(1, NALPHA1):
            if phi[a] < phib:
                best, phib = a, phi[a]
        if armijo.any():
            pick = int(np.argmax(armijo))
            margin = min(margins[:pick + 1])
        else:
            pick = best
            al2, phi2 = merit(NALPHA1, NALPHA)
            armijo2 = phi2 <= phi0 + c1 * al2 * D
            margins += list(np.abs(phi2 - (phi0 + c1 * al2 * D)) / scale)
            best2 = -1
            for a in range(NALPHA - NALPHA1):
                if phi2[a] < phib:
                    best2, phib = a, phi2[a]
            if armijo2.any():
                pick = NALPHA1 + int(np.argmax(armijo2))
                margin = min(margins[:pick + 1])
            else:
                if best2 >= 0:
                    pick = NALPHA1 + best2
                margin = min(min(margins), abs(phib - phi0) / scale)
            al, phi = np.concatenate([al, al2]), np.concatenate([phi, phi2])
        # ---- k_sqp_update ----
        iters += 1
        accepted = bool(phi[pick] < phi0)
        out["steps"].append(dict(a=pick, accepted=accepted, margin=float(margin), stage2=len(phi) > NALPHA1))
        if not accepted:
            if s["flag"][3]:
                status = 2
            else:
                s["flag"][2], s["flag"][0] = 1, 0
            continue
        s["sprev"][:] = al[pick] * s["d"]
        y = y + s["sprev"]
        C = Cpart + N.T @ y
        s["flag"][0], s["flag"][1] = 1, s["flag"][4]
    return out


QUANTITIES = ("C", "f", "viol", "B", "nu", "lam")


def rel_diff(a, b):
    """max |a - b| scaled by max(1, |b|_inf)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max(initial=0.0)) / max(1.0, float(np.abs(b).max(initial=0.0)))


def rounding_spread(lib, red, C0, K, ref, seeds=3, **kw):
    """How far rounding alone moves the snapshots of one problem: `ref` (the lockstep() result) against
    reruns whose core sees its inputs moved by one unit in the last place (Core(noise=)).  Returns
    (spread {(k, quantity): largest rel_diff}, first k whose discrete outcome -- status, iterations, active
    set, chosen step -- differs in a rerun, or None).  A problem can amplify rounding by many orders of
    magnitude (a first quasi-Newton update from a huge step, a restoration step with a large penalty); a
    comparison with another implementation of the same arithmetic cannot be tighter than this."""
    spread = {(k, q): 0.0 for k in range(K + 1) for q in QUANTITIES}
    flip = None
    for seed in range(seeds):
        r = lockstep(Core(lib, noise=np.random.default_rng(seed)), red, C0, K, **kw)
        for k in range(K + 1):
            a, b = r["snaps"][k], ref["snaps"][k]
            same = (a["status"] == b["status"] and a["iters"] == b["iters"] and np.array_equal(a["istate"], b["istate"])
                    and [s["a"] for s in r["steps"][:k]] == [s["a"] for s in ref["steps"][:k]])
            if not same:
                flip = k if flip is None else min(flip, k)
                break
            for q in QUANTITIES:
                spread[(k, q)] = max(spread[(k, q)], rel_diff(a[q], b[q]))
    return spread, flip


# ---- shared memory of one k_sqp_step CTA (ntg_sqp.cuh sqp_smem_doubles / sqp_smem_ints) ------------------

def sqp_threads(nr):
    return 32 if nr < 32 else 64


def sqp_smem_bytes(nr, m):
    nt, ld = sqp_threads(nr), nr | 1
    nd = 4 * nr * ld + m * ld + 5 * m + 9 * nr + 2 + 4 * nr + m + nt + 4
    ni = nr + 1 + m + nt + 4
    return 8 * nd + 4 * ni
