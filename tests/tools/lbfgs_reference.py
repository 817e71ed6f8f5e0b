"""Numpy restatement of the projected L-BFGS of ntgb_solve_eq_lbfgs (ntg_b200/csrc/ntg_lbfgs.h), for the CPU
tests: the projector, the two-loop recursion, the pair and reset rules, and a whole solve driven by any
evaluation function -- the same algorithm in the textbook form (Nocedal & Wright, Algorithm 7.4), so that the
header's ring indexing and reductions have something independent to be checked against."""
import numpy as np

SKIP_EPS = 1e-10    # ntg_lbfgs.h kSkipEps
N1, N2 = 4, 12      # two_stage_search: steps 2^-a, a < 4 for every problem, then 4 <= a < 16


def row_basis(A, tol=1e-11):
    """Q1 [r][n]: orthonormal rows spanning the rows of A"""
    if A.shape[0] == 0:
        return np.zeros((0, A.shape[1]))
    _, s, Vt = np.linalg.svd(A, full_matrices=False)
    return Vt[: int((s > tol * s[0]).sum())]


def project(Q1, v):
    """P v = v - Q1' (Q1 v)"""
    return v - Q1.T @ (Q1 @ v)


class History:
    """the pairs kept, oldest first, and what the header keeps next to them"""

    def __init__(self, mem):
        self.mem, self.S, self.U, self.gamma = mem, [], [], 1.0
        self.sv = self.gp = None    # the last step and the projected gradient where it started (pending pair)

    def push(self, s, u):
        """the pair rule: kept (the oldest dropped when full) unless s'u <= SKIP_EPS |s| |u|"""
        su = float(s @ u)
        if not su > SKIP_EPS * np.linalg.norm(s) * np.linalg.norm(u):
            return False
        self.S.append(s.copy()); self.U.append(u.copy())
        if len(self.S) > self.mem:
            self.S.pop(0); self.U.pop(0)
        self.gamma = su / float(u @ u)
        return True

    def reset(self):
        self.S, self.U = [], []


def two_loop(h, q):
    """H q with H0 = gamma I"""
    q = q.copy()
    rho = [1.0 / float(s @ u) for s, u in zip(h.S, h.U)]
    al = []
    for s, u, r in reversed(list(zip(h.S, h.U, rho))):
        a = r * float(s @ q)
        al.append(a)
        q -= a * u
    q *= h.gamma
    for (s, u, r), a in zip(zip(h.S, h.U, rho), reversed(al)):
        b = r * float(u @ q)
        q += (a - b) * s
    return q


def direction(Q1, h, f, g, gtol):
    """-> (status, d, d'g): status 1 converged, 2 NaN, 0 with the direction"""
    pg = project(Q1, g)
    gmax = np.abs(pg).max() if pg.size else 0.0
    if not gmax > gtol * max(1.0, abs(f)):
        return (1 if gmax == gmax else 2), None, 0.0
    if h.sv is not None:
        h.push(h.sv, pg - h.gp)
    h.gp = pg
    if h.S:
        d = -project(Q1, two_loop(h, pg))
        dg = float(d @ g)
        if dg < 0.0:
            return 0, d, dg
        h.reset()
    dd = float(pg @ pg)
    scale = 1.0 / np.sqrt(dd) if np.sqrt(dd) > 1.0 else 1.0
    return 0, -scale * pg, -dd * scale


def search(fcost, C, d, f0, dg, c1):
    """two_stage_search on the plain cost -> (alpha, phi): the first Armijo step among 1 .. 1/8, else among
    2^-4 .. 2^-15, else the smallest cost seen (ties to the earlier step)"""
    alphas = [2.0 ** -a for a in range(N1 + N2)]
    phis = [fcost(C + a * d) for a in alphas[:N1]]
    for a, ph in zip(alphas[:N1], phis):
        if ph <= f0 + c1 * a * dg:
            return a, ph
    best = int(np.argmin(phis))
    ab, pb = alphas[best], phis[best]
    for a in alphas[N1:]:
        ph = fcost(C + a * d)
        if ph <= f0 + c1 * a * dg:
            return a, ph
        if ph < pb:
            ab, pb = a, ph
    return ab, pb


def solve(fg, Q1, Cpart, C, max_iter=500, gtol=1e-9, c1=1e-4, mem=8):
    """projected L-BFGS from C on {Cpart + null(A)}; fg(C) -> (f, g).  -> (C, status, iterations)"""
    h = History(mem)
    C = Cpart + project(Q1, C - Cpart)
    for it in range(max_iter):
        f, g = fg(C)
        st, d, dg = direction(Q1, h, f, g, gtol)
        if st:
            return C, st, it
        a, ph = search(lambda x: fg(x)[0], C, d, f, dg, c1)
        if not ph < f:
            if not h.S:
                return C, 2, it + 1
            h.reset()
            h.sv = None
            continue
        Cn = Cpart + project(Q1, C + a * d - Cpart)
        h.sv = Cn - C
        C = Cn
    return C, 0, max_iter
