/*
 * ntg_lbfgs.h -- the per-problem core of the projected L-BFGS solver (ntgb_solve_eq_lbfgs): a smooth cost
 * on the affine set A C = b, with no null-space basis.  The projector onto null(A) is P v = v - Q1 (Q1' v),
 * Q1 [r][nC] the orthonormal rows of the row space of A (the first r columns of the Q that ntg_core.cu's
 * reduce_linear builds), so the work per problem is O(nC (r + memory)) whatever the number nC - r of free
 * directions.
 *
 *   pairs      s = C_k - C_{k-1} (the step taken), u = P (g_k - g_{k-1}); the pair is skipped when
 *              s'u <= kSkipEps |s| |u| (too little curvature seen to keep H positive definite)
 *   H0         gamma I, gamma = s'u / u'u of the newest pair kept
 *   direction  d = -P (H P g) by the two-loop recursion on the ring of the last `memory` pairs, projected
 *              again so that rounding in the recursion does not leave null(A); if d'g >= 0 the history is
 *              dropped and d = -P g
 *   converged  |P g|_inf <= gtol max(1, |f|) (status 1); a NaN there is status 2
 *   steps      C <- Cpart + P (C + a d - Cpart): every accepted step lands on the affine set again
 *
 * The code is plain C++ over sqp::Coop (tid, nt and a fixed-order reduction, ntg_sqp.cuh): k_lbfgs_dir,
 * k_lbfgs_update and k_lbfgs_init run it with one CTA per problem, and tests/tools/lbfgs_host.cpp compiles
 * THE SAME TEXT with g++ for a group of one thread, checked against tests/tools/lbfgs_reference.py.
 * Every reduction's order depends only on nC and the CTA size, never on the batch.
 */
#ifndef NTG_LBFGS_H_
#define NTG_LBFGS_H_

#include <math.h>

#include "ntg_sqp.cuh"

namespace ntgb {
namespace lbfgs {

constexpr int kMaxMemory = 32;     /* curvature pairs kept per problem, at most */
constexpr double kSkipEps = 1e-10; /* skip a pair when s'u <= kSkipEps |s| |u| */

/* one problem's arrays */
struct View {
    const double *Q1; /* [r][n], shared by all problems */
    int r, n, mem;
    double *ring;     /* [mem][2][n]: pair i is s = ring + 2 i n, u = s + n */
    double *rho;      /* [mem] 1 / s'u of pair i */
    double *sv;       /* [n] the last step taken */
    double *gp;       /* [n] P g where it was taken */
};

/* one problem's scalars: the ring's next slot, the pairs kept, 1 when sv / gp hold a step not yet paired,
 * the scale of H0 */
struct State {
    int head, npair, pend;
    double gamma;
};

/* Q1 is shared by the whole batch and only read: through L2 on the device */
NTG_HD inline double ld_shared(const double *p)
{
#ifdef __CUDA_ARCH__
    return __ldcg(p);
#else
    return *p;
#endif
}

/* v <- P v, one row of Q1 at a time (modified Gram-Schmidt: the same projector as v - Q1 (Q1' v) for
 * orthonormal rows, with less rounding) */
template <class C>
NTG_HD void project(const C &cg, double *red, const double *Q1, int r, int n, double *v)
{
    for (int k = 0; k < r; k++) {
        const double *q = Q1 + (size_t)k * n;
        double w = 0.0;
        for (int e = cg.tid; e < n; e += cg.nt) w += ld_shared(q + e) * v[e];
        w = cg.template reduce<false>(w, red);
        for (int e = cg.tid; e < n; e += cg.nt) v[e] -= w * ld_shared(q + e);
    }
}

/* x'y over the group */
template <class C>
NTG_HD double dot(const C &cg, double *red, const double *x, const double *y, int n)
{
    double a = 0.0;
    for (int e = cg.tid; e < n; e += cg.nt) a += x[e] * y[e];
    return cg.template reduce<false>(a, red);
}

/* q <- H q: the two-loop recursion over the npair newest pairs, H0 = gamma I */
template <class C>
NTG_HD void two_loop(const C &cg, double *red, const View &v, const State &s, double *q)
{
    const int n = v.n;
    double al[kMaxMemory];
    for (int j = 0; j < s.npair; j++) { /* newest first */
        const int i = (s.head - 1 - j + 2 * v.mem) % v.mem;
        const double *si = v.ring + (size_t)2 * i * n, *ui = si + n;
        const double a = v.rho[i] * dot(cg, red, si, q, n);
        al[j] = a;
        for (int e = cg.tid; e < n; e += cg.nt) q[e] -= a * ui[e];
    }
    for (int e = cg.tid; e < n; e += cg.nt) q[e] *= s.gamma;
    for (int j = s.npair - 1; j >= 0; j--) { /* oldest first */
        const int i = (s.head - 1 - j + 2 * v.mem) % v.mem;
        const double *si = v.ring + (size_t)2 * i * n, *ui = si + n;
        const double b = v.rho[i] * dot(cg, red, ui, q, n);
        for (int e = cg.tid; e < n; e += cg.nt) q[e] += (al[j] - b) * si[e];
    }
}

/* One direction step of one problem at cost f and gradient g.  Returns 1 (converged) or 2 (NaN) and
 * leaves d undefined, or 0 with the search direction in d and its slope dg = d'g.  Pairs the pending
 * step with this gradient first.  A steepest-descent direction (no pair kept) longer than 1 is scaled
 * to length 1: a unit step along a raw gradient can be far too long. */
template <class C>
NTG_HD int direction(const C &cg, double *red, const View &v, State &s, double f, const double *g, double gtol,
                     double *d, double &dg)
{
    const int n = v.n;
    for (int e = cg.tid; e < n; e += cg.nt) d[e] = g[e];
    project(cg, red, v.Q1, v.r, n, d);
    double gmax = 0.0, gg = 0.0;
    for (int e = cg.tid; e < n; e += cg.nt) {
        gmax = fmax(gmax, fabs(d[e]));
        gg += d[e] * d[e];
    }
    gmax = cg.template reduce<true>(gmax, red);
    gg = cg.template reduce<false>(gg, red); /* fmax drops a NaN, the sum keeps it */
    if (gg != gg) return 2;
    const double fa = fabs(f);
    if (!(gmax > gtol * (fa > 1.0 ? fa : 1.0))) return 1;
    if (s.pend) {
        double su = 0.0, ss = 0.0, uu = 0.0;
        for (int e = cg.tid; e < n; e += cg.nt) {
            const double se = v.sv[e], ue = d[e] - v.gp[e];
            su += se * ue;
            ss += se * se;
            uu += ue * ue;
        }
        su = cg.template reduce<false>(su, red);
        ss = cg.template reduce<false>(ss, red);
        uu = cg.template reduce<false>(uu, red);
        if (su > kSkipEps * sqrt(ss) * sqrt(uu)) {
            double *si = v.ring + (size_t)2 * s.head * n, *ui = si + n;
            for (int e = cg.tid; e < n; e += cg.nt) {
                si[e] = v.sv[e];
                ui[e] = d[e] - v.gp[e];
            }
            v.rho[s.head] = 1.0 / su; /* every thread writes the same value */
            s.gamma = su / uu;
            s.head = (s.head + 1) % v.mem;
            s.npair = s.npair < v.mem ? s.npair + 1 : v.mem;
        }
    }
    for (int e = cg.tid; e < n; e += cg.nt) v.gp[e] = d[e];
    if (s.npair > 0) {
        two_loop(cg, red, v, s, d);
        project(cg, red, v.Q1, v.r, n, d);
        for (int e = cg.tid; e < n; e += cg.nt) d[e] = -d[e];
        dg = dot(cg, red, d, g, n);
        if (dg < 0.0) return 0;
        s.npair = 0; /* not a descent direction: drop the history */
    }
    const double dn = sqrt(gg), scale = dn > 1.0 ? 1.0 / dn : 1.0;
    for (int e = cg.tid; e < n; e += cg.nt) d[e] = -scale * v.gp[e];
    dg = -gg * scale;
    return 0;
}

/* C <- Cpart + P (C + a d - Cpart) and sv <- the step taken (new C - old C); d == nullptr: the projection of
 * C onto the affine set, as at entry */
template <class C>
NTG_HD void affine_step(const C &cg, double *red, const View &v, const double *Cpart, double *Cv, const double *d,
                        double a)
{
    const int n = v.n;
    for (int e = cg.tid; e < n; e += cg.nt) v.sv[e] = (d != nullptr ? Cv[e] + a * d[e] : Cv[e]) - Cpart[e];
    project(cg, red, v.Q1, v.r, n, v.sv);
    for (int e = cg.tid; e < n; e += cg.nt) {
        const double c = Cpart[e] + v.sv[e];
        v.sv[e] = c - Cv[e];
        Cv[e] = c;
    }
}

/* After the line search: decreased (phi_best < phi0) -> take the step, pair it at the next direction;
 * else drop the history and retry from steepest descent, or return 2 (no further decrease) when the
 * direction already was steepest descent.  Returns 0 otherwise. */
template <class C>
NTG_HD int accept(const C &cg, double *red, const View &v, State &s, const double *Cpart, double *Cv, const double *d,
                  double a, double phi0, double phi_best)
{
    if (!(phi_best < phi0)) {
        if (s.npair == 0) return 2;
        s.npair = 0;
        s.pend = 0;
        return 0;
    }
    affine_step(cg, red, v, Cpart, Cv, d, a);
    s.pend = 1;
    return 0;
}

} /* namespace lbfgs */
} /* namespace ntgb */

#endif
