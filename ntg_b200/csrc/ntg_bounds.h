/*
 * ntg_bounds.h -- per-problem constraint bounds of the batched solvers (ntgb_solve_eq_bounds,
 * ntgb_solve_sqp_bounds) as plain host/device code: how one problem's COMPACT bounds (one value per
 * constraint, the layout of ntgb_setup.lowerb / upperb) expand into the rows the solvers use, which
 * bounds are rejected, and the minimum-norm solution Cpart = M be of its eliminated equality rows.
 *
 * k_bounds_prep (ntg_core.cu) runs this with one warp per problem (start = lane, step = 32); the CPU
 * test suite compiles THE SAME TEXT with g++ (start 0, step 1) and checks the expansion bit for bit
 * against the oracle's bounds() (tests/test_bounds_host.py, tests/tools/bounds_host.cpp).
 */
#ifndef NTG_BOUNDS_H_
#define NTG_BOUNDS_H_

#include <stddef.h>

#ifndef NTG_HD
#if defined(__CUDACC__)
#define NTG_HD __host__ __device__
#else
#define NTG_HD
#endif
#endif

namespace ntgb {

/* why a problem's bounds are rejected (bits; any of them gives the problem NTGB_STATUS_BAD_BOUNDS) */
constexpr unsigned kBoundsNaN = 1u;          /* a NaN bound                                          */
constexpr unsigned kBoundsCrossed = 2u;      /* lower > upper                                         */
constexpr unsigned kBoundsNotEqual = 4u;     /* a row the setup eliminates as an equality: lower != upper */
constexpr unsigned kBoundsInconsistent = 8u; /* eliminated equality rows without a common solution
                                              * (only possible when the setup's equality rows are dependent) */

/* constraint counts of the setup: compact bounds are [nlic | nltc | nlfc | nnlic | nnltc | nnlfc] */
struct BoundsLayout {
    int nlic, nltc, nlfc, nnlic, nnltc, nnlfc, nbps;
    NTG_HD int nb() const { return nlic + nltc + nlfc + nnlic + nnltc + nnlfc; }
    NTG_HD int nclin() const { return nlic + nltc * nbps + nlfc; }
    NTG_HD int ncnln() const { return nnlic + nnltc * nbps + nnlfc; }
};

/* compact index of expanded linear row r (NPSOL's order: initial, trajectory breakpoint-fastest, final;
 * reference src/constraints.c:5-33, ntgb_get_bounds) */
NTG_HD inline int bounds_lin_src(const BoundsLayout &L, int r)
{
    if (r < L.nlic) return r;
    r -= L.nlic;
    if (r < L.nltc * L.nbps) return L.nlic + r / L.nbps;
    return L.nlic + L.nltc + (r - L.nltc * L.nbps);
}

/* compact index of expanded nonlinear row r */
NTG_HD inline int bounds_nl_src(const BoundsLayout &L, int r)
{
    const int base = L.nlic + L.nltc + L.nlfc;
    if (r < L.nnlic) return base + r;
    r -= L.nnlic;
    if (r < L.nnltc * L.nbps) return base + L.nnlic + r / L.nbps;
    return base + L.nnlic + L.nnltc + (r - L.nnltc * L.nbps);
}

/*
 * One problem's compact bounds lo / up [nb] into
 *   hl / hu [n_li + ncnln]  the SQP's general rows: linear rows li[0..n_li) (the ones the setup keeps as
 *                           inequalities), then every nonlinear row;
 *   be [me]                 right-hand sides of the eliminated linear rows eq[0..me) (eq == nullptr:
 *                           row r itself).
 * Handles entries start, start + step, ... of each list and returns the rejection bits seen there.
 * Values are copied, never rounded: |b| >= 1e19 stays "no bound" (ntg_sqp.cuh kBig).
 */
NTG_HD inline unsigned bounds_expand(const BoundsLayout &L, const double *lo, const double *up, const int *li, int n_li,
                                     const int *eq, int me, double *hl, double *hu, double *be, int start, int step)
{
    unsigned bad = 0;
    const int nb = L.nb();
    for (int k = start; k < nb; k += step) {
        const double l = lo[k], u = up[k];
        if (l != l || u != u) bad |= kBoundsNaN;
        else if (l > u) bad |= kBoundsCrossed;
    }
    const int m = n_li + L.ncnln();
    for (int i = start; i < m; i += step) {
        const int k = i < n_li ? bounds_lin_src(L, li[i]) : bounds_nl_src(L, i - n_li);
        hl[i] = lo[k];
        hu[i] = up[k];
    }
    for (int r = start; r < me; r += step) {
        const int k = bounds_lin_src(L, eq != nullptr ? eq[r] : r);
        const double l = lo[k], u = up[k];
        if (l == l && u == u && l != u) bad |= kBoundsNotEqual;
        be[r] = l;
    }
    return bad;
}

/* element e of Cpart = M be (M [nC][me] row-major: reduce_linear's operator) */
NTG_HD inline double bounds_cpart(const double *M, int me, const double *be, int e)
{
    double a = 0.0;
    for (int j = 0; j < me; j++) a += M[(size_t)e * me + j] * be[j];
    return a;
}

/* residual Ae_r . Cpart - b_r of one eliminated row (Ae_r [nC]), summed in reduce_linear's order */
NTG_HD inline double bounds_residual(const double *Ae_r, int nC, const double *Cpart, double b)
{
    double a = -b;
    for (int i = 0; i < nC; i++) a += Ae_r[i] * Cpart[i];
    return a;
}

/* max that keeps a NaN (fmax drops it): the largest residual of a problem */
NTG_HD inline double bounds_max(double a, double b) { return (b != b || b > a) ? b : a; }

/* reduce_linear's tolerance for inconsistent equality rows: max |residual| > 1e-8 (1 + |b|_inf); a NaN
 * residual (an infinite right-hand side) is inconsistent too */
NTG_HD inline bool bounds_inconsistent(double res, double bmax) { return !(res <= 1e-8 * (1.0 + bmax)); }

} /* namespace ntgb */

#endif /* NTG_BOUNDS_H_ */
