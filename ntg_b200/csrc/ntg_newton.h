/*
 * ntg_newton.h -- the banded Newton solver of ntgb_solve_eq_newton: a smooth cost on the affine set A C = b, with
 * the Hessian measured from coloured gradient differences and factored per problem in band form.
 *
 * Structure (host, once per setup).  With B-splines a breakpoint touches only the coefficients
 * offset[j][bp] .. offset[j][bp] + order_j - 1 of output j, so the cost couples exactly the coefficients that
 * share a breakpoint of the outputs in its active-variable lists (the initial cost at the first breakpoint, the
 * final cost at the last).  The equality rows are local too.  Ordering the columns by the first breakpoint that
 * touches them (ties by output, then by index) interleaves the outputs in time and makes the pattern of
 * H + A'A a band of half-bandwidth w that does not grow with the horizon.  A greedy distance-2 colouring of the
 * H pattern in that order (no two columns of one colour share a row) lets one difference of gradients
 * recover every column of its colour: K colours cost 2K gradient evaluations (central differences).
 *
 * Per problem and iteration:
 *   band       H from the differences, symmetrised: H_ij = (dg_col(j)[i] / 2h_j + dg_col(i)[j] / 2h_i) / 2
 *   matrix     M = H + rho A'A + tau I, rho = max diag H / max diag A'A (A'A is singular where H is not
 *              and the other way round on the lane change: linear trajectories cost nothing), tau the
 *              Levenberg-Marquardt shift carried per problem
 *   factor     banded Cholesky streaming a (w+1) x (w+1) window: O(nC w^2), nothing of size nC x nC.  On a
 *              nonpositive pivot tau = max(4 tau, beta), beta = 1e-3 max diag(H + rho A'A), and again, up to
 *              kMaxShift times; then the direction is -P g
 *   step       range-space: Y = M^-1 [g, Q1'], S = Q1 M^-1 Q1' (r x r, dense Cholesky), S lam = -Q1 M^-1 g,
 *              d = -M^-1 (g + Q1' lam), so that Q1 d = 0.  Q1 [r][nC] is the orthonormal basis of the rows'
 *              span (the same Q1 as ntg_lbfgs.h), so dependent rows cannot make S singular.
 *
 * The code is plain C++ over sqp::Coop, as ntg_lbfgs.h: k_newton_factor and k_newton_dir (ntg_core.cu) run it
 * with one CTA per problem, tests/tools/newton_host.cpp compiles THE SAME TEXT with g++ for a group of one
 * thread.  No reduction here depends on the number of threads: maxima only, and every dot product and
 * triangular solve is walked by one thread in a fixed order.
 */
#ifndef NTG_NEWTON_H_
#define NTG_NEWTON_H_

#include <math.h>

#include "ntg_sqp.cuh"

#include <algorithm>
#include <vector>

namespace ntgb {
namespace newton {

constexpr int kMaxRows = 128;     /* rank of the equality rows, at most: S is r x r per problem */
constexpr int kMaxHalfBand = 64;  /* half-bandwidth, at most: the factor's window is (w+1)^2 doubles of shared memory */
constexpr int kMaxShift = 8;      /* shifted refactorizations per iteration before falling back to -P g */
constexpr int kMaxStall = 2;      /* consecutive iterations without a strict decrease that end a solve (status 2) */
constexpr double kBetaRel = 1e-3; /* beta = kBetaRel max diag (H + rho A'A) */

/* what the host derives once per setup */
struct Structure {
    int nC = 0, w = 0, K = 0;
    std::vector<int> perm;            /* [nC] column at permuted position i */
    std::vector<int> color;           /* [nC] colour of column c (original order) */
    std::vector<unsigned char> hmask; /* [nC][w+1] 1: (perm[i], perm[i-d]) is in the pattern of H */
    std::vector<double> ata;          /* [nC][w+1] (A'A)(perm[i], perm[i-d]) */
};

/* cost_out[0 / 1 / 2]: bit j set when output j is in the initial / trajectory / final cost's active-variable
 * list.  off [nout][nbps] the K0 offsets (ntgb_create checks that every window lies inside its output).
 * A [m][nC] row-major: the equality rows. */
inline void build_structure(int nout, int nbps, const int *order, const int *ncoef, const int *off, const unsigned *cost_out,
                           const double *A, int m, Structure &S)
{
    std::vector<int> iC(nout + 1, 0);
    for (int j = 0; j < nout; j++) iC[j + 1] = iC[j] + ncoef[j];
    const int nC = iC[nout];
    S = Structure();
    S.nC = nC;
    std::vector<std::vector<int>> adj((size_t)nC); /* pattern of H, column by column, original order */
    std::vector<int> clique;
    auto add_clique = [&](const std::vector<int> &q) {
        for (int a : q)
            for (int b : q) adj[a].push_back(b);
    };
    for (int bp = 0; bp < nbps; bp++) {
        clique.clear();
        for (int j = 0; j < nout; j++) {
            const bool hit = (cost_out[1] >> j & 1u) || (bp == 0 && (cost_out[0] >> j & 1u)) ||
                             (bp == nbps - 1 && (cost_out[2] >> j & 1u));
            if (!hit) continue;
            for (int k = 0; k < order[j]; k++) clique.push_back(iC[j] + off[(size_t)j * nbps + bp] + k);
        }
        add_clique(clique);
    }
    for (int c = 0; c < nC; c++) {
        adj[c].push_back(c); /* the diagonal is always measured */
        std::sort(adj[c].begin(), adj[c].end());
        adj[c].erase(std::unique(adj[c].begin(), adj[c].end()), adj[c].end());
    }
    /* order: first breakpoint touching the column, then output, then index */
    std::vector<long long> key(nC);
    for (int j = 0; j < nout; j++)
        for (int l = 0; l < ncoef[j]; l++) {
            int first = nbps;
            for (int bp = 0; bp < nbps; bp++) {
                const int o = off[(size_t)j * nbps + bp];
                if (o <= l && l < o + order[j]) { first = bp; break; }
            }
            key[iC[j] + l] = ((long long)first * nout + j) * nC + l;
        }
    S.perm.resize(nC);
    for (int c = 0; c < nC; c++) S.perm[c] = c;
    std::sort(S.perm.begin(), S.perm.end(), [&](int a, int b) { return key[a] < key[b]; });
    std::vector<int> pos(nC);
    for (int i = 0; i < nC; i++) pos[S.perm[i]] = i;
    /* rows of A: their nonzero columns */
    std::vector<std::vector<int>> rows((size_t)m);
    for (int r = 0; r < m; r++)
        for (int c = 0; c < nC; c++)
            if (A[(size_t)r * nC + c] != 0.0) rows[r].push_back(c);
    int w = 0;
    for (int c = 0; c < nC; c++)
        for (int i : adj[c]) w = std::max(w, std::abs(pos[i] - pos[c]));
    for (const auto &q : rows)
        for (int a : q)
            for (int b : q) w = std::max(w, std::abs(pos[a] - pos[b]));
    S.w = w;
    const int W = w + 1;
    /* greedy distance-2 colouring in permuted order */
    S.color.assign(nC, -1);
    std::vector<int> seen;
    for (int i = 0; i < nC; i++) {
        const int c = S.perm[i];
        seen.assign((size_t)S.K + 1, 0);
        for (int row : adj[c])
            for (int c2 : adj[row])
                if (S.color[c2] >= 0) seen[S.color[c2]] = 1;
        int k = 0;
        while (seen[k]) k++;
        S.color[c] = k;
        S.K = std::max(S.K, k + 1);
    }
    S.hmask.assign((size_t)nC * W, 0);
    for (int c = 0; c < nC; c++)
        for (int i : adj[c])
            if (pos[i] >= pos[c]) S.hmask[(size_t)pos[i] * W + (pos[i] - pos[c])] = 1;
    S.ata.assign((size_t)nC * W, 0.0);
    for (int r = 0; r < m; r++)
        for (int a : rows[r])
            for (int b : rows[r])
                if (pos[a] >= pos[b]) S.ata[(size_t)pos[a] * W + (pos[a] - pos[b])] += A[(size_t)r * nC + a] * A[(size_t)r * nC + b];
}

/* the difference step of column c at C_c (central differences: eps^(1/3) scaled) */
NTG_HD inline double fd_step(double c)
{
    const double a = fabs(c);
    return 6.0554544523933395e-06 * (a > 1.0 ? a : 1.0); /* cbrt(DBL_EPSILON) */
}

/* shared setup data of one solve */
struct Desc {
    const int *perm, *color;          /* [nC] */
    const unsigned char *hmask;       /* [nC][w+1] */
    const double *ata;                /* [nC][w+1] */
    const double *Q1;                 /* [r][nC] */
    int nC, w, K, r;
    double ata_max;                   /* max diag A'A, 0 without rows */
};

/* band [nC][w+1] <- H + rho A'A + tau I in permuted order from G [2K][nC] (point 2k: C + h on colour k,
 * 2k + 1: C - h).  Returns the largest diagonal of H + rho A'A through hmax (0 when none is positive). */
template <class Co>
NTG_HD void assemble(const Co &cg, double *red, const Desc &D, const double *C, const double *G, double tau, double *band,
                     double &dmax)
{
    const int n = D.nC, W = D.w + 1;
    const size_t nn = (size_t)n;
    for (int q = cg.tid; q < n * W; q += cg.nt) {
        const int i = q / W, d = q - i * W;
        double v = 0.0;
        if (d <= i && D.hmask[q]) {
            const int ci = D.perm[i], cj = D.perm[i - d];
            const double xi = C[ci], xj = C[cj], hi = fd_step(xi), hj = fd_step(xj);
            const double *Gj = G + (size_t)2 * D.color[cj] * nn, *Gi = G + (size_t)2 * D.color[ci] * nn;
            const double vj = (Gj[ci] - Gj[nn + ci]) / ((xj + hj) - (xj - hj));
            const double vi = (Gi[cj] - Gi[nn + cj]) / ((xi + hi) - (xi - hi));
            v = 0.5 * (vj + vi);
        }
        band[q] = v;
    }
    cg.sync();
    double hm = 0.0;
    for (int i = cg.tid; i < n; i += cg.nt) hm = fmax(hm, band[(size_t)i * W]);
    hm = cg.template reduce<true>(hm, red);
    const double rho = D.ata_max > 0.0 && hm > 0.0 ? hm / D.ata_max : (D.ata_max > 0.0 ? 1.0 : 0.0);
    double mm = 0.0;
    for (int q = cg.tid; q < n * W; q += cg.nt) {
        double v = band[q] + rho * D.ata[q];
        if (q % W == 0) {
            mm = fmax(mm, v);
            v += tau;
        }
        band[q] = v;
    }
    dmax = cg.template reduce<true>(mm, red);
    cg.sync();
}

/* in-place Cholesky of the band [n][w+1] (row i: entries (i, i-d), d = 0..w; entries before column 0 are
 * ignored), streaming a window win [(w+1)][(w+1)] of the rows j .. j+w.  Returns false at a pivot that is not
 * positive (band is then partly overwritten). */
template <class Co>
NTG_HD bool band_cholesky(const Co &cg, int n, int w, double *band, double *win)
{
    const int W = w + 1;
    for (int q = cg.tid; q < W * W; q += cg.nt) {
        const int i = q / W;
        win[q] = i < n ? band[q] : 0.0;
    }
    for (int j = 0; j < n; j++) {
        cg.sync();
        const int sj = j % W;
        const double piv = win[sj * W];
        if (!(piv > 0.0)) return false;
        const double l = sqrt(piv);
        const int hi = j + w < n - 1 ? j + w : n - 1;
        cg.sync();
        for (int i = j + 1 + cg.tid; i <= hi; i += cg.nt) win[(i % W) * W + (i - j)] /= l;
        if (cg.tid == 0) win[sj * W] = l;
        cg.sync();
        /* trailing update of the window: (i, k), j < k <= i <= hi */
        const int m = hi - j;
        for (int q = cg.tid; q < m * m; q += cg.nt) {
            const int a = q / m, b = q - a * m;
            if (b > a) continue;
            const int i = j + 1 + a, k = j + 1 + b;
            win[(i % W) * W + (i - k)] -= win[(i % W) * W + (i - j)] * win[(k % W) * W + (k - j)];
        }
        cg.sync();
        /* row j is final: out to the band; row j + W in */
        for (int d = cg.tid; d < W; d += cg.nt) {
            band[(size_t)j * W + d] = win[sj * W + d];
            win[sj * W + d] = j + W < n ? band[(size_t)(j + W) * W + d] : 0.0;
        }
    }
    cg.sync();
    return true;
}

/* x <- M^-1 x for the factor L [n][w+1] (L L' = M, permuted order); x in ORIGINAL order, perm maps.  One
 * thread walks it. */
NTG_HD inline void band_solve(int n, int w, const double *L, const int *perm, double *x)
{
    const int W = w + 1;
    for (int i = 0; i < n; i++) {
        const double *Li = L + (size_t)i * W;
        double a = x[perm[i]];
        const int dm = i < w ? i : w;
        for (int d = 1; d <= dm; d++) a -= Li[d] * x[perm[i - d]];
        x[perm[i]] = a / Li[0];
    }
    for (int i = n - 1; i >= 0; i--) {
        double a = x[perm[i]];
        const int dm = n - 1 - i < w ? n - 1 - i : w;
        for (int d = 1; d <= dm; d++) a -= L[(size_t)(i + d) * W + d] * x[perm[i + d]];
        x[perm[i]] = a / L[(size_t)i * W];
    }
}

/* the range-space step with the factor L of M: Y [r+1][n] (row 0 = M^-1 g, row 1 + k = M^-1 Q1[k]), S [r][r],
 * lam [r]; d = -M^-1 (g + Q1' lam).  Returns false when S is not positive definite. */
template <class Co>
NTG_HD bool range_step(const Co &cg, const Desc &D, const double *L, const double *g, double *Y, double *S, double *lam,
                       double *d)
{
    const int n = D.nC, r = D.r;
    for (int k = cg.tid; k <= r; k += cg.nt) {
        double *y = Y + (size_t)k * n;
        const double *src = k == 0 ? g : D.Q1 + (size_t)(k - 1) * n;
        for (int e = 0; e < n; e++) y[e] = src[e];
        band_solve(n, D.w, L, D.perm, y);
    }
    cg.sync();
    /* S = Q1 Y[1..r]' and the right-hand side -Q1 Y[0] in lam */
    for (int q = cg.tid; q < r * (r + 1); q += cg.nt) {
        const int k = q / (r + 1), l = q - k * (r + 1);
        const double *a = D.Q1 + (size_t)k * n, *y = Y + (size_t)l * n;
        double s = 0.0;
        for (int e = 0; e < n; e++) s += a[e] * y[e];
        if (l == 0)
            lam[k] = -s;
        else
            S[(size_t)k * r + (l - 1)] = s;
    }
    cg.sync();
    /* symmetrise, dense Cholesky in place (lower), one column at a time */
    for (int q = cg.tid; q < r * r; q += cg.nt) {
        const int k = q / r, l = q - k * r;
        if (l < k) S[q] = 0.5 * (S[q] + S[(size_t)l * r + k]);
    }
    for (int j = 0; j < r; j++) {
        cg.sync();
        const double piv = S[(size_t)j * r + j];
        if (!(piv > 0.0)) return false;
        const double l = sqrt(piv);
        cg.sync();
        for (int i = j + 1 + cg.tid; i < r; i += cg.nt) S[(size_t)i * r + j] /= l;
        if (cg.tid == 0) S[(size_t)j * r + j] = l;
        cg.sync();
        const int m = r - 1 - j;
        for (int q = cg.tid; q < m * m; q += cg.nt) {
            const int a = q / m, b = q - a * m;
            if (b > a) continue;
            const int i = j + 1 + a, k = j + 1 + b;
            S[(size_t)i * r + k] -= S[(size_t)i * r + j] * S[(size_t)k * r + j];
        }
    }
    cg.sync();
    if (cg.tid == 0) {
        for (int i = 0; i < r; i++) {
            double a = lam[i];
            for (int k = 0; k < i; k++) a -= S[(size_t)i * r + k] * lam[k];
            lam[i] = a / S[(size_t)i * r + i];
        }
        for (int i = r - 1; i >= 0; i--) {
            double a = lam[i];
            for (int k = i + 1; k < r; k++) a -= S[(size_t)k * r + i] * lam[k];
            lam[i] = a / S[(size_t)i * r + i];
        }
    }
    cg.sync();
    /* d = -(Y0 + sum_k lam_k Y_k) */
    for (int e = cg.tid; e < n; e += cg.nt) {
        double a = Y[e];
        for (int k = 0; k < r; k++) a += lam[k] * Y[(size_t)(k + 1) * n + e];
        d[e] = -a;
    }
    cg.sync();
    return true;
}

/* one problem's carried scalars */
struct State {
    double tau, beta; /* the shift, and beta of the last factorization */
    int stall;        /* consecutive iterations without a strict decrease */
};

/* the shift and stopping rule after the search.  armijo: the search found a step a with sufficient decrease
 * (with the rounding allowance); fnew its cost, f0 the cost at the start.  Returns true when the step is taken.
 * Sets *done = 2 after kMaxStall consecutive iterations without fnew < f0: the cost no longer resolves a
 * decrease (the rounding floor), so raising tau further would only shorten steps that cannot help. */
NTG_HD inline bool after_search(State &s, bool armijo, double a, double fnew, double f0, int *done)
{
    if (armijo) {
        if (a == 1.0)
            s.tau *= 0.25;
        else if (a < 0.25)
            s.tau = fmax(4.0 * s.tau, s.beta);
        s.stall = fnew < f0 ? 0 : s.stall + 1;
    } else {
        s.tau = fmax(4.0 * s.tau, s.beta);
        s.stall++;
    }
    *done = s.stall >= kMaxStall ? 2 : 0;
    return armijo;
}

} /* namespace newton */
} /* namespace ntgb */

#endif
