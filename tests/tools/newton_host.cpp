/* tests/tools/newton_host.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 * The host structure and the per-problem algebra of ntgb_solve_eq_newton (ntg_b200/csrc/ntg_newton.h) compiled
 * with g++ for a group of one thread, so that tests/test_newton_host.py can check them without a GPU: the same
 * text k_newton_factor and k_newton_dir run. */
#include <cstring>

#include "ntg_newton.h"

namespace {

const ntgb::sqp::Coop kOne{0, 1, 0, 1};
ntgb::newton::Structure g_s;

}  // namespace

extern "C" {

/* -> 0; K, w; then newton_host_fetch copies perm, color, hmask, ata */
int newton_host_structure(int nout, int nbps, const int *order, const int *ncoef, const int *off, const unsigned *cost_out,
                          const double *A, int m, int *K, int *w)
{
    ntgb::newton::build_structure(nout, nbps, order, ncoef, off, cost_out, A, m, g_s);
    *K = g_s.K;
    *w = g_s.w;
    return 0;
}

void newton_host_fetch(int *perm, int *color, unsigned char *hmask, double *ata)
{
    std::memcpy(perm, g_s.perm.data(), sizeof(int) * g_s.perm.size());
    std::memcpy(color, g_s.color.data(), sizeof(int) * g_s.color.size());
    std::memcpy(hmask, g_s.hmask.data(), g_s.hmask.size());
    std::memcpy(ata, g_s.ata.data(), sizeof(double) * g_s.ata.size());
}

double newton_host_step_of(double c) { return ntgb::newton::fd_step(c); }

/* band <- H + rho A'A + tau I; returns max diag (H + rho A'A) */
double newton_host_assemble(int n, int w, int K, int r, const int *perm, const int *color, const unsigned char *hmask,
                            const double *ata, double ata_max, const double *C, const double *G, double tau, double *band)
{
    const ntgb::newton::Desc D{perm, color, hmask, ata, nullptr, n, w, K, r, ata_max};
    double dmax = 0.0;
    ntgb::newton::assemble(kOne, nullptr, D, C, G, tau, band, dmax);
    return dmax;
}

int newton_host_factor(int n, int w, double *band)
{
    std::vector<double> win((size_t)(w + 1) * (w + 1));
    return ntgb::newton::band_cholesky(kOne, n, w, band, win.data()) ? 1 : 0;
}

void newton_host_solve(int n, int w, const double *L, const int *perm, double *x)
{
    ntgb::newton::band_solve(n, w, L, perm, x);
}

int newton_host_range_step(int n, int w, int r, const int *perm, const double *Q1, const double *L, const double *g,
                           double *d)
{
    const ntgb::newton::Desc D{perm, nullptr, nullptr, nullptr, Q1, n, w, 0, r, 0.0};
    std::vector<double> Y((size_t)(r + 1) * n), S((size_t)r * r + 1), lam((size_t)r + 1);
    return ntgb::newton::range_step(kOne, D, L, g, Y.data(), S.data(), lam.data(), d) ? 1 : 0;
}

/* st = {tau, beta, stall}; returns done */
int newton_host_after_search(double *st, int armijo, double a, double fnew, double f0)
{
    ntgb::newton::State s{st[0], st[1], (int)st[2]};
    int done = 0;
    ntgb::newton::after_search(s, armijo != 0, a, fnew, f0, &done);
    st[0] = s.tau;
    st[1] = s.beta;
    st[2] = s.stall;
    return done;
}
}
