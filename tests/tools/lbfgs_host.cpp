/* tests/tools/lbfgs_host.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 * The per-problem core of ntgb_solve_eq_lbfgs (ntg_b200/csrc/ntg_lbfgs.h) compiled with g++ for a group of one
 * thread, so that tests/test_lbfgs_host.py can check it against tests/tools/lbfgs_reference.py without a GPU:
 * the same text k_lbfgs_dir, k_lbfgs_update and k_lbfgs_init run.  st = {head, npair, pend}. */
#include "ntg_lbfgs.h"

namespace {

const ntgb::sqp::Coop kOne{0, 1, 0, 1};

ntgb::lbfgs::View view(const double *Q1, int r, int n, int mem, double *ring, double *rho, double *sv, double *gp)
{
    return ntgb::lbfgs::View{Q1, r, n, mem, ring, rho, sv, gp};
}

}  // namespace

extern "C" {

void lbfgs_host_project(const double *Q1, int r, int n, double *v) { ntgb::lbfgs::project(kOne, nullptr, Q1, r, n, v); }

int lbfgs_host_direction(const double *Q1, int r, int n, int mem, double *ring, double *rho, double *sv, double *gp,
                         int *st, double *gamma, double f, const double *g, double gtol, double *d, double *dg)
{
    ntgb::lbfgs::State s{st[0], st[1], st[2], *gamma};
    const int rc = ntgb::lbfgs::direction(kOne, nullptr, view(Q1, r, n, mem, ring, rho, sv, gp), s, f, g, gtol, d, *dg);
    st[0] = s.head;
    st[1] = s.npair;
    st[2] = s.pend;
    *gamma = s.gamma;
    return rc;
}

int lbfgs_host_accept(const double *Q1, int r, int n, int mem, double *ring, double *rho, double *sv, double *gp, int *st,
                      double *gamma, const double *Cpart, double *C, const double *d, double a, double phi0, double phi_best)
{
    ntgb::lbfgs::State s{st[0], st[1], st[2], *gamma};
    const int rc = ntgb::lbfgs::accept(kOne, nullptr, view(Q1, r, n, mem, ring, rho, sv, gp), s, Cpart, C, d, a, phi0,
                                       phi_best);
    st[0] = s.head;
    st[1] = s.npair;
    st[2] = s.pend;
    *gamma = s.gamma;
    return rc;
}
}
