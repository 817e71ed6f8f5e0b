/* tests/tools/warm_host.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 * The SQP warm-start row of ntgb_solve_sqp_warm (ntg_b200/csrc/ntg_warm.h) compiled with g++, so that
 * tests/test_warm_host.py can check its layout and its match / clamp rules without a GPU: the same text
 * k_sqp_init and k_sqp_warm_store run, k_sqp_warm_store's warp split replaced by start / step. */
#include "ntg_warm.h"

extern "C" {

size_t warm_host_doubles(int nr) { return ntgb::warm_doubles(nr); }

uint64_t warm_host_digest(int nC, int nr, int m, int n_li, const int *li_idx, const double *N)
{
    return ntgb::warm_digest(nC, nr, m, n_li, li_idx, N);
}

void warm_host_encode(double *row, int nr, int m, uint64_t digest, double nu, const double *B, int start, int step)
{
    ntgb::warm_encode(row, ntgb::WarmKey{nr, m, digest}, nu, B, start, step);
}

/* k_sqp_init's start of one problem: 1 and B [nr][nr], nu from a matching row, else 0, B = I, nu = 0 */
int warm_host_load(const double *row, int nr, int m, uint64_t digest, double *B, double *nu)
{
    return ntgb::warm_load(row, ntgb::WarmKey{nr, m, digest}, B, nu) ? 1 : 0;
}
}
