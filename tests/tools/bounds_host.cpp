// Test infrastructure: the per-problem bounds logic of ntgb_solve_*_bounds (ntg_b200/csrc/ntg_bounds.h)
// compiled for the host, run the way k_bounds_prep runs it but with one thread (start 0, step 1).
// stdin (whitespace separated; doubles in any strtod form, e.g. Python's float.hex()):
//   nlic nltc nlfc nnlic nnltc nnlfc nbps nC
//   n_li li[n_li]      linear rows kept as general rows
//   me eq[me]          eliminated linear rows
//   M[nC*me]           Cpart = M be, row-major
//   Ae[me*nC]          eliminated rows, row-major
//   P, then per problem lo[nb] up[nb]
// stdout, one line per problem, doubles as %a:
//   bad hl[m] hu[m] be[me] Cpart[nC]
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "ntg_bounds.h"

static double rd()
{
    char buf[128];
    if (std::scanf("%127s", buf) != 1) std::exit(2);
    return std::strtod(buf, nullptr);
}

static int ri()
{
    int v;
    if (std::scanf("%d", &v) != 1) std::exit(2);
    return v;
}

int main()
{
    ntgb::BoundsLayout L;
    L.nlic = ri(); L.nltc = ri(); L.nlfc = ri(); L.nnlic = ri(); L.nnltc = ri(); L.nnlfc = ri(); L.nbps = ri();
    const int nC = ri();
    const int n_li = ri();
    std::vector<int> li(n_li + 1);
    for (int i = 0; i < n_li; i++) li[i] = ri();
    const int me = ri();
    std::vector<int> eq(me + 1);
    for (int i = 0; i < me; i++) eq[i] = ri();
    std::vector<double> M((size_t)nC * me + 1), Ae((size_t)me * nC + 1);
    for (size_t i = 0; i < (size_t)nC * me; i++) M[i] = rd();
    for (size_t i = 0; i < (size_t)me * nC; i++) Ae[i] = rd();
    const int P = ri(), nb = L.nb(), m = n_li + L.ncnln();
    std::vector<double> lo(nb + 1), up(nb + 1), hl(m + 1), hu(m + 1), be(me + 1), Cp(nC + 1);
    for (int p = 0; p < P; p++) {
        for (int k = 0; k < nb; k++) lo[k] = rd();
        for (int k = 0; k < nb; k++) up[k] = rd();
        unsigned bad = ntgb::bounds_expand(L, lo.data(), up.data(), li.data(), n_li, eq.data(), me, hl.data(), hu.data(),
                                           be.data(), 0, 1);
        for (int e = 0; e < nC; e++) Cp[e] = ntgb::bounds_cpart(M.data(), me, be.data(), e);
        double res = 0.0, bmax = 0.0;
        for (int r = 0; r < me; r++) {
            res = ntgb::bounds_max(res, std::fabs(ntgb::bounds_residual(Ae.data() + (size_t)r * nC, nC, Cp.data(), be[r])));
            bmax = std::fmax(bmax, std::fabs(be[r]));
        }
        if (ntgb::bounds_inconsistent(res, bmax)) bad |= ntgb::kBoundsInconsistent;
        std::printf("%u", bad);
        for (int i = 0; i < m; i++) std::printf(" %a", hl[i]);
        for (int i = 0; i < m; i++) std::printf(" %a", hu[i]);
        for (int r = 0; r < me; r++) std::printf(" %a", be[r]);
        for (int e = 0; e < nC; e++) std::printf(" %a", Cp[e]);
        std::printf("\n");
    }
    return 0;
}
