/*
 * ntg_warm.h -- one problem's row of SQP warm-start state (ntgb_solve_sqp_warm) as plain host/device
 * code: the layout of a row, the digest that ties a row to the setup's reduced space, and the rules
 * that decide what a solve starts from.
 *
 *   row [0]            format tag kWarmTag
 *       [1] [2]        nr, m: reduced variables and general rows of the setup
 *       [3] [4]        digest of the reduction, low and high 32 bits (exact integers in doubles, so a
 *                      row survives any copy that keeps its values)
 *       [5]            nu, the weight of the L1 merit function
 *       [6 ..]         B [nr][nr], the quasi-Newton Hessian of the reduced Lagrangian, row-major
 *
 * A row is used only when its tag, nr, m and digest all equal the setup's; every other row (all zeros,
 * another setup's, garbage) is a cold start: B = I, nu = 0, exactly what ntgb_solve_sqp starts from.
 * From a matching row nu is taken as 0 unless it is finite and >= 0, and B is read from its lower
 * triangle and mirrored, so the solver always starts from a symmetric matrix; one that is not positive
 * definite (or holds a NaN) is replaced by I by the Cholesky test of ntg_sqp.cuh's sqp_step.
 *
 * k_sqp_init (ntg_core.cu) reads rows with one thread per problem (warm_load), k_sqp_warm_store writes
 * them with one warp per problem (warm_encode, start = lane, step = 32); the CPU test suite compiles
 * THE SAME TEXT with g++ (tests/test_warm_host.py, tests/tools/warm_host.cpp).
 */
#ifndef NTG_WARM_H_
#define NTG_WARM_H_

#include <stddef.h>
#include <stdint.h>

#ifndef NTG_HD
#if defined(__CUDACC__)
#define NTG_HD __host__ __device__
#else
#define NTG_HD
#endif
#endif

namespace ntgb {

constexpr double kWarmTag = 1314150193.0; /* 0x4E545731, "NTW1" */
constexpr int kWarmNu = 5;                 /* position of nu; the header is [0, kWarmNu) */
constexpr int kWarmB = 6;                  /* position of B[0][0] */

/* what a row must carry to be used with this setup */
struct WarmKey {
    int nr, m;
    uint64_t digest;
};

/* doubles in one row */
NTG_HD inline size_t warm_doubles(int nr) { return (size_t)kWarmB + (size_t)nr * (size_t)nr; }

/* FNV-1a (64 bit) over the bytes of nC, nr, m, n_li (int32 each), li_idx[n_li] (int32) and N [nr][nC]
 * (doubles): the reduced space C = Cpart + N y and the general rows that y's Hessian belongs to.
 * Host only; the host QR that builds N is deterministic, so identical setups get identical digests. */
inline uint64_t warm_digest(int nC, int nr, int m, int n_li, const int *li_idx, const double *N)
{
    uint64_t h = 14695981039346656037ull;
    auto eat = [&h](const void *p, size_t n) {
        const unsigned char *b = static_cast<const unsigned char *>(p);
        for (size_t i = 0; i < n; i++) {
            h ^= b[i];
            h *= 1099511628211ull;
        }
    };
    const int32_t head[4] = {nC, nr, m, n_li};
    eat(head, sizeof head);
    for (int i = 0; i < n_li; i++) {
        const int32_t v = li_idx[i];
        eat(&v, sizeof v);
    }
    eat(N, sizeof(double) * (size_t)nr * (size_t)nC);
    return h;
}

/* does this row belong to this setup? (a NaN anywhere in the header compares unequal: no) */
NTG_HD inline bool warm_match(const double *row, const WarmKey &k)
{
    return row[0] == kWarmTag && row[1] == (double)k.nr && row[2] == (double)k.m &&
           row[3] == (double)(k.digest & 0xffffffffull) && row[4] == (double)(k.digest >> 32);
}

/* nu of a matching row: NaN, infinite or negative -> 0 */
NTG_HD inline double warm_nu(const double *row)
{
    const double v = row[kWarmNu];
    return (v >= 0.0 && v <= 1.7976931348623157e308) ? v : 0.0;
}

/* B[i][j] of a matching row, from its lower triangle */
NTG_HD inline double warm_b(const double *row, int nr, int i, int j)
{
    return i >= j ? row[kWarmB + (size_t)i * nr + j] : row[kWarmB + (size_t)j * nr + i];
}

/* one problem's starting B [nr][nr] and nu: from the row if it matches (row may be nullptr), else B = I and
 * nu = 0; returns whether it matched */
NTG_HD inline bool warm_load(const double *row, const WarmKey &k, double *B, double *nu)
{
    const int nr = k.nr;
    const bool hot = row != nullptr && warm_match(row, k);
    for (int e = 0; e < nr * nr; e++) B[e] = hot ? warm_b(row, nr, e / nr, e % nr) : (e / nr == e % nr) ? 1.0 : 0.0;
    *nu = hot ? warm_nu(row) : 0.0;
    return hot;
}

/* write entries start, start + step, ... of a row: header, nu and B [nr][nr] (row-major) */
NTG_HD inline void warm_encode(double *row, const WarmKey &k, double nu, const double *B, int start, int step)
{
    const size_t n = warm_doubles(k.nr);
    for (size_t e = (size_t)start; e < n; e += (size_t)step) {
        double v;
        switch ((int)(e < (size_t)kWarmB ? e : (size_t)kWarmB)) {
        case 0: v = kWarmTag; break;
        case 1: v = (double)k.nr; break;
        case 2: v = (double)k.m; break;
        case 3: v = (double)(k.digest & 0xffffffffull); break;
        case 4: v = (double)(k.digest >> 32); break;
        case kWarmNu: v = nu; break;
        default: v = B[e - kWarmB]; break;
        }
        row[e] = v;
    }
}

} /* namespace ntgb */

#endif /* NTG_WARM_H_ */
