/*
 * ntg_core.cu -- core of libntg_b200.so: the C ABI of include/ntg_b200.h.
 *
 *   - pack registry (callback host address -> instantiated device evaluator)
 *   - K0: one-time device build of the collocation tables (replaces
 *     ConcatCollocMatrix / CollocMatrix + PGS, reference src/colloc.c:15-117)
 *   - problem handles, batched evaluation entry points (device and host
 *     buffers), table / pattern / bounds getters
 *   - "next" rows of SURVEY.md section 8(f): linear-constraint matrix and batched
 *     A*C (src/constraints.c:198-261), bound expansion (src/constraints.c:5-33),
 *     batched SplineInterp (src/colloc.c:449-484)
 *
 * Built with -fmad=false: every table and linear-constraint entry is plain
 * IEEE double evaluated in the reference's order.
 * There is no CPU evaluation path in this library.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "ntg_b200.h"
#include "ntg_kernel_args.h"
#include "pgs_device.cuh"
#include "ntg_sqp.cuh"
#include "ntg_bounds.h"
#include "ntg_warm.h"
#include "ntg_lbfgs.h"
#include "ntg_newton.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t e_ = (expr);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return fail(NTGB_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                 \
    } while (0)

std::mutex g_reg_mu;
std::vector<ntgb_pack> &registry()
{
    static std::vector<ntgb_pack> r;
    return r;
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

/* device scratch of one solver, sized and carved by scratch_carve */
struct Scratch {
    void *p = nullptr;
    size_t bytes = 0;
};

/* work space of one stream-ordered solver entry point (ntgb_solve_*_async), sized by its reserve call for up to
 * P problems */
struct AsyncWork {
    Scratch s;
    int P = 0;
};

} /* namespace */

struct ntgb_problem {
    int device = 0;
    ntgb_dims dims{};
    ntgb_devtab tab{};
    const ntgb_pack *pack = nullptr;
    ntgb_pack pack_copy{};
    int sm_count = 0, max_smem_optin = 0;
    /* host copies of the setup */
    std::vector<int> order, mult, maxderiv, ninterv, ncoef;
    std::vector<std::vector<double>> knots, augknots;
    std::vector<double> bps;
    int nlic = 0, nltc = 0, nlfc = 0, nnlic = 0, nnltc = 0, nnlfc = 0;
    std::vector<double> lic, ltc, lfc; /* row-major [n][nz] */
    std::vector<double> lowerb, upperb;
    /* host copies of K0 output */
    std::vector<double> hB;            /* reference block layout, outputs concatenated */
    std::vector<size_t> hB_off;        /* start of output j in hB */
    std::vector<int> hoff, hleft;      /* [nout][nbps] */
    std::vector<int> col0;             /* [ncnln][nout] */
    std::vector<double> A;             /* nclin x nC column-major */
    /* device-side linear constraints in band form */
    double *dAband = nullptr;          /* [nclin][S] */
    int *dAcol0 = nullptr;             /* [nclin][nout] */
    double *dlin_lb = nullptr, *dlin_ub = nullptr; /* [nclin] expanded */
    /* spline-interp device description */
    double *daug[NTGB_MAXOUT] = {nullptr};
    double *dknots[NTGB_MAXOUT] = {nullptr};
    std::vector<void *> allocs;
    /* scratch for ntgb_eval_host: two device buffer sets of `cap` problems each, one stream each,
     * so chunk k+1's H2D/compute overlaps chunk k's D2H */
    struct HostScratch {
        int cap = 0, jac_layout = -1;
        bool hasZ = false;
        double *C = nullptr, *f = nullptr, *g = nullptr, *c = nullptr, *J = nullptr, *Z = nullptr,
               *result = nullptr;
        size_t Jbytes = 0;
        cudaStream_t stream = nullptr;
    } hs[2];
    int *d_abort = nullptr; /* device flag: a callback wrote *mode = -1 */
    /* small calls of ntgb_eval_host (an NPSOL callback is P = 1): one page-locked, device-mapped
     * staging block that the kernel reads its coefficients from and writes its results to -- a
     * launch and a synchronize instead of eight copies */
    struct {
        char *buf = nullptr;
        size_t bytes = 0;
        size_t j_off = 0, j_bytes = 0; /* region of the last Jacobian written and its layout */
        int j_layout = NTGB_JAC_NONE;
        size_t lastP = 0;
    } zc;
    std::vector<double> lin_lb, lin_ub; /* expanded linear bounds, [nclin] */
    /* reduced form of the solvers: equality rows eliminated (C = Cpart + N y), the other linear rows
     * kept as general constraints next to the nonlinear ones */
    struct {
        bool ready = false;
        int nr = 0, n_li = 0, m = 0;
        double *N = nullptr, *Cpart = nullptr; /* N [nr][nC] (basis vector k contiguous), Cpart [nC] */
        int r = 0;                  /* rank of the eliminated rows, nC - nr */
        double *Q1 = nullptr;       /* [r][nC] orthonormal rows spanning the eliminated rows (ntgb_solve_eq_lbfgs) */
        double *M = nullptr, *Ae = nullptr; /* Cpart = M be, M [nC][me]; eliminated rows Ae [me][nC] */
        int *li_idx = nullptr;      /* [n_li] linear row of general constraint i */
        double *hl = nullptr, *hu = nullptr; /* [m] bounds: linear inequality rows, then the nonlinear rows */
        double *A = nullptr;        /* dense nclin x nC, column-major (for A_in^T mu) */
        std::vector<double> hN;     /* host copy of N */
        std::vector<int> eq, li;    /* linear rows: eliminated equalities / kept as general constraints */
        uint64_t digest = 0;        /* ntg_warm.h warm_digest of this reduced form: SQP warm-start rows match it */
    } alm;
    /* ntgb_solve_sqp: on top of alm's reduced form */
    struct {
        bool ready = false;
        double *ArN = nullptr; /* [n_li][nr] */
        double *W = nullptr;   /* [me][nC] (Ae Ae')^-1 Ae */
        int *eq_idx = nullptr; /* [me] */
        int me = 0;
    } sqp;
    /* per-call device arrays, kept between calls: one scratch per driver, so that no call's arrays alias
     * another solver's (ntgb_solve_eq, ntgb_solve_nlp, ntgb_solve_sqp, ntgb_linesearch, per-problem bounds) */
    struct { Scratch eq, nlp, sqp, ls, bnd, lbfgs, newton; } scratch;
    /* ntgb_solve_eq_newton: bit j of cost_out[0 / 1 / 2] = output j in the initial / trajectory / final cost's
     * active variables; the structure ntg_newton.h derives from them, built on the first call that needs it */
    unsigned cost_out[3] = {0, 0, 0};
    struct {
        bool ready = false;
        int K = 0, w = 0;
        std::vector<int> hperm;
        int *perm = nullptr, *color = nullptr;
        unsigned char *hmask = nullptr;
        double *ata = nullptr;
        double ata_max = 0.0;
    } newton;
    /* ntgb_solve_eq_async / ntgb_solve_sqp_async: their own work spaces, apart from `scratch`, so that no
     * synchronous call moves an array that a captured graph uses; halving = the step table 2^-a, a < 16 */
    struct {
        AsyncWork eq, sqp;
        double *halving = nullptr;
    } async;
};

namespace {

/* launch and return THIS launch's status (cudaGetLastError() could hand back a stale error that
 * another library left on the thread) */
template <class... KArgs, class... Args>
cudaError_t launch(void (*kern)(KArgs...), unsigned grid, unsigned block, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.stream = st;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

template <class T>
int dev_alloc(ntgb_problem *pb, T **ptr, size_t n)
{
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, (n > 0 ? n : 1) * sizeof(T));
    if (e != cudaSuccess) return fail(NTGB_ENOMEM, "cudaMalloc(%zu bytes): %s", n * sizeof(T), cudaGetErrorString(e));
    pb->allocs.push_back(p);
    *ptr = static_cast<T *>(p);
    return 0;
}

template <class T>
int dev_upload(ntgb_problem *pb, T **ptr, const T *src, size_t n)
{
    int rc = dev_alloc(pb, ptr, n);
    if (rc) return rc;
    if (n) CUDA_TRY(cudaMemcpy(*ptr, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

/* one pass over a scratch layout: take(n, p...) hands each p the next n elements, every array starting on a
 * 256-byte boundary as if it had been allocated alone; with a null base the pass only counts bytes */
struct Carve {
    char *base;
    size_t off = 0;
    template <class... T>
    void take(size_t n, T *&...p)
    {
        (one(p, n), ...);
    }
    template <class T>
    void one(T *&p, size_t n)
    {
        off = (off + 255) & ~(size_t)255;
        p = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += n * sizeof(T);
    }
};

/* layout(Carve &) takes every array of a call once, in order: it runs once to size s and once to hand out the
 * pointers.  s grows when the call needs more and never shrinks; the old buffer may still be in use by work
 * queued on st, so st is synchronized before it is freed.  grow == false (a reserved work space): a layout
 * larger than s is an error. */
template <class Layout>
int scratch_carve(Scratch &s, cudaStream_t st, Layout layout, bool grow = true)
{
    Carve size{nullptr};
    layout(size);
    if (size.off > s.bytes) {
        if (!grow)
            return fail(NTGB_EINVAL, "internal error: a reserved work space of %zu bytes cannot hold %zu", s.bytes, size.off);
        CUDA_TRY(cudaStreamSynchronize(st));
        cudaFree(s.p);
        s.p = nullptr;
        s.bytes = 0;
        CUDA_TRY(cudaMalloc(&s.p, size.off));
        s.bytes = size.off;
    }
    Carve c{static_cast<char *>(s.p)};
    layout(c);
    if (c.off != size.off)
        return fail(NTGB_EINVAL, "internal error: a scratch layout of %zu bytes carved %zu", size.off, c.off);
    return 0;
}

/* 1 when all P problems have counted themselves finished in *count, 0 when not, < 0 on a CUDA error */
int all_finished(const int *count, int P, cudaStream_t st)
{
    int done = 0;
    CUDA_TRY(cudaMemcpyAsync(&done, count, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return done >= P ? 1 : 0;
}

/* step table of the solvers' line searches: alpha[a] = 2^-a, n <= 16 */
int upload_halving(double *alpha, int n, cudaStream_t st)
{
    double ha[16];
    for (int a = 0; a < n; a++) ha[a] = std::ldexp(1.0, -a);
    CUDA_TRY(cudaMemcpyAsync(alpha, ha, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    return 0;
}

/* ------------------------------- K0 kernels ------------------------------- */

/* augmented knots (PGS `knots`, reference src/colloc.c:92-93) */
__global__ void k0_augknots(const double *brk, int ninterv, int order, int mult, double *aug, int naug)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < naug) aug[i] = ntgb::pgs_augknot(brk, ninterv, order, mult, i);
}

/* one thread per breakpoint: interv + bsplvd on the augmented knots, interv on
 * the raw knots for the block offset (reference src/colloc.c:95-111) */
__global__ void k0_tables(const double *aug, int naug, const double *brk, int nknots, const double *bps,
                          int nbps, int order, int mult, int md, double *Bn, double *Bt, int *off,
                          int *left_out)
{
    const int bp = blockIdx.x * blockDim.x + threadIdx.x;
    if (bp >= nbps) return;
    double a[PGS_MAXK * PGS_MAXK];
    double db[PGS_MAXK * PGS_MAXK];
    const double x = bps[bp];
    const int left = ntgb::pgs_interv(aug, naug, x);
    for (int i = 0; i < order * md; i++) db[i] = 0.0;
    ntgb::pgs_bsplvd(aug, order, x, left, a, db, md);
    for (int k = 0; k < order; k++)
        for (int d = 0; d < md; d++) {
            const double v = db[d * order + k];
            Bn[((size_t)bp * order + k) * md + d] = v;
            Bt[((size_t)k * md + d) * nbps + bp] = v;
        }
    const int lk = ntgb::pgs_interv(brk, nknots, x);
    off[bp] = (lk - 1) * (order - mult);
    left_out[bp] = left;
}

/* batched linear constraints: lin[p][r] = sum over the band of A[r][.]*C[p][.]
 * (what NPSOL computes as A*x for its linear rows) and the linear violation */
__global__ void k_linear(const double *Aband, const int *Acol0, const double *lb, const double *ub,
                         int nclin, int nout, int S, ntgb_devtab T, int P, const double *C,
                         double *lin, double *viol)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (long long)P * nclin) return;
    const int p = (int)(q / nclin), r = (int)(q - (long long)p * nclin);
    const double *Cp = C + (size_t)p * T.nC;
    double acc = 0.0;
    for (int j = 0; j < nout; j++) {
        const int c0 = Acol0[r * nout + j];
        for (int k = 0; k < T.order[j]; k++) acc = acc + Aband[(size_t)r * S + T.jk0[j] + k] * Cp[c0 + k];
    }
    if (lin) lin[(size_t)p * nclin + r] = acc;
    if (viol) {
        double v = 0.0;
        if (lb[r] - acc > v) v = lb[r] - acc;
        if (acc - ub[r] > v) v = acc - ub[r];
        if (v > 0.0) atomicMax(reinterpret_cast<unsigned long long *>(viol + p),
                               (unsigned long long)__double_as_longlong(v));
    }
}

/* batched SplineInterp, reference src/colloc.c:449-484: one thread per
 * (problem, time, output); interv + bsplvd at an arbitrary x on the device */
struct InterpDesc {
    int nout, nC, nz;
    int order[NTGB_MAXOUT], mult[NTGB_MAXOUT], md[NTGB_MAXOUT], ninterv[NTGB_MAXOUT], ncoef[NTGB_MAXOUT];
    int iC[NTGB_MAXOUT], iz[NTGB_MAXOUT];
    const double *aug[NTGB_MAXOUT];
    const double *knots[NTGB_MAXOUT];
};

__global__ void k_spline_interp(InterpDesc D, int P, const double *C, int nt, const double *t, double *out)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)P * nt * D.nout;
    if (q >= total) return;
    const int j = (int)(q % D.nout);
    const long long pi = q / D.nout;
    const int i = (int)(pi % nt);
    const int p = (int)(pi / nt);
    const int order = D.order[j], md = D.md[j];
    double a[PGS_MAXK * PGS_MAXK];
    double db[PGS_MAXK * PGS_MAXK];
    const double x = t[i];
    const int naug = D.ncoef[j] + order;
    const int left1 = ntgb::pgs_interv(D.aug[j], naug, x);
    for (int e = 0; e < order * md; e++) db[e] = 0.0;
    ntgb::pgs_bsplvd(D.aug[j], order, x, left1, a, db, md);
    const int left2 = ntgb::pgs_interv(D.knots[j], D.ninterv[j] + 1, x);
    const int offset = (left2 - 1) * (order - D.mult[j]);
    const double *coefs = C + (size_t)p * D.nC + D.iC[j];
    for (int d = 0; d < md; d++) {
        double f = 0.0;
        for (int k = 0; k < order; k++) f = f + db[d * order + k] * coefs[offset + k];
        out[((size_t)p * nt + i) * D.nz + D.iz[j] + d] = f;
    }
}

/* trial points of the line search: Ct[(p*nalpha + a)][.] = C[p][.] + alpha[a]*dC[p][.] */
__global__ void k_ls_trial(const double *C, const double *dC, const double *alpha, int P, int nalpha, int nC,
                           double *Ct)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)P * nalpha * nC;
    if (q >= total) return;
    const int e = (int)(q % nC);
    const long long pa = q / nC;
    const int a = (int)(pa % nalpha);
    const long long p = pa / nalpha;
    Ct[q] = C[p * nC + e] + alpha[a] * dC[p * nC + e];
}

/* per problem: first alpha satisfying Armijo on phi = f + mu*max(viol_nl, viol_lin), else argmin */
__global__ void k_ls_pick(const double *res, const double *lv, const double *alpha, int P, int nalpha, double mu,
                          double c1, const double *phi0, const double *dphi0, const double *C, const double *dC,
                          int nC, double *alpha_best, double *phi_best, double *C_new)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    int best = 0, chosen = -1;
    double phib = 0.0;
    for (int a = 0; a < nalpha; a++) {
        const size_t i = (size_t)p * nalpha + a;
        double v = res[2 * i + 1];
        if (lv != nullptr && lv[i] > v) v = lv[i];
        const double phi = res[2 * i] + mu * v;
        if (a == 0 || phi < phib) { phib = phi; best = a; }
        if (chosen < 0 && phi0 != nullptr) {
            const double slope = dphi0 != nullptr ? dphi0[p] : 0.0;
            if (phi <= phi0[p] + c1 * alpha[a] * slope) chosen = a;
        }
    }
    if (chosen < 0) chosen = best;
    const size_t ic = (size_t)p * nalpha + chosen;
    double v = res[2 * ic + 1];
    if (lv != nullptr && lv[ic] > v) v = lv[ic];
    if (alpha_best) alpha_best[p] = alpha[chosen];
    if (phi_best) phi_best[p] = res[2 * ic] + mu * v;
    if (C_new)
        for (int e = 0; e < nC; e++) C_new[(size_t)p * nC + e] = C[(size_t)p * nC + e] + alpha[chosen] * dC[(size_t)p * nC + e];
}

/* ---- ntgb_solve_eq: reduced-space BFGS, one thread per problem ------------------------------
 * Per-problem vectors are stored component-major ([k][P]) so that a warp's accesses coalesce. */
constexpr int kSolveMaxNr = 32;

__global__ void k_solve_init(int P, int nC, int nr, const double *N, const double *Cpart, int Cstride, double *C,
                             double *y, double *H, int *state, int *iters, int *fails)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    /* per-problem bounds (Cstride = nC): k_bounds_prep has set state / iters, a rejected problem keeps its C */
    if (Cstride != 0 && state[p] == NTGB_STATUS_BAD_BOUNDS) return;
    Cpart += (size_t)p * Cstride;
    double *Cp = C + (size_t)p * nC;
    for (int k = 0; k < nr; k++) {
        double a = 0.0;
        for (int e = 0; e < nC; e++) a += N[(size_t)k * nC + e] * (Cp[e] - Cpart[e]);
        y[(size_t)k * P + p] = a;
    }
    for (int e = 0; e < nC; e++) {
        double a = Cpart[e];
        for (int k = 0; k < nr; k++) a += N[(size_t)k * nC + e] * y[(size_t)k * P + p];
        Cp[e] = a;
    }
    for (int k = 0; k < nr; k++)
        for (int l = 0; l < nr; l++) H[((size_t)k * nr + l) * P + p] = k == l ? 1.0 : 0.0;
    state[p] = 0;
    iters[p] = 0;
    fails[p] = -1; /* -1 no previous step, 1 last step failed (both: H = I, steepest descent);
                      2 previous step exists and H is still the identity; 0 normal;
                      -2 no previous step but H carries over (set by the augmented-Lagrangian driver) */
}

/* reduced gradient, convergence test, BFGS update of the inverse Hessian, search direction */
__global__ void k_solve_dir(int P, int nC, int nr, const double *N, const double *f, const double *g, double gtol,
                            const double *y, double *yp, double *grp, double *H, double *d, double *dC,
                            double *phi0, double *dphi0, int *state, int *fails, int *count)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    double *dCp = dC + (size_t)p * nC;
    phi0[p] = f[p];
    if (state[p] != 0) {
        for (int e = 0; e < nC; e++) dCp[e] = 0.0;
        dphi0[p] = 0.0;
        return;
    }
    double gr[kSolveMaxNr], s[kSolveMaxNr], u[kSolveMaxNr];
    const double *gp = g + (size_t)p * nC;
    double gmax = 0.0, gg = 0.0;
    for (int k = 0; k < nr; k++) {
        double a = 0.0;
        for (int e = 0; e < nC; e++) a += N[(size_t)k * nC + e] * gp[e];
        gr[k] = a;
        gmax = fmax(gmax, fabs(a));
        gg += a * a;
    }
    const double fabsv = fabs(f[p]);
    if (!(gmax > gtol * (fabsv > 1.0 ? fabsv : 1.0))) {
        /* converged (or NaN: nothing sensible left to do) */
        state[p] = gmax == gmax ? 1 : 2;
        atomicAdd(count, 1);
        for (int e = 0; e < nC; e++) dCp[e] = 0.0;
        dphi0[p] = 0.0;
        return;
    }
#define HH(k, l) H[((size_t)(k) * nr + (l)) * P + p]
    int fl = fails[p];
    if (fl == 0 || fl == 2) {
        /* s = y - y_prev, u = gr - gr_prev */
        double su = 0.0, ss = 0.0, uu = 0.0;
        for (int k = 0; k < nr; k++) {
            s[k] = y[(size_t)k * P + p] - yp[(size_t)k * P + p];
            u[k] = gr[k] - grp[(size_t)k * P + p];
            su += s[k] * u[k]; ss += s[k] * s[k]; uu += u[k] * u[k];
        }
        if (su > 1e-10 * sqrt(ss * uu) && su > 0.0) {
            if (fl == 2) /* first update after a (re)start: scale the identity to the curvature seen */
                for (int k = 0; k < nr; k++) HH(k, k) = su / uu;
            double Hu[kSolveMaxNr], uHu = 0.0;
            for (int k = 0; k < nr; k++) {
                double a = 0.0;
                for (int l = 0; l < nr; l++) a += HH(k, l) * u[l];
                Hu[k] = a;
                uHu += a * u[k];
            }
            const double rho = 1.0 / su, c2 = (su + uHu) * rho * rho;
            for (int k = 0; k < nr; k++)
                for (int l = 0; l < nr; l++)
                    HH(k, l) += c2 * s[k] * s[l] - rho * (Hu[k] * s[l] + s[k] * Hu[l]);
        }
    }
    double slope = 0.0, dd = 0.0;
    for (int k = 0; k < nr; k++) {
        double a = 0.0;
        for (int l = 0; l < nr; l++) a -= HH(k, l) * gr[l];
        s[k] = a;
        slope += a * gr[k];
        dd += a * a;
    }
    if (!(slope < -1e-12 * sqrt(gg * dd))) {
        /* not a descent direction: restart from steepest descent */
        for (int k = 0; k < nr; k++)
            for (int l = 0; l < nr; l++) HH(k, l) = k == l ? 1.0 : 0.0;
        for (int k = 0; k < nr; k++) s[k] = -gr[k];
        slope = -gg;
        dd = gg;
        fl = 1;
        fails[p] = 1;
    }
#undef HH
    /* a unit step along a raw gradient can be far too long: bound the first trial step */
    const double dn = sqrt(dd);
    const bool steepest = fl == -1 || fl == 1;
    const double scale = (steepest && dn > 1.0) ? 1.0 / dn : 1.0;
    if (fl == 2) fails[p] = 0;
    for (int k = 0; k < nr; k++) {
        s[k] *= scale;
        d[(size_t)k * P + p] = s[k];
        yp[(size_t)k * P + p] = y[(size_t)k * P + p];
        grp[(size_t)k * P + p] = gr[k];
    }
    for (int e = 0; e < nC; e++) {
        double a = 0.0;
        for (int k = 0; k < nr; k++) a += N[(size_t)k * nC + e] * s[k];
        dCp[e] = a;
    }
    dphi0[p] = slope * scale;
}

/* accept the line-search step (or count a failure), rebuild C from the reduced variables */
__global__ void k_solve_update(int P, int nC, int nr, const double *N, const double *Cpart, int Cstride,
                               const double *phi0, const double *alpha_best, const double *phi_best, const double *d,
                               double *y, double *H, double *C, int *state, int *iters, int *fails, int *count)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P || state[p] != 0) return;
    Cpart += (size_t)p * Cstride;
    iters[p] += 1;
    if (!(phi_best[p] < phi0[p])) {
        /* no decrease along d: retry once from steepest descent, then give up */
        const bool was_reset = fails[p] == -1 || fails[p] == 1;
        if (was_reset) { state[p] = 2; atomicAdd(count, 1); return; }
        for (int k = 0; k < nr; k++)
            for (int l = 0; l < nr; l++) H[((size_t)k * nr + l) * P + p] = k == l ? 1.0 : 0.0;
        fails[p] = 1;
        return;
    }
    fails[p] = (fails[p] == -1 || fails[p] == 1) ? 2 : 0;
    const double a = alpha_best[p];
    for (int k = 0; k < nr; k++) y[(size_t)k * P + p] += a * d[(size_t)k * P + p];
    double *Cp = C + (size_t)p * nC;
    for (int e = 0; e < nC; e++) {
        double v = Cpart[e];
        for (int k = 0; k < nr; k++) v += N[(size_t)k * nC + e] * y[(size_t)k * P + p];
        Cp[e] = v;
    }
}

/* Host: the minimum-norm solution of A*C = b (A m x n, column-major) and nr = n - rank(A), by Householder QR
 * with column pivoting of A^T.  Optional outputs: N, the orthonormal null-space basis of A ([nr][n], the last
 * nr columns of Q); Q1, the orthonormal basis of its row space ([r][n], the first r columns of Q, r = n - nr);
 * Mop, the linear operator of that solution, Cpart = Mop b for any right-hand side b ([n][m] row-major; zero
 * columns for the rows the pivoting found dependent), which the per-problem-bounds solvers apply on the device. */
int reduce_linear(const std::vector<double> &A, int m, int n, const std::vector<double> &b, std::vector<double> *N,
                  std::vector<double> &Cpart, int &nr, std::vector<double> *Mop = nullptr, std::vector<double> *Q1 = nullptr)
{
    std::vector<double> M((size_t)n * std::max(m, 1)), Q((size_t)n * n, 0.0), v(n);
    std::vector<int> perm(m);
    for (int j = 0; j < m; j++) {
        perm[j] = j;
        for (int i = 0; i < n; i++) M[i + (size_t)j * n] = A[j + (size_t)i * m];
    }
    for (int i = 0; i < n; i++) Q[i + (size_t)i * n] = 1.0;
    int r = 0;
    double norm0 = 0.0;
    for (int k = 0; k < std::min(n, m); k++) {
        int jb = k;
        double nb = -1.0;
        for (int j = k; j < m; j++) {
            double a = 0.0;
            for (int i = k; i < n; i++) a += M[i + (size_t)j * n] * M[i + (size_t)j * n];
            if (a > nb) { nb = a; jb = j; }
        }
        const double norm = std::sqrt(nb);
        if (k == 0) norm0 = norm;
        if (!(norm > 1e-11 * std::max(norm0, 1e-300))) break;
        if (jb != k) {
            for (int i = 0; i < n; i++) std::swap(M[i + (size_t)k * n], M[i + (size_t)jb * n]);
            std::swap(perm[k], perm[jb]);
        }
        double *col = &M[(size_t)k * n];
        const double alpha = col[k] > 0.0 ? -norm : norm;
        double vv = 0.0;
        for (int i = k; i < n; i++) { v[i] = col[i]; }
        v[k] -= alpha;
        for (int i = k; i < n; i++) vv += v[i] * v[i];
        if (vv > 0.0) {
            for (int j = k; j < m; j++) {
                double t = 0.0;
                for (int i = k; i < n; i++) t += v[i] * M[i + (size_t)j * n];
                t = 2.0 * t / vv;
                for (int i = k; i < n; i++) M[i + (size_t)j * n] -= t * v[i];
            }
            for (int i = 0; i < n; i++) {
                double t = 0.0;
                for (int l = k; l < n; l++) t += Q[i + (size_t)l * n] * v[l];
                t = 2.0 * t / vv;
                for (int l = k; l < n; l++) Q[i + (size_t)l * n] -= t * v[l];
            }
        }
        r++;
    }
    /* A^T Pi = Q R  =>  R1^T (Q1^T C) = (Pi^T b)[0:r] */
    std::vector<double> w(r);
    for (int i = 0; i < r; i++) {
        double a = b[perm[i]];
        for (int l = 0; l < i; l++) a -= M[l + (size_t)i * n] * w[l];
        w[i] = a / M[i + (size_t)i * n];
    }
    Cpart.assign(n, 0.0);
    for (int l = 0; l < r; l++)
        for (int i = 0; i < n; i++) Cpart[i] += Q[i + (size_t)l * n] * w[l];
    if (Mop) {
        /* column j = the same back substitution for b = e_j */
        Mop->assign((size_t)n * m, 0.0);
        std::vector<double> wj(r);
        for (int j = 0; j < m; j++) {
            for (int i = 0; i < r; i++) {
                double a = perm[i] == j ? 1.0 : 0.0;
                for (int l = 0; l < i; l++) a -= M[l + (size_t)i * n] * wj[l];
                wj[i] = a / M[i + (size_t)i * n];
            }
            for (int l = 0; l < r; l++)
                for (int i = 0; i < n; i++) (*Mop)[(size_t)i * m + j] += Q[i + (size_t)l * n] * wj[l];
        }
    }
    double bmax = 0.0, res = 0.0;
    for (int j = 0; j < m; j++) {
        double a = -b[j];
        for (int i = 0; i < n; i++) a += A[j + (size_t)i * m] * Cpart[i];
        res = std::max(res, std::fabs(a));
        bmax = std::max(bmax, std::fabs(b[j]));
    }
    if (res > 1e-8 * (1.0 + bmax)) return fail(NTGB_EINVAL, "linear equality constraints are inconsistent (residual %g)", res);
    nr = n - r;
    if (N) {
        N->resize((size_t)nr * n);
        for (int k = 0; k < nr; k++)
            for (int i = 0; i < n; i++) (*N)[(size_t)k * n + i] = Q[i + (size_t)(r + k) * n];
    }
    if (Q1) {
        Q1->resize((size_t)r * n);
        for (int k = 0; k < r; k++)
            for (int i = 0; i < n; i++) (*Q1)[(size_t)k * n + i] = Q[i + (size_t)k * n];
    }
    return 0;
}

/* ---- ntgb_solve_nlp: augmented Lagrangian on top of the reduced-space BFGS kernels above ----
 * general constraints h = [A_in*C ; c(C)], bounds hl <= h <= hu, multipliers lam, penalty rho.
 * PHR form: t = h + lam/rho, p = clamp(t, hl, hu), mu = rho*(t - p),
 *           L_A = f + sum( rho/2*(t-p)^2 - lam^2/(2 rho) ),  grad L_A = g + dh^T mu. */
__device__ __forceinline__ double alm_row(double h, double lam, double rho, double lo, double hi, double &mu,
                                          double &viol)
{
    const double t = h + lam / rho;
    const double pr = t < lo ? lo : (t > hi ? hi : t);
    mu = rho * (t - pr);
    double v = 0.0;
    if (lo - h > v) v = lo - h;
    if (h - hi > v) v = h - hi;
    const double sc = fmax(1.0, fmax(fabs(lo) < 1e19 ? fabs(lo) : 0.0, fabs(hi) < 1e19 ? fabs(hi) : 0.0));
    viol = v / sc;
    return 0.5 * rho * (t - pr) * (t - pr) - 0.5 * lam * lam / rho;
}

/* one warp per evaluation point q (a problem, or a line-search trial of problem q / nalpha):
 * multipliers (optional), augmented Lagrangian value, scaled violation */
__global__ void k_alm_mu(int Q, int nalpha, int ncnln, int nclin, int n_li, const int *li_idx, const double *hl,
                         const double *hu, const double *lam, const double *rho, const double *f, const double *c,
                         const double *lin, double *mu, double *LA, double *viol, int LAstride, const int *pidx)
{
    const int q = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= Q) return;
    const int p = pidx != nullptr ? pidx[q / nalpha] : q / nalpha;
    const int m = n_li + ncnln;
    const double r = rho[p];
    double acc = 0.0, vmax = 0.0;
    for (int i = lane; i < m; i += 32) {
        const double h = i < n_li ? lin[(size_t)q * nclin + li_idx[i]] : c[(size_t)q * ncnln + (i - n_li)];
        double mui, vi;
        acc += alm_row(h, lam[(size_t)p * m + i], r, hl[i], hu[i], mui, vi);
        vmax = fmax(vmax, vi);
        if (mu != nullptr) mu[(size_t)q * m + i] = mui;
    }
    for (int d = 16; d > 0; d >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, d);
        vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
    }
    if (lane == 0) {
        LA[(size_t)q * LAstride] = f[q] + acc;
        if (viol != nullptr) viol[q] = vmax;
    }
}

/* gradient of the augmented Lagrangian, one thread per (problem, column): g + J^T mu_nl + A_in^T mu_li,
 * J in band layout (include/ntg_b200.h, NTGB_JAC_BAND) gathered over the column's support */
__global__ void k_alm_grad(int P, ntgb_devtab T, int nclin, int n_li, const int *li_idx, const double *Adense,
                           const double *g, const double *J, const double *mu, double *gA)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (long long)P * T.nC) return;
    const int p = (int)(q / T.nC), c = (int)(q - (long long)p * T.nC);
    const int m = n_li + T.ncnln, nbps = T.nbps, S = T.S;
    const double *mup = mu + (size_t)p * m;
    double acc = g[q];
    for (int i = 0; i < n_li; i++) acc += mup[i] * Adense[(size_t)c * nclin + li_idx[i]];
    if (T.ncnln > 0) {
        const double *Jp = J + (size_t)p * T.ncnln * S;
        const double *mun = mup + n_li;
        for (int j = 0; j < T.nout; j++) {
            const int cl = c - T.iC[j];
            if (cl < 0 || cl >= T.ncoef[j]) continue;
            const int ord = T.order[j], s0 = T.jk0[j];
            if (cl < ord) /* initial rows: columns from iC_j, src/colloc.c:254 */
                for (int r = 0; r < T.nnlic; r++) acc += mun[r] * Jp[(size_t)r * S + s0 + cl];
            if (T.nnltc > 0) {
                const int lo = T.col_lo[c], hi = T.col_hi[c];
                for (int bp = lo; bp <= hi; bp++) {
                    const int k = cl - T.off[j][bp];
                    if (k < 0 || k >= ord) continue;
                    for (int mm = 0; mm < T.nnltc; mm++)
                        acc += mun[T.nnlic + mm * nbps + bp] *
                               Jp[ntgb_band_index(T.nnlic, T.nnltc, S, nbps, T.band_tile, mm, s0 + k, bp)];
                }
            }
            if (T.nnlfc > 0) {
                const int k = cl - T.off[j][nbps - 1];
                const int rb = T.nnlic + T.nnltc * nbps;
                if (k >= 0 && k < ord)
                    for (int r = 0; r < T.nnlfc; r++) acc += mun[rb + r] * Jp[(size_t)(rb + r) * S + s0 + k];
            }
        }
    }
    gA[q] = acc;
}

/* between two rounds: multipliers <- mu, penalty up if the violation stalls, BFGS restarted;
 * a problem is finished when it is feasible to ctol and its inner iteration had converged */
__global__ void k_alm_outer(int P, int m, int nr, const double *mu, double *lam, double *rho, const double *viol,
                            double *violprev, double ctol, double rho_mul, double rho_max, int last, double *H, int *state, int *fails,
                            int *fin, int *count)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    if (fin[p] == 0) {
        const bool inner_ok = state[p] != 0; /* reduced gradient below gtol (1) or no further decrease (2) */
        if (viol[p] <= ctol && inner_ok) {
            fin[p] = state[p];
        } else if (!last) {
            for (int i = 0; i < m; i++) lam[(size_t)p * m + i] = mu[(size_t)p * m + i];
            if (viol[p] > 0.25 * violprev[p] && rho[p] * rho_mul <= rho_max) rho[p] *= rho_mul;
            violprev[p] = viol[p];
            /* the merit function changed: the next BFGS update would pair gradients of two different
             * functions, so it is skipped (-2 = no previous step, inverse Hessian kept) */
            state[p] = 0;
            fails[p] = -2;
        }
    }
    if (fin[p] != 0) {
        state[p] = 1; /* inert for the inner kernels */
        atomicAdd(count, 1);
    }
}

__global__ void k_alm_prep(int P, int m, double rho0, double *lam, double *rho, double *violprev, int *fin)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    for (int i = 0; i < m; i++) lam[(size_t)p * m + i] = 0.0;
    rho[p] = rho0;
    violprev[p] = 1e300;
    fin[p] = 0;
}

/* k_ls_trial for the second stage of two_stage_search: the trial points of the n problems listed in idx.  Kept
 * apart from k_ls_trial: an optional index list there made ntgb_linesearch slower (65 536 problems x 12 steps:
 * 749.7 against 741.6 us on a B200 at 1000 W) and ntgb_solve_nlp 0.7 % slower. */
__global__ void k_ls_trial_idx(const double *C, const double *dC, const double *alpha, const int *idx, int n, int nalpha,
                               int nC, double *Ct)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)n * nalpha * nC;
    if (q >= total) return;
    const int e = (int)(q % nC);
    const long long ia = q / nC;
    const int a = (int)(ia % nalpha);
    const long long p = idx[ia / nalpha];
    Ct[q] = C[p * nC + e] + alpha[a] * dC[p * nC + e];
}

/* stage 1 of two_stage_search: first coarse alpha with Armijo decrease, else the best one seen; problems without an
 * Armijo step (and still running) are appended to idx */
__global__ void k_alm_pick1(const double *res, const double *alpha, int P, int nalpha, double c1, const double *phi0,
                            const double *dphi0, const int *state, double *alpha_best, double *phi_best, int *idx,
                            int *nidx)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    int best = 0, chosen = -1;
    double phib = 0.0;
    for (int a = 0; a < nalpha; a++) {
        const double phi = res[2 * ((size_t)p * nalpha + a)];
        if (a == 0 || phi < phib) { phib = phi; best = a; }
        if (chosen < 0 && phi <= phi0[p] + c1 * alpha[a] * dphi0[p]) chosen = a;
    }
    const int pick = chosen >= 0 ? chosen : best;
    alpha_best[p] = alpha[pick];
    phi_best[p] = res[2 * ((size_t)p * nalpha + pick)];
    if (chosen < 0 && state[p] == 0) idx[atomicAdd(nidx, 1)] = p;
}

/* stage 2: the fine alphas of the listed problems */
__global__ void k_alm_pick2(const double *res, const double *alpha, const int *idx, int n, int nalpha, double c1,
                            const double *phi0, const double *dphi0, double *alpha_best, double *phi_best)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = idx[i];
    int best = -1, chosen = -1;
    double phib = phi_best[p];
    for (int a = 0; a < nalpha; a++) {
        const double phi = res[2 * ((size_t)i * nalpha + a)];
        if (phi < phib) { phib = phi; best = a; }
        if (chosen < 0 && phi <= phi0[p] + c1 * alpha[a] * dphi0[p]) chosen = a;
    }
    const int pick = chosen >= 0 ? chosen : best;
    if (pick >= 0) {
        alpha_best[p] = alpha[pick];
        phi_best[p] = res[2 * ((size_t)i * nalpha + pick)];
    }
}

int check_avs(const AV *av, int n, const ntgb_setup *s, const char *what)
{
    if (n < 0 || (n > 0 && av == nullptr)) return fail(NTGB_EINVAL, "%s: bad active-variable list", what);
    for (int i = 0; i < n; i++)
        if (av[i].output < 0 || av[i].output >= s->nout || av[i].deriv < 0 ||
            av[i].deriv >= s->maxderiv[av[i].output])
            return fail(NTGB_EINVAL, "%s[%d] = {%d,%d} out of range", what, i, av[i].output, av[i].deriv);
    return 0;
}

void add_mask(unsigned (*mask)[NTGB_MAXOUT], const AV *av, int n, int cls_bits)
{
    for (int cls = 0; cls < 4; cls++) {
        const bool first = cls & 1, last = cls & 2;
        const bool hit = (cls_bits == 0) || (cls_bits == 1 && first) || (cls_bits == 2 && last);
        if (!hit) continue;
        for (int i = 0; i < n; i++) mask[cls][av[i].output] |= 1u << av[i].deriv;
    }
}

const ntgb_pack *match_pack(const ntgb_setup *s)
{
    std::lock_guard<std::mutex> lk(g_reg_mu);
    for (const ntgb_pack &pk : registry()) {
        bool ok = true, any = false;
        auto chk = [&](int count, const void *want, const void *have) {
            if (count != 0 && want != nullptr) {
                any = true;
                if (want != have) ok = false;
            }
        };
        chk(s->nicf, (const void *)s->icf, (const void *)pk.icf);
        chk(s->nucf, (const void *)s->ucf, (const void *)pk.ucf);
        chk(s->nfcf, (const void *)s->fcf, (const void *)pk.fcf);
        chk(s->nnlic, (const void *)s->nlicf, (const void *)pk.nlicf);
        chk(s->nnltc, (const void *)s->nltcf, (const void *)pk.nltcf);
        chk(s->nnlfc, (const void *)s->nlfcf, (const void *)pk.nlfcf);
        if (ok && any) return &pk;
    }
    return nullptr;
}

/* one Jacobian-style band row on the host from a constant derivative vector
 * (linear constraints: InitialConstraintsMatrix etc., src/constraints.c:225-261) */
void host_band_row(const ntgb_problem *pb, const double *dz, int bp, double *band)
{
    for (int j = 0; j < pb->dims.nout; j++) {
        const int order = pb->order[j], md = pb->maxderiv[j];
        const double *B = pb->hB.data() + pb->hB_off[j] + (size_t)bp * order * md;
        for (int k = 0; k < order; k++) {
            double acc = 0.0;
            for (int l = 0; l < md; l++) acc = acc + dz[pb->tab.iz[j] + l] * B[k * md + l];
            band[pb->tab.jk0[j] + k] = acc;
        }
    }
}

/* reduced form shared by the batched solvers: linear equality rows eliminated (C = Cpart + N y), the other
 * linear rows and the nonlinear rows kept as general constraints.  The part every solver uses (the row split,
 * Cpart, M, Ae, the general rows' bounds) is built on the first call; the basis each solver needs on top of it
 * on the first call that asks for it: want_N, the null-space basis N and the warm digest (ntgb_solve_eq,
 * ntgb_solve_nlp, ntgb_solve_sqp); want_Q1, the row-space basis Q1 (ntgb_solve_eq_lbfgs, which puts nothing
 * of size nC x nr on the device).  A later call that needs the other basis repeats the host QR, which
 * gives the same bits. */
int reduced_form(ntgb_problem *pb, bool want_N, bool want_Q1)
{
    auto &al = pb->alm;
    const bool need_N = want_N && !al.N, need_Q1 = want_Q1 && !al.Q1;
    if (al.ready && !need_N && !need_Q1) return 0;
    const ntgb_dims &dm = pb->dims;
    const int nC = dm.nC, nclin = dm.nclin, ncnln = dm.ncnln;
    int rc;
    /* split the linear rows: equalities are eliminated, the rest become general constraints */
    std::vector<int> eq, li;
    for (int i = 0; i < nclin; i++) (pb->lin_lb[i] == pb->lin_ub[i] ? eq : li).push_back(i);
    const int me = (int)eq.size();
    std::vector<double> Ae((size_t)std::max(me, 1) * nC, 0.0), be((size_t)me);
    for (int r = 0; r < me; r++) {
        be[r] = pb->lin_lb[eq[r]];
        for (int c = 0; c < nC; c++) Ae[r + (size_t)c * me] = pb->A[eq[r] + (size_t)c * nclin];
    }
    std::vector<double> N, Cpart, Mop, Q1;
    int nr = 0;
    if ((rc = reduce_linear(Ae, me, nC, be, need_N ? &N : nullptr, Cpart, nr, al.ready ? nullptr : &Mop,
                            need_Q1 ? &Q1 : nullptr)))
        return rc;
    if (!al.ready) {
        al.nr = nr;
        al.eq = eq;
        al.li = li;
        al.n_li = (int)li.size();
        al.m = al.n_li + ncnln;
        if ((rc = dev_upload(pb, &al.Cpart, Cpart.data(), Cpart.size()))) return rc;
        /* for per-problem right-hand sides: Cpart = M be and the rows to check the residual against */
        std::vector<double> Aer((size_t)std::max(me, 1) * nC, 0.0);
        for (int r = 0; r < me; r++)
            for (int c = 0; c < nC; c++) Aer[(size_t)r * nC + c] = Ae[r + (size_t)c * me];
        if (Mop.empty()) Mop.push_back(0.0);
        if ((rc = dev_upload(pb, &al.M, Mop.data(), Mop.size()))) return rc;
        if ((rc = dev_upload(pb, &al.Ae, Aer.data(), Aer.size()))) return rc;
        if (li.empty()) li.push_back(0);
        if ((rc = dev_upload(pb, &al.li_idx, li.data(), li.size()))) return rc;
        /* bounds of the general constraints: NPSOL's bl/bu behind the variables and, for the
         * linear rows, the expanded linear bounds */
        std::vector<double> bl((size_t)nC + nclin + ncnln), bu(bl.size());
        if ((rc = ntgb_get_bounds(pb, bl.data(), bu.data()))) return rc;
        std::vector<double> hl((size_t)std::max(al.m, 1), 0.0), hu((size_t)std::max(al.m, 1), 0.0);
        for (int i = 0; i < al.n_li; i++) { hl[i] = pb->lin_lb[al.li[i]]; hu[i] = pb->lin_ub[al.li[i]]; }
        for (int i = 0; i < ncnln; i++) { hl[al.n_li + i] = bl[(size_t)nC + nclin + i]; hu[al.n_li + i] = bu[(size_t)nC + nclin + i]; }
        if ((rc = dev_upload(pb, &al.hl, hl.data(), hl.size()))) return rc;
        if ((rc = dev_upload(pb, &al.hu, hu.data(), hu.size()))) return rc;
        std::vector<double> Ad = pb->A;
        if (Ad.empty()) Ad.push_back(0.0);
        if ((rc = dev_upload(pb, &al.A, Ad.data(), Ad.size()))) return rc;
        al.ready = true;
    }
    if (need_N) {
        al.hN = N;
        al.digest = ntgb::warm_digest(nC, nr, al.m, al.n_li, al.li.data(), N.data());
        if (N.empty()) N.push_back(0.0);
        if ((rc = dev_upload(pb, &al.N, N.data(), N.size()))) return rc;
    }
    if (need_Q1) {
        al.r = nC - nr;
        if (Q1.empty()) Q1.push_back(0.0);
        if ((rc = dev_upload(pb, &al.Q1, Q1.data(), Q1.size()))) return rc;
    }
    return 0;
}

/* the reduced form of the solvers that work on y (C = Cpart + N y) */
int alm_prepare(ntgb_problem *pb) { return reduced_form(pb, true, false); }

/* the SQP entry points (`who`): alm's reduced form, which must leave a free direction, and once per problem
 * the reduced gradients ArN of the linear inequality rows and W = (Ae Ae')^-1 Ae for the multipliers of the
 * eliminated equality rows */
int sqp_prepare(ntgb_problem *pb, const char *who)
{
    int rc;
    if ((rc = alm_prepare(pb))) return rc;
    const auto &al = pb->alm;
    if (al.nr < 1) return fail(NTGB_EINVAL, "%s: the linear equalities leave no free direction", who);
    auto &sq = pb->sqp;
    if (sq.ready) return 0;
    const int nC = pb->dims.nC, nclin = pb->dims.nclin, nr = al.nr, n_li = al.n_li;
    std::vector<double> ArN((size_t)std::max(n_li, 1) * nr, 0.0);
    for (int i = 0; i < n_li; i++)
        for (int k = 0; k < nr; k++) {
            double a = 0.0;
            for (int e = 0; e < nC; e++) a += pb->A[al.li[i] + (size_t)e * nclin] * al.hN[(size_t)k * nC + e];
            ArN[(size_t)i * nr + k] = a;
        }
    if ((rc = dev_upload(pb, &sq.ArN, ArN.data(), ArN.size()))) return rc;
    const int me = (int)al.eq.size();
    std::vector<double> W((size_t)std::max(me, 1) * nC, 0.0), G((size_t)std::max(me, 1) * std::max(me, 1), 0.0);
    for (int r = 0; r < me; r++)
        for (int s = 0; s < me; s++) {
            double a = 0.0;
            for (int e = 0; e < nC; e++) a += pb->A[al.eq[r] + (size_t)e * nclin] * pb->A[al.eq[s] + (size_t)e * nclin];
            G[(size_t)r * me + s] = a;
        }
    /* Gauss-Jordan with partial pivoting on [G | Ae]; dependent rows get zero multipliers */
    for (int r = 0; r < me; r++)
        for (int e = 0; e < nC; e++) W[(size_t)r * nC + e] = pb->A[al.eq[r] + (size_t)e * nclin];
    double gmax = 0.0;
    for (int r = 0; r < me; r++) gmax = std::max(gmax, std::fabs(G[(size_t)r * me + r]));
    std::vector<char> dead(std::max(me, 1), 0);
    for (int k = 0; k < me; k++) {
        int piv = -1;
        double best = 1e-12 * std::max(gmax, 1e-300);
        for (int r = k; r < me; r++)
            if (std::fabs(G[(size_t)r * me + k]) > best) { best = std::fabs(G[(size_t)r * me + k]); piv = r; }
        if (piv < 0) { dead[k] = 1; continue; }
        if (piv != k) {
            for (int s = 0; s < me; s++) std::swap(G[(size_t)k * me + s], G[(size_t)piv * me + s]);
            for (int e = 0; e < nC; e++) std::swap(W[(size_t)k * nC + e], W[(size_t)piv * nC + e]);
        }
        const double d = G[(size_t)k * me + k];
        for (int s = 0; s < me; s++) G[(size_t)k * me + s] /= d;
        for (int e = 0; e < nC; e++) W[(size_t)k * nC + e] /= d;
        for (int r = 0; r < me; r++) {
            if (r == k) continue;
            const double t = G[(size_t)r * me + k];
            if (t == 0.0) continue;
            for (int s = 0; s < me; s++) G[(size_t)r * me + s] -= t * G[(size_t)k * me + s];
            for (int e = 0; e < nC; e++) W[(size_t)r * nC + e] -= t * W[(size_t)k * nC + e];
        }
    }
    for (int k = 0; k < me; k++)
        if (dead[k])
            for (int e = 0; e < nC; e++) W[(size_t)k * nC + e] = 0.0;
    if ((rc = dev_upload(pb, &sq.W, W.data(), W.size()))) return rc;
    std::vector<int> eqi = al.eq;
    if (eqi.empty()) eqi.push_back(0);
    if ((rc = dev_upload(pb, &sq.eq_idx, eqi.data(), eqi.size()))) return rc;
    sq.me = me;
    sq.ready = true;
    return 0;
}

/* IntegrateVector / IntegrateFMatrixCols (src/integrator.c:16-62) for a batch: one thread per (problem,
 * column) walks its n samples in the reference's order, with the reference's expression per rule */
__global__ void k_integrate(int rule, long long nchain, int n, const double *f, const double *t, double *I)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nchain) return;
    const double *fq = f + q * n;
    double acc = 0.0;
    if (rule == NTGB_QUAD_TRAPEZOID)
        for (int i = 0; i < n - 1; i++) acc += (t[i + 1] - t[i]) * (fq[i + 1] + fq[i]) / 2;
    else if (rule == NTGB_QUAD_FEULER)
        for (int i = 0; i < n - 1; i++) acc += (t[i + 1] - t[i]) * fq[i];
    else
        for (int i = 0; i < n - 1; i++) acc += (t[i + 1] - t[i]) * fq[i + 1];
    I[q] = acc;
}

/* ---- ntgb_solve_sqp: one CTA per problem runs ntg_sqp.cuh's sqp_step in shared memory ---------- */
namespace sqp = ntgb::sqp;

__global__ void k_scale_copy(long long n, double a, const double *x, double *y)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a * x[i];
}

struct SqpDesc {
    int nC, nr, m, n_li, nclin, ncnln;
    const double *N;      /* [nr][nC] */
    const double *ArN;    /* [n_li][nr] reduced gradients of the linear inequality rows */
    const int *li_idx;    /* [n_li] */
    const double *hl, *hu; /* [m] per problem, problem p's at hl + p*hstride (0: one shared set) */
    int Cstride, hstride;  /* per-problem strides of Cpart (0 or nC) and hl / hu (0 or m) */
    double gtol, ctol, rho_pen;
};

/* per-problem solver state, problem-major */
struct SqpArrays {
    double *y, *B, *lam, *sprev, *grLold, *grold, *d, *scal;
    int *flag, *istate;
};

/* warm (ntgb_solve_sqp_warm, nullptr otherwise): a row matching the setup (ntg_warm.h) gives B, nu and
 * the flags "no previous step, B is not the identity"; any other row starts cold like warm == nullptr */
__global__ void k_sqp_init(int P, SqpDesc D, SqpArrays S, const double *Cpart, double *C, int *state, int *iters,
                           const double *warm, ntgb::WarmKey wk)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int nC = D.nC, nr = D.nr;
    /* per-problem bounds: k_bounds_prep has set state / iters; a rejected problem keeps its C */
    const bool rejected = D.Cstride != 0 && state[p] == NTGB_STATUS_BAD_BOUNDS;
    Cpart += (size_t)p * D.Cstride;
    double *Cp = C + (size_t)p * nC, *y = S.y + (size_t)p * nr;
    if (!rejected) {
        for (int k = 0; k < nr; k++) {
            double a = 0.0;
            for (int e = 0; e < nC; e++) a += D.N[(size_t)k * nC + e] * (Cp[e] - Cpart[e]);
            y[k] = a;
        }
        for (int e = 0; e < nC; e++) {
            double a = Cpart[e];
            for (int k = 0; k < nr; k++) a += D.N[(size_t)k * nC + e] * y[k];
            Cp[e] = a;
        }
    }
    double nu;
    const bool hot = ntgb::warm_load(warm != nullptr && !rejected ? warm + (size_t)p * ntgb::warm_doubles(nr) : nullptr, wk,
                                     S.B + (size_t)p * nr * nr, &nu);
    for (int i = 0; i < D.m; i++) {
        S.lam[(size_t)p * D.m + i] = 0.0;
        S.istate[(size_t)p * D.m + i] = 0;
    }
    for (int k = 0; k < 8; k++) {
        S.scal[(size_t)p * 8 + k] = 0.0;
        S.flag[(size_t)p * 8 + k] = 0;
    }
    S.scal[(size_t)p * 8] = nu;
    if (!hot) S.flag[(size_t)p * 8 + 3] = 1; /* B is the identity */
    if (rejected) {
        S.scal[(size_t)p * 8 + 3] = NAN; /* reported violation */
        return;
    }
    state[p] = 0;
    iters[p] = 0;
}

/* one warp per problem after the iteration loop: B and nu of problem p's last pass into its row of warm;
 * rows of problems rejected by k_bounds_prep are not touched */
__global__ void k_sqp_warm_store(int P, SqpArrays S, ntgb::WarmKey wk, const int *state, double *warm)
{
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= P || state[q] == NTGB_STATUS_BAD_BOUNDS) return;
    const int nr = wk.nr;
    ntgb::warm_encode(warm + (size_t)q * ntgb::warm_doubles(nr), wk, S.scal[(size_t)q * 8], S.B + (size_t)q * nr * nr,
                      (int)(threadIdx.x & 31), 32);
}

/* reduced gradient, row values and reduced row gradients of problem p into shared memory, then one
 * SQP iteration up to the search direction (ntg_sqp.cuh), then dC = N d */
__global__ void k_sqp_step(int P, ntgb_devtab T, SqpDesc D, SqpArrays S, const double *f, const double *g, const double *c,
                           const double *J, const double *lin, double *dC, double *phi0, double *dphi0, int *state, int *count)
{
    extern __shared__ double sq_smem[];
    const int p = blockIdx.x;
    if (p >= P) return;
    const int nC = D.nC, nr = D.nr, m = D.m, n_li = D.n_li, nt = (int)blockDim.x, tid = (int)threadIdx.x;
    double *dCp = dC + (size_t)p * nC;
    if (state[p] != 0) {
        for (int e = tid; e < nC; e += nt) dCp[e] = 0.0;
        if (tid == 0) dphi0[p] = 0.0, phi0[p] = 0.0;
        return;
    }
    sqp::Qp w;
    double *Bm, *Lm, *vec, *gr, *hrow;
    const size_t nd = sqp::sqp_smem_doubles(nr, m, nt);
    sqp::sqp_carve(sq_smem, reinterpret_cast<int *>(sq_smem + nd), nr, m, nt, w, Bm, Lm, vec, gr, hrow);
    const int ld = w.ld;
    const double *gp = g + (size_t)p * nC;
    for (int k = tid; k < nr; k += nt) {
        double a = 0.0;
        for (int e = 0; e < nC; e++) a += D.N[(size_t)k * nC + e] * gp[e];
        gr[k] = a;
    }
    for (int i = tid; i < m; i += nt)
        hrow[i] = i < n_li ? lin[(size_t)p * D.nclin + D.li_idx[i]] : c[(size_t)p * D.ncnln + (i - n_li)];
    /* reduced row gradients, one row per thread and step.  Nonlinear row r of the band-compact Jacobian
     * (include/ntg_b200.h): slot jk0[j] + k of output j holds the derivative with respect to coefficient
     * iC[j] + offset + k.  The band values are fetched EIGHT at a time before they are used: behind the
     * shared-memory updates the compiler cannot move a global load, and one exposed load latency per
     * slot was 14 % of the kernel. */
    const double *Jp = J + (size_t)p * T.ncnln * T.S;
    for (int i = tid; i < m; i += nt) {
        double *Ai = w.A + (size_t)i * ld;
        if (i < n_li) {
            for (int k = 0; k < nr; k++) Ai[k] = D.ArN[(size_t)i * nr + k];
            continue;
        }
        const int r = i - n_li;
        for (int k = 0; k < nr; k++) Ai[k] = 0.0;
        int kind, mm = 0, bp = 0; /* 0 initial (src/colloc.c:254: columns from iC_j), 1 trajectory, 2 final */
        if (r < T.nnlic) kind = 0;
        else if (r < T.nnlic + T.nnltc * T.nbps) {
            kind = 1;
            mm = (r - T.nnlic) / T.nbps;
            bp = (r - T.nnlic) - mm * T.nbps;
        } else {
            kind = 2;
            bp = T.nbps - 1;
        }
        for (int j = 0; j < T.nout; j++) {
            const int ord = T.order[j], s0 = T.jk0[j];
            const int col0 = T.iC[j] + (kind == 0 ? 0 : T.off[j][bp]);
            const double *Jr;
            size_t stride;
            if (kind == 1) {
                const int t = bp / T.band_tile;
                Jr = Jp + ntgb_band_index(T.nnlic, T.nnltc, T.S, T.nbps, T.band_tile, mm, s0, bp);
                stride = (size_t)(T.nbps - t * T.band_tile < T.band_tile ? T.nbps - t * T.band_tile : T.band_tile);
            } else {
                Jr = Jp + (size_t)r * T.S + s0;
                stride = 1;
            }
            for (int k0 = 0; k0 < ord; k0 += 8) {
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; u++) v[u] = k0 + u < ord ? __ldg(Jr + (size_t)(k0 + u) * stride) : 0.0;
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    if (v[u] == 0.0) continue;
                    const double *Nc = D.N + (col0 + k0 + u);
                    for (int q = 0; q < nr; q++) Ai[q] += v[u] * Nc[(size_t)q * nC];
                }
            }
        }
    }
    __syncthreads();
    const sqp::Coop cg{tid, nt, tid & 31, nt < 32 ? nt : 32};
    const sqp::StepState st{S.y + (size_t)p * nr, S.B + (size_t)p * nr * nr, S.lam + (size_t)p * m, S.sprev + (size_t)p * nr,
                            S.grLold + (size_t)p * nr, S.grold + (size_t)p * nr, S.d + (size_t)p * nr, S.scal + (size_t)p * 8, S.flag + (size_t)p * 8,
                            S.istate + (size_t)p * m};
    const sqp::StepOpts so{D.gtol, D.ctol, D.rho_pen};
    sqp::sqp_step(cg, w, st, so, f[p], gr, hrow, D.hl + (size_t)p * D.hstride, D.hu + (size_t)p * D.hstride, Bm, Lm, vec);
    __syncthreads();
    const int status = st.flag[5];
    if (status != 0) {
        for (int e = tid; e < nC; e += nt) dCp[e] = 0.0;
        if (tid == 0) {
            state[p] = status;
            atomicAdd(count, 1);
            phi0[p] = st.scal[1];
            dphi0[p] = 0.0;
        }
        return;
    }
    for (int e = tid; e < nC; e += nt) {
        double a = 0.0;
        for (int k = 0; k < nr; k++) a += D.N[(size_t)k * nC + e] * w.x[k];
        dCp[e] = a;
    }
    if (tid == 0) {
        phi0[p] = st.scal[1];
        dphi0[p] = st.scal[2];
    }
}

/* L1 merit of trial point q (one warp each): f + nu * sum of the rows' bound violations */
__global__ void k_sqp_merit(int Q, int nalpha, SqpDesc D, const double *scal, const double *f, const double *c,
                            const double *lin, double *res, const int *pidx)
{
    const int q = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= Q) return;
    const int p = pidx != nullptr ? pidx[q / nalpha] : q / nalpha;
    const double *hl = D.hl + (size_t)p * D.hstride, *hu = D.hu + (size_t)p * D.hstride;
    double acc = 0.0;
    for (int i = lane; i < D.m; i += 32) {
        const double h = i < D.n_li ? lin[(size_t)q * D.nclin + D.li_idx[i]] : c[(size_t)q * D.ncnln + (i - D.n_li)];
        const double lo = hl[i], hi = hu[i];
        double v = 0.0;
        if (lo > -sqp::kBig && lo - h > v) v = lo - h;
        if (hi < sqp::kBig && h - hi > v) v = h - hi;
        acc += v;
    }
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) res[2 * (size_t)q] = f[q] + scal[(size_t)p * 8] * acc;
}

/* accept the step (y, C, s = alpha d) or ask for a restart from B = I; give up when that fails too */
__global__ void k_sqp_update(int P, SqpDesc D, SqpArrays S, const double *Cpart, const double *phi0, const double *alpha_best,
                             const double *phi_best, double *C, int *state, int *iters, int *count)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P || state[p] != 0) return;
    const int nC = D.nC, nr = D.nr;
    int *flag = S.flag + (size_t)p * 8;
    Cpart += (size_t)p * D.Cstride;
    iters[p] += 1;
    if (!(phi_best[p] < phi0[p])) {
        if (flag[3]) {
            state[p] = 2;
            atomicAdd(count, 1);
        } else {
            flag[2] = 1;
            flag[0] = 0;
        }
        return;
    }
    const double a = alpha_best[p];
    double *y = S.y + (size_t)p * nr, *sp = S.sprev + (size_t)p * nr;
    const double *d = S.d + (size_t)p * nr;
    for (int k = 0; k < nr; k++) {
        sp[k] = a * d[k];
        y[k] += sp[k];
    }
    double *Cp = C + (size_t)p * nC;
    for (int e = 0; e < nC; e++) {
        double v = Cpart[e];
        for (int k = 0; k < nr; k++) v += D.N[(size_t)k * nC + e] * y[k];
        Cp[e] = v;
    }
    flag[0] = 1;
    flag[1] = flag[4];
}

/* NPSOL-order outputs: clambda / istate over [linear rows ; nonlinear rows].  The multipliers of the
 * eliminated equality rows are the least-squares solution of Ae' le = g - A_in' l_in - J' l_nl
 * (W = (Ae Ae')^-1 Ae, host-built); gL is that right-hand side in the full space (k_alm_grad). */
__global__ void k_sqp_outputs(int P, SqpDesc D, SqpArrays S, int me, const int *eq_idx, const double *W, const double *gL,
                              const int *state, double *lambda, int *istate)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int ntot = D.nclin + D.ncnln;
    if (state[p] == NTGB_STATUS_BAD_BOUNDS) { /* rejected by k_bounds_prep: no multipliers, no active set */
        for (int i = 0; i < ntot; i++) {
            if (lambda != nullptr) lambda[(size_t)p * ntot + i] = 0.0;
            if (istate != nullptr) istate[(size_t)p * ntot + i] = 0;
        }
        return;
    }
    if (lambda != nullptr) {
        double *lp = lambda + (size_t)p * ntot;
        for (int i = 0; i < D.m; i++) lp[i < D.n_li ? D.li_idx[i] : D.nclin + (i - D.n_li)] = S.lam[(size_t)p * D.m + i];
        for (int r = 0; r < me; r++) {
            double a = 0.0;
            for (int e = 0; e < D.nC; e++) a += W[(size_t)r * D.nC + e] * gL[(size_t)p * D.nC + e];
            lp[eq_idx[r]] = a;
        }
    }
    if (istate != nullptr) {
        int *ip = istate + (size_t)p * ntot;
        for (int i = 0; i < D.m; i++) ip[i < D.n_li ? D.li_idx[i] : D.nclin + (i - D.n_li)] = S.istate[(size_t)p * D.m + i];
        for (int r = 0; r < me; r++) ip[eq_idx[r]] = 3;
    }
}

/* ---- per-problem bounds (ntgb_solve_eq_bounds / ntgb_solve_sqp_bounds) ----------------------------- */
struct BoundsDesc {
    ntgb::BoundsLayout L;
    int nC, n_li, m, me;
    const int *li_idx;  /* [n_li] linear rows kept as general rows */
    const int *eq_idx;  /* [me] eliminated linear rows, nullptr: row r */
    const double *M;    /* [nC][me] Cpart = M be */
    const double *Ae;   /* [me][nC] eliminated rows */
};

/* one warp per problem, once per call: problem p's compact bounds -> hl / hu [m] (SQP order), be [me],
 * Cpart = M be, and the checks of ntg_bounds.h; a rejected problem gets status 5 and counts as finished */
__global__ void k_bounds_prep(int P, BoundsDesc B, const double *lowerb, const double *upperb, double *hl, double *hu,
                              double *be, double *Cpart, int *state, int *iters, int *count)
{
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= P) return;
    const int nb = B.L.nb();
    const double *lo = lowerb + (size_t)q * nb, *up = upperb + (size_t)q * nb;
    double *bep = be + (size_t)q * B.me, *Cp = Cpart + (size_t)q * B.nC;
    unsigned bad = ntgb::bounds_expand(B.L, lo, up, B.li_idx, B.n_li, B.eq_idx, B.me, hl + (size_t)q * B.m,
                                       hu + (size_t)q * B.m, bep, lane, 32);
    __syncwarp();
    for (int e = lane; e < B.nC; e += 32) Cp[e] = ntgb::bounds_cpart(B.M, B.me, bep, e);
    __syncwarp();
    double res = 0.0, bmax = 0.0;
    for (int r = lane; r < B.me; r += 32) {
        res = ntgb::bounds_max(res, fabs(ntgb::bounds_residual(B.Ae + (size_t)r * B.nC, B.nC, Cp, bep[r])));
        bmax = fmax(bmax, fabs(bep[r]));
    }
    for (int d = 16; d > 0; d >>= 1) {
        bad |= __shfl_xor_sync(0xffffffffu, bad, d);
        res = ntgb::bounds_max(res, __shfl_xor_sync(0xffffffffu, res, d));
        bmax = fmax(bmax, __shfl_xor_sync(0xffffffffu, bmax, d));
    }
    if (ntgb::bounds_inconsistent(res, bmax)) bad |= ntgb::kBoundsInconsistent;
    if (lane == 0) {
        state[q] = bad ? NTGB_STATUS_BAD_BOUNDS : 0;
        iters[q] = 0;
        if (bad) atomicAdd(count, 1);
    }
}

/* what k_bounds_prep writes: problem p's Cpart / hl / hu at Cpart + p*nC, hl + p*m, hu + p*m */
struct BoundsArrays {
    double *Cpart, *hl, *hu, *be;

    void take(Carve &c, size_t P, const BoundsDesc &B)
    {
        c.take(P * B.nC, Cpart);
        c.take(P * B.m, hl, hu);
        c.take(P * B.me, be);
    }
};

/* per-problem bounds, once per call: k_bounds_prep into the caller's arrays */
int bounds_prepare(int P, const double *lowerb, const double *upperb, const BoundsDesc &B, const BoundsArrays &ba,
                   cudaStream_t st, int *state, int *iters, int *count)
{
    const long long threads = (long long)P * 32;
    CUDA_TRY(launch(k_bounds_prep, (unsigned)((threads + 127) / 128), 128, st, P, B, lowerb, upperb, ba.hl, ba.hu, ba.be,
                    ba.Cpart, state, iters, count));
    return 0;
}

ntgb::BoundsLayout bounds_layout(const ntgb_problem *pb)
{
    return ntgb::BoundsLayout{pb->nlic, pb->nltc, pb->nlfc, pb->nnlic, pb->nnltc, pb->nnlfc, pb->dims.nbps};
}

/* ---- two-stage Armijo search of ntgb_solve_nlp and ntgb_solve_sqp ------------------------------------------
 * the steps 1 .. 1/8 for every problem in one evaluation; the steps 2^-4 .. 2^-15 only for the problems that
 * found no Armijo step among them (compacted by index), in a second one */
constexpr int kN1 = 4, kN2 = 12, kNalpha = kN1 + kN2;

struct TwoStage {
    double *alphas;                 /* [kNalpha] 2^-a */
    double *Ct, *ft, *ct, *lint;    /* trial points and what is evaluated there, up to Q = P*kNalpha of them */
    double *res;                    /* [Q][2]: the merit at trial q in res[2q] */
    int *idx, *nidx;                /* [P] problems of the second stage, and their number */
    double *ab, *pbest;             /* [P] chosen step and its merit */

    /* the evaluator counts trial points in int */
    static int check_size(int P)
    {
        return (size_t)P * kNalpha > 0x7fffffffull ? fail(NTGB_EINVAL, "P*nalpha too large") : 0;
    }
    void take(Carve &c, size_t P, const ntgb_dims &dm)
    {
        const size_t Q = P * kNalpha;
        c.take(kNalpha, alphas);
        c.take(Q * dm.nC, Ct);
        c.take(Q, ft);
        c.take(Q * std::max(dm.ncnln, 1), ct);
        c.take(Q * std::max(dm.nclin, 1), lint);
        c.take(2 * Q, res);
        c.take(P, idx, ab, pbest);
        c.take(1, nidx);
    }
    /* once per call; upload == false: alphas already holds the step table */
    int start(int P, cudaStream_t st, bool upload = true) const
    {
        int rc;
        if (upload && (rc = upload_halving(alphas, kNalpha, st))) return rc;
        CUDA_TRY(cudaMemsetAsync(res, 0, sizeof(double) * 2 * kNalpha * (size_t)P, st));
        return 0;
    }
};

/* the search from C along dC for P problems; merit(n, nalpha, pidx) launches the merit kernel on the n trial
 * points just evaluated, trial q belonging to problem pidx[q / nalpha] (pidx == nullptr: q / nalpha).
 * single: all kNalpha steps of every problem in one evaluation and one pick, so that the host never waits for
 * the size of the second stage.  For a running problem k_alm_pick1 over the 16 steps chooses what the two
 * stages choose: the first Armijo step in order, else the smallest merit, ties to the earlier step. */
template <class Merit>
int two_stage_search(ntgb_problem *pb, int P, const double *C, const double *dC, double c1, const double *phi0,
                     const double *dphi0, const int *state, const TwoStage &ts, cudaStream_t st, Merit merit,
                     bool single = false)
{
    const int nC = pb->dims.nC;
    ntgb_eval_args et;
    memset(&et, 0, sizeof et);
    et.C = ts.Ct; et.mode_obj = 0; et.mode_con = pb->dims.ncnln > 0 ? 0 : -1; et.f = ts.ft; et.c = ts.ct;
    et.jac_layout = NTGB_JAC_NONE; et.stream = st;
    auto trials = [&](int n, int nalpha, const double *alpha, const int *pidx) -> int {
        const unsigned grid = (unsigned)(((long long)n * nalpha * nC + 255) / 256);
        if (pidx == nullptr)
            CUDA_TRY(launch(k_ls_trial, grid, 256, st, C, dC, alpha, n, nalpha, nC, ts.Ct));
        else
            CUDA_TRY(launch(k_ls_trial_idx, grid, 256, st, C, dC, alpha, pidx, n, nalpha, nC, ts.Ct));
        et.P = n * nalpha;
        int rc;
        if ((rc = ntgb_eval(pb, &et))) return rc;
        if (pb->alm.n_li > 0 && (rc = ntgb_eval_linear(pb, et.P, ts.Ct, ts.lint, nullptr, st))) return rc;
        return merit(et.P, nalpha, pidx);
    };
    int rc;
    const int n1 = single ? kNalpha : kN1;
    if ((rc = trials(P, n1, ts.alphas, nullptr))) return rc;
    CUDA_TRY(cudaMemsetAsync(ts.nidx, 0, sizeof(int), st));
    CUDA_TRY(launch(k_alm_pick1, (unsigned)((P + 127) / 128), 128, st, ts.res, ts.alphas, P, n1, c1, phi0, dphi0, state,
                    ts.ab, ts.pbest, ts.idx, ts.nidx));
    if (single) return 0;
    int n2 = 0;
    CUDA_TRY(cudaMemcpyAsync(&n2, ts.nidx, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (n2 <= 0) return 0;
    if ((rc = trials(n2, kN2, ts.alphas + kN1, ts.idx))) return rc;
    CUDA_TRY(launch(k_alm_pick2, (unsigned)((n2 + 127) / 128), 128, st, ts.res, ts.alphas + kN1, ts.idx, n2, kN2, c1, phi0,
                    dphi0, ts.ab, ts.pbest));
    return 0;
}

/* arrays of ntgb_linesearch for n = P*nalpha trial points */
struct LsArrays {
    double *Ct, *res, *lv; /* trial coefficients, result table, linear violation */

    void take(Carve &c, size_t n, int nC)
    {
        c.take(n * nC, Ct);
        c.take(n * 2, res);
        c.take(n, lv);
    }
};

/* body of ntgb_linesearch, on the caller's arrays */
int linesearch_run(ntgb_problem *pb, int P, const double *C, const double *dC, int nalpha, const double *alpha, double mu,
                   double c1, const double *phi0, const double *dphi0, double *alpha_best, double *phi_best, double *C_new,
                   cudaStream_t st, const LsArrays &la)
{
    const ntgb_dims &d = pb->dims;
    const size_t n = (size_t)P * nalpha;
    const long long total = (long long)n * d.nC;
    CUDA_TRY(launch(k_ls_trial, (unsigned)((total + 255) / 256), 256, st, C, dC, alpha, P, nalpha, d.nC, la.Ct));
    ntgb_eval_args a;
    memset(&a, 0, sizeof a);
    a.P = (int)n; a.C = la.Ct; a.mode_obj = 0; a.mode_con = d.ncnln > 0 ? 0 : -1;
    a.result = la.res; a.jac_layout = NTGB_JAC_NONE; a.stream = st;
    int rc;
    if ((rc = ntgb_eval(pb, &a))) return rc;
    const bool lin = d.nclin > 0;
    if (lin && (rc = ntgb_eval_linear(pb, (int)n, la.Ct, nullptr, la.lv, st))) return rc;
    CUDA_TRY(launch(k_ls_pick, (unsigned)((P + 127) / 128), 128, st, la.res, lin ? la.lv : nullptr, alpha, P,
                    nalpha, mu, c1, phi0, dphi0, C, dC, d.nC, alpha_best, phi_best, C_new));
    return 0;
}

/* how a solver driver runs: Sync (ntgb_solve_eq*, ntgb_solve_sqp*), Reserve (ntgb_solve_*_reserve: the refusals,
 * the one-time host work and the work space for P problems; nothing is queued) or Async (ntgb_solve_*_async:
 * from the reserved work space, exactly max_iter iterations, no synchronization, no host copy, no allocation) */
enum class Run { Sync, Reserve, Async };

/* the Reserve step of a driver whose Async arrays are carved by layout: the step table once per problem, then
 * the work space grows to the layout of P problems (never shrinks).  Work queued on any stream may still use
 * the old work space, so the device is synchronized first. */
template <class Layout>
int reserve_work(ntgb_problem *pb, AsyncWork &w, int P, Layout layout)
{
    int rc;
    if (!pb->async.halving && ((rc = dev_alloc(pb, &pb->async.halving, kNalpha)) ||
                               (rc = upload_halving(pb->async.halving, kNalpha, nullptr))))
        return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    if ((rc = scratch_carve(w.s, nullptr, layout))) return rc;
    w.P = std::max(w.P, P);
    return 0;
}

/* the problem class of ntgb_solve_eq and ntgb_solve_eq_lbfgs (`who`): no nonlinear row, every linear row an
 * equality */
int check_eq_only(const ntgb_problem *pb, const char *who)
{
    const ntgb_dims &dm = pb->dims;
    if (dm.ncnln > 0) return fail(NTGB_EINVAL, "%s: problem has %d nonlinear constraints", who, dm.ncnln);
    for (int i = 0; i < dm.nclin; i++)
        if (pb->lin_lb[i] != pb->lin_ub[i]) return fail(NTGB_EINVAL, "%s: linear constraint %d is not an equality", who, i);
    return 0;
}

int solve_eq_impl(ntgb_problem *pb, Run run, int P, double *C, const double *lowerb, const double *upperb, double *f,
                  int *iters, int *status, const ntgb_solve_opts *opts, void *stream);
int solve_lbfgs_impl(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                     int *iters, int *status, const ntgb_lbfgs_opts &o, void *stream);
int solve_newton_impl(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                      int *iters, int *status, const ntgb_newton_opts &o, void *stream);
int newton_prepare(ntgb_problem *pb);
int solve_sqp_impl(ntgb_problem *pb, Run run, int P, double *C, const double *lowerb, const double *upperb, double *warm,
                   double *f, double *viol_out, int *iters, int *status, double *lambda, int *istate,
                   const ntgb_sqp_opts *opts, void *stream);

} /* namespace */

extern "C" {

const char *ntgb_last_error(void) { return g_err.c_str(); }
#define NTGB_STR2(x) #x
#define NTGB_STR(x) NTGB_STR2(x)
const char *ntgb_version(void) { return "ntg_b200 0.2 (sm_100a, kernel ABI " NTGB_STR(NTGB_KERNEL_ABI) ")"; }

int ntgb_register_pack(const ntgb_pack *pack)
{
    if (!pack || !pack->launch || !pack->name) return fail(NTGB_EINVAL, "ntgb_register_pack: null pack");
    /* ntgb_devtab / ntgb_eval_args travel BY VALUE into the pack's launcher: a pack built against
     * another revision of ntg_kernel_args.h would reinterpret them silently */
    if (pack->abi != NTGB_KERNEL_ABI)
        return fail(NTGB_EINVAL, "callback pack '%s' was built for kernel ABI %d, this library is ABI %d: rebuild the pack "
                    "(python -m ntg_b200.build)", pack->name, pack->abi, NTGB_KERNEL_ABI);
    std::lock_guard<std::mutex> lk(g_reg_mu);
    for (ntgb_pack &pk : registry())
        if (strcmp(pk.name, pack->name) == 0) {
            pk = *pack;
            return 0;
        }
    registry().push_back(*pack);
    return 0;
}

const ntgb_pack *ntgb_find_pack(const char *name)
{
    std::lock_guard<std::mutex> lk(g_reg_mu);
    for (const ntgb_pack &pk : registry())
        if (strcmp(pk.name, name) == 0) return &pk;
    return nullptr;
}

int ntgb_num_packs(void)
{
    std::lock_guard<std::mutex> lk(g_reg_mu);
    return (int)registry().size();
}

void ntgb_destroy(ntgb_problem *pb)
{
    if (!pb) return;
    DeviceGuard dg(pb->device);
    for (void *p : pb->allocs) cudaFree(p);
    if (pb->zc.buf) cudaFreeHost(pb->zc.buf);
    auto &s = pb->scratch;
    for (Scratch *sc : {&s.eq, &s.nlp, &s.sqp, &s.ls, &s.bnd, &s.lbfgs, &s.newton, &pb->async.eq.s, &pb->async.sqp.s})
        cudaFree(sc->p);
    for (auto &h : pb->hs) {
        double *hsp[] = {h.C, h.f, h.g, h.c, h.J, h.Z, h.result};
        for (double *p : hsp)
            if (p) cudaFree(p);
        if (h.stream) cudaStreamDestroy(h.stream);
    }
    delete pb;
}

int ntgb_create(ntgb_problem **out, const ntgb_setup *s, int device)
{
    if (!out || !s) return fail(NTGB_EINVAL, "ntgb_create: null argument");
    *out = nullptr;
    if (s->nout < 1 || s->nout > NTGB_MAXOUT)
        return fail(NTGB_EINVAL, "nout = %d outside [1,%d]", s->nout, NTGB_MAXOUT);
    if (s->nbps < 2 || !s->bps) return fail(NTGB_EINVAL, "need at least 2 breakpoints");
    if (!s->kninterv || !s->knots || !s->order || !s->mult || !s->maxderiv)
        return fail(NTGB_EINVAL, "ntgb_create: null spline description");
    for (int j = 0; j < s->nout; j++) {
        /* maxderiv <= order <= 20: PGS bsplvd/bsplvb limits (SURVEY.md Q4) */
        if (s->order[j] < 1 || s->order[j] > NTGB_MAXORDER)
            return fail(NTGB_EINVAL, "order[%d] = %d outside [1,%d]", j, s->order[j], NTGB_MAXORDER);
        if (s->maxderiv[j] < 1 || s->maxderiv[j] > s->order[j])
            return fail(NTGB_EINVAL, "maxderiv[%d] = %d outside [1,order]", j, s->maxderiv[j]);
        if (s->mult[j] < 0 || s->mult[j] >= s->order[j])
            return fail(NTGB_EINVAL, "mult[%d] = %d outside [0,order)", j, s->mult[j]);
        if (s->kninterv[j] < 1 || !s->knots[j]) return fail(NTGB_EINVAL, "output %d: bad knots", j);
        /* a breakpoint in front of the first knot is undefined in the reference (interv returns
         * left = 1 and bsplvb reads t(left+1-j) before the knot array); refuse it */
        for (int i = 0; i < s->nbps; i++)
            if (s->bps[i] < s->knots[j][0])
                return fail(NTGB_EINVAL, "breakpoint %d (%.17g) lies before the first knot of output %d (%.17g)", i,
                            s->bps[i], j, s->knots[j][0]);
    }
    int rc;
    if ((rc = check_avs(s->initialcostav, s->ninitialcostav, s, "initialcostav"))) return rc;
    if ((rc = check_avs(s->trajectorycostav, s->ntrajectorycostav, s, "trajectorycostav"))) return rc;
    if ((rc = check_avs(s->finalcostav, s->nfinalcostav, s, "finalcostav"))) return rc;
    if ((rc = check_avs(s->initialconstrav, s->ninitialconstrav, s, "initialconstrav"))) return rc;
    if ((rc = check_avs(s->trajectoryconstrav, s->ntrajectoryconstrav, s, "trajectoryconstrav"))) return rc;
    if ((rc = check_avs(s->finalconstrav, s->nfinalconstrav, s, "finalconstrav"))) return rc;

    const ntgb_pack *pk = match_pack(s);
    if (!pk)
        return fail(NTGB_ENOPACK,
                    "no registered device pack provides these callbacks (%d packs loaded): compile the "
                    "callback file with tools/ntg_pack.py and load the resulting shared object",
                    ntgb_num_packs());
    if (pk->max_nout != s->nout)
        return fail(NTGB_ELIMIT, "pack '%s' is compiled for nout = %d, problem has %d", pk->name, pk->max_nout, s->nout);
    for (int j = 0; j < s->nout; j++) {
        if (pk->maxderiv[j] != s->maxderiv[j])
            return fail(NTGB_ELIMIT, "pack '%s' is compiled for maxderiv[%d] = %d, problem has %d", pk->name, j,
                        pk->maxderiv[j], s->maxderiv[j]);
        if (s->order[j] > pk->max_order)
            return fail(NTGB_ELIMIT, "pack '%s' is compiled for order <= %d, output %d has %d", pk->name,
                        pk->max_order, j, s->order[j]);
    }
    if ((s->nnlic && s->nnlic != pk->max_nnlic) || (s->nnltc && s->nnltc != pk->max_nnltc) ||
        (s->nnlfc && s->nnlfc != pk->max_nnlfc))
        return fail(NTGB_ELIMIT, "pack '%s' is compiled for (nnlic,nnltc,nnlfc) = (%d,%d,%d), problem has (%d,%d,%d)",
                    pk->name, pk->max_nnlic, pk->max_nnltc, pk->max_nnlfc, s->nnlic, s->nnltc, s->nnlfc);

    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(NTGB_ECUDA, "no CUDA device available (%s); this library has no CPU path",
                    ce == cudaSuccess ? "device count 0" : cudaGetErrorString(ce));
    if (device < 0 || device >= ndev) return fail(NTGB_EINVAL, "device %d not in [0,%d)", device, ndev);
    DeviceGuard dg(device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", device);

    ntgb_problem *pb = new ntgb_problem();
    pb->device = device;
    pb->pack_copy = *pk;
    pb->pack = &pb->pack_copy;
    struct Cleanup {
        ntgb_problem *p;
        ~Cleanup() { if (p) ntgb_destroy(p); }
    } cleanup{pb};

    CUDA_TRY(cudaDeviceGetAttribute(&pb->sm_count, cudaDevAttrMultiProcessorCount, device));
    /* The persistent evaluators fill every SM (registers and shared memory).  When another kernel
     * must run beside them -- the NCCL all-gather of the result tables in a multi-GPU job -- a few
     * SMs left free keep it from delaying a handful of evaluator CTAs, which would finish last. */
    if (const char *e = getenv("NTG_B200_SM_RESERVE")) {
        const int r = atoi(e);
        if (r > 0 && r < pb->sm_count) pb->sm_count -= r;
    }
    CUDA_TRY(cudaDeviceGetAttribute(&pb->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));

    ntgb_devtab &T = pb->tab;
    const int nout = s->nout, nbps = s->nbps;
    T.nout = nout; T.nbps = nbps;
    T.nicf = s->nicf; T.nucf = s->nucf; T.nfcf = s->nfcf;
    T.nnlic = s->nnlic; T.nnltc = s->nnltc; T.nnlfc = s->nnlfc;
    pb->nlic = s->nlic; pb->nltc = s->nltc; pb->nlfc = s->nlfc;
    pb->nnlic = s->nnlic; pb->nnltc = s->nnltc; pb->nnlfc = s->nnlfc;
    pb->bps.assign(s->bps, s->bps + nbps);
    pb->hB_off.resize(nout);
    size_t btot = 0;
    for (int j = 0; j < nout; j++) {
        const int order = s->order[j], mult = s->mult[j], md = s->maxderiv[j], ni = s->kninterv[j];
        const int n = ni * (order - mult) + mult; /* reference src/colloc.c:67 */
        pb->order.push_back(order); pb->mult.push_back(mult); pb->maxderiv.push_back(md);
        pb->ninterv.push_back(ni); pb->ncoef.push_back(n);
        pb->knots.emplace_back(s->knots[j], s->knots[j] + ni + 1);
        T.order[j] = order; T.mult[j] = mult; T.maxderiv[j] = md; T.ncoef[j] = n;
        T.iC[j] = T.nC; T.iz[j] = T.nz; T.jk0[j] = T.S;
        T.nC += n; T.nz += md; T.S += order;
        pb->hB_off[j] = btot;
        btot += (size_t)nbps * order * md;
    }
    for (int j = 0; j < nout; j++) T.iZ[j] = T.iz[j] * nbps; /* reference src/colloc.c:43 */
    T.nZ = T.nz * nbps;
    T.ncnln = s->nnlic + s->nnltc * nbps + s->nnlfc;
    pb->dims.nout = nout; pb->dims.nbps = nbps; pb->dims.nC = T.nC; pb->dims.nz = T.nz; pb->dims.nZ = T.nZ;
    pb->dims.nclin = s->nlic + s->nltc * nbps + s->nlfc;
    pb->dims.ncnln = T.ncnln; pb->dims.sorder = T.S; pb->dims.device = device;

    /* active-variable masks: updateZ is only called for kinds whose count != 0
     * (reference src/ntg.c:287-292, :348-353) */
    if (s->nicf != 0) add_mask(T.avmask, s->initialcostav, s->ninitialcostav, 1);
    if (s->nucf != 0) add_mask(T.avmask, s->trajectorycostav, s->ntrajectorycostav, 0);
    if (s->nfcf != 0) add_mask(T.avmask, s->finalcostav, s->nfinalcostav, 2);
    if (s->nnlic != 0) add_mask(T.avmask, s->initialconstrav, s->ninitialconstrav, 1);
    if (s->nnltc != 0) add_mask(T.avmask, s->trajectoryconstrav, s->ntrajectoryconstrav, 0);
    if (s->nnlfc != 0) add_mask(T.avmask, s->finalconstrav, s->nfinalconstrav, 2);
    {
        const int ncost[3] = {s->nicf, s->nucf, s->nfcf}, nav[3] = {s->ninitialcostav, s->ntrajectorycostav, s->nfinalcostav};
        const AV *av[3] = {s->initialcostav, s->trajectorycostav, s->finalcostav};
        for (int k = 0; k < 3; k++)
            if (ncost[k] != 0)
                for (int i = 0; i < nav[k]; i++) pb->cost_out[k] |= 1u << av[k][i].output;
    }

    /* ---- K0: tables on the device ---- */
    double *dbps = nullptr;
    if ((rc = dev_upload(pb, &dbps, pb->bps.data(), (size_t)nbps))) return rc;
    T.bps = dbps;
    pb->hB.resize(btot);
    pb->hoff.resize((size_t)nout * nbps);
    pb->hleft.resize((size_t)nout * nbps);
    pb->augknots.resize(nout);
    for (int j = 0; j < nout; j++) {
        const int order = T.order[j], mult = T.mult[j], md = T.maxderiv[j], ni = pb->ninterv[j];
        const int naug = T.ncoef[j] + order;
        double *dk = nullptr, *daug = nullptr, *dBn = nullptr, *dBt = nullptr;
        int *doff = nullptr, *dleft = nullptr;
        if ((rc = dev_upload(pb, &dk, pb->knots[j].data(), (size_t)ni + 1))) return rc;
        if ((rc = dev_alloc(pb, &daug, (size_t)naug))) return rc;
        if ((rc = dev_alloc(pb, &dBn, (size_t)nbps * order * md))) return rc;
        if ((rc = dev_alloc(pb, &dBt, (size_t)nbps * order * md))) return rc;
        if ((rc = dev_alloc(pb, &doff, (size_t)nbps))) return rc;
        if ((rc = dev_alloc(pb, &dleft, (size_t)nbps))) return rc;
        CUDA_TRY(launch(k0_augknots, (naug + 127) / 128, 128, nullptr, dk, ni, order, mult, daug, naug));
        CUDA_TRY(launch(k0_tables, (nbps + 63) / 64, 64, nullptr, daug, naug, dk, ni + 1, dbps, nbps, order, mult, md,
                        dBn, dBt, doff, dleft));
        T.Bn[j] = dBn; T.Bt[j] = dBt; T.off[j] = doff;
        pb->daug[j] = daug; pb->dknots[j] = dk;
        pb->augknots[j].resize(naug);
        CUDA_TRY(cudaMemcpy(pb->augknots[j].data(), daug, sizeof(double) * naug, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(pb->hB.data() + pb->hB_off[j], dBn, sizeof(double) * (size_t)nbps * order * md,
                            cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(pb->hoff.data() + (size_t)j * nbps, doff, sizeof(int) * nbps, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(pb->hleft.data() + (size_t)j * nbps, dleft, sizeof(int) * nbps, cudaMemcpyDeviceToHost));
        for (int bp = 0; bp < nbps; bp++) {
            const int o = pb->hoff[(size_t)j * nbps + bp];
            if (o < 0 || o + order > T.ncoef[j])
                return fail(NTGB_EINVAL, "output %d breakpoint %d: coefficient window [%d,%d) outside [0,%d)", j, bp, o,
                            o + order, T.ncoef[j]);
        }
    }

    /* column support for the gradient gather: first/last breakpoint whose band holds column c */
    {
        std::vector<int> lo(T.nC, nbps), hi(T.nC, -1);
        for (int j = 0; j < nout; j++)
            for (int bp = 0; bp < nbps; bp++) {
                const int o = pb->hoff[(size_t)j * nbps + bp];
                for (int k = 0; k < T.order[j]; k++) {
                    const int c = T.iC[j] + o + k;
                    if (bp < lo[c]) lo[c] = bp;
                    if (bp > hi[c]) hi[c] = bp;
                }
            }
        int *dlo = nullptr, *dhi = nullptr;
        if ((rc = dev_upload(pb, &dlo, lo.data(), (size_t)T.nC))) return rc;
        if ((rc = dev_upload(pb, &dhi, hi.data(), (size_t)T.nC))) return rc;
        T.col_lo = dlo; T.col_hi = dhi;
        /* runs of equal offset per output, and the run each column's gather starts in */
        std::vector<int> seg0(T.nC, 0);
        std::vector<std::vector<int>> runs_st((size_t)nout), runs_so((size_t)nout);
        for (int j = 0; j < nout; j++) {
            std::vector<int> &st = runs_st[j], &so = runs_so[j];
            for (int bp = 0; bp < nbps; bp++) {
                const int o = pb->hoff[(size_t)j * nbps + bp];
                if (bp == 0 || o != so.back()) { st.push_back(bp); so.push_back(o); }
            }
            T.nseg[j] = (int)so.size();
            st.push_back(nbps);
            so.push_back(0);
            int *dst = nullptr, *dso = nullptr;
            if ((rc = dev_upload(pb, &dst, st.data(), st.size()))) return rc;
            if ((rc = dev_upload(pb, &dso, so.data(), so.size()))) return rc;
            T.seg_start[j] = dst; T.seg_off[j] = dso;
            for (int cl = 0; cl < T.ncoef[j]; cl++) {
                const int c = T.iC[j] + cl;
                const int i0 = lo[c] > 0 ? lo[c] - 1 : 0;
                int sidx = 0;
                while (sidx + 1 < T.nseg[j] && st[sidx + 1] <= i0) sidx++;
                seg0[c] = sidx;
            }
        }
        int *dseg0 = nullptr;
        if ((rc = dev_upload(pb, &dseg0, seg0.data(), (size_t)T.nC))) return rc;
        T.col_seg0 = dseg0;

        /* K1s quadrature schedule (ntg_kernel_args.h): longest-chain-first packing of the nC+1
         * chains into NS slots, one table per NS = 1 .. sched_maxns (a 256-thread CTA whose largest
         * tile has n problems runs NS = min(256 / n, sched_maxns) slots of n lanes) */
        T.sched_maxns = 0;
        T.sched = nullptr;
        T.img_w = nullptr;
        T.img_i = nullptr;
        if (nbps <= NTGB_SCHED_BLOCK) {
            const int ncol = T.nC + 1, stride = NTGB_SCHED_BLOCK + 1 + ncol;
            const int maxns = ncol < NTGB_SCHED_MAXNS ? ncol : NTGB_SCHED_MAXNS;
            std::vector<int> len((size_t)ncol), order((size_t)ncol);
            for (int c = 0; c < T.nC; c++) {
                const int i0 = lo[c] > 0 ? lo[c] - 1 : 0;
                const int nend = (hi[c] < nbps - 2 ? hi[c] : nbps - 2) + 1;
                len[c] = nend > i0 ? nend - i0 : 0;
            }
            len[T.nC] = nbps - 1;
            for (int c = 0; c < ncol; c++) order[c] = c;
            std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return len[a] > len[b]; });
            std::vector<int> sched((size_t)maxns * stride, 0);
            for (int NS = 1; NS <= maxns; NS++) {
                std::vector<long long> load((size_t)NS, 0);
                std::vector<std::vector<int>> lists((size_t)NS);
                for (int c : order) {
                    int best = 0;
                    for (int q = 1; q < NS; q++)
                        if (load[q] < load[best]) best = q;
                    load[best] += len[c] + 4; /* + a fixed cost per chain */
                    lists[best].push_back(c);
                }
                int *st = &sched[(size_t)(NS - 1) * stride], *cols = st + NTGB_SCHED_BLOCK + 1, pos = 0;
                for (int q = 0; q < NS; q++) {
                    st[q] = pos;
                    for (int c : lists[q]) cols[pos++] = c;
                }
                for (int q = NS; q <= NTGB_SCHED_BLOCK; q++) st[q] = pos;
            }
            int *dsched = nullptr;
            if ((rc = dev_upload(pb, &dsched, sched.data(), sched.size()))) return rc;
            T.sched = dsched;
            T.sched_maxns = maxns;

            /* K1s steady-state image (ntg_kernel_args.h): what the kernel's prologue would build for
             * funobj mode 2 + funcon mode 2, in the layout of its shared memory (ntg_eval_small.cuh:
             * SmallSmem::pitch, the weights, the run tables, the chain description per column) */
            int pitch = (nbps + 1) & ~1;
            if (((pitch >> 1) & 1) == 0) pitch += 2;
            std::vector<double> imgw((size_t)2 * (pitch + 2), 0.0);
            for (int n = 0; n < pitch + 2; n++) {
                const double *b = pb->bps.data();
                const double lo_w = (n >= 1 && n < nbps) ? (b[n] - b[n - 1]) * 0.5 : 0.0;
                const double hi_w = (n + 1 < nbps) ? (b[n + 1] - b[n]) * 0.5 : 0.0;
                imgw[n] = (n >= 1 && n < nbps) ? b[n] - b[n - 1] : 0.0;
                imgw[(size_t)pitch + 2 + n] = lo_w + hi_w;
            }
            int segtot = 0;
            for (int j = 0; j < nout; j++) segtot += T.nseg[j] + 1;
            const int par0 = 2 * segtot + 4;
            std::vector<int> imgi((size_t)par0 + (size_t)ncol * 9, 0);
            {
                int base = 0;
                for (int j = 0; j < nout; j++) {
                    for (int i = 0; i <= T.nseg[j]; i++) {
                        imgi[(size_t)base + i] = runs_st[j][i];
                        imgi[(size_t)segtot + base + i] = runs_so[j][i];
                    }
                    base += T.nseg[j] + 1;
                }
            }
            imgi[(size_t)2 * segtot + 0] = 0;
            imgi[(size_t)2 * segtot + 1] = nbps;
            imgi[(size_t)2 * segtot + 2] = 0;
            const bool doI = T.nicf != 0, doU = T.nucf != 0, doF = T.nfcf != 0;
            for (int c = 0; c <= T.nC; c++) {
                int *pp = &imgi[(size_t)par0 + (size_t)c * 9];
                if (c == T.nC) {
                    pp[1] = doU ? nbps - 1 : 0;
                    pp[3] = 2 * segtot;
                    pp[8] = 2 * segtot + 2;
                    pp[4] = T.S * pitch; /* x (problems per tile) in the kernel: f_s follows D_s */
                    pp[5] = 1;
                    continue;
                }
                int sb = 0;
                for (int j = 0; j < nout; j++) {
                    const int clj = c - T.iC[j];
                    if (clj >= 0 && clj < T.ncoef[j]) {
                        const int ord = T.order[j];
                        if (doU) {
                            pp[0] = lo[c] > 0 ? lo[c] - 1 : 0;
                            pp[1] = (hi[c] < nbps - 2 ? hi[c] : nbps - 2) + 1;
                            pp[2] = seg0[c];
                        }
                        pp[3] = sb;
                        pp[8] = segtot + sb;
                        pp[4] = T.jk0[j] * pitch;
                        pp[5] = ord;
                        pp[6] = clj;
                        int iDI = 0, iDF = 0;
                        if (doI && clj < ord) iDI = T.jk0[j] + clj + 1;
                        if (doF) {
                            const int k = clj - runs_so[j][(size_t)T.nseg[j] - 1];
                            if (k >= 0 && k < ord) iDF = T.jk0[j] + k + 1;
                        }
                        pp[7] = iDI | (iDF << 16);
                    }
                    sb += T.nseg[j] + 1;
                }
            }
            double *dimgw = nullptr;
            int *dimgi = nullptr;
            if ((rc = dev_upload(pb, &dimgw, imgw.data(), imgw.size()))) return rc;
            if ((rc = dev_upload(pb, &dimgi, imgi.data(), imgi.size()))) return rc;
            T.img_w = dimgw;
            T.img_i = dimgi;
        }

    }

    /* do all outputs share one spline setup (one table serves all)? */
    T.one_table = 1;
    for (int j = 1; j < nout; j++)
        if (T.order[j] != T.order[0] || T.mult[j] != T.mult[0] || T.maxderiv[j] != T.maxderiv[0] ||
            pb->ninterv[j] != pb->ninterv[0] || pb->knots[j] != pb->knots[0])
            T.one_table = 0;

    /* quadrature plans for the cluster kernels (long horizons, one shared table) */
    T.plan_ptr = nullptr; T.plan = nullptr; T.plan_cl = 0; T.plan_bpc = 0; T.plan_cwin = 0; T.plan_n = 0;
    T.band_tile = nbps; /* band-compact Jacobian: one tile unless a cluster splits the horizon */
    T.plan_halo = -1;
    T.plan_share = 0;
    if (T.one_table && nbps > 256 && nbps <= 8 * 224) {
        const int ncoef0 = T.ncoef[0], ord0 = T.order[0];
        /* support of every local column, in breakpoints */
        std::vector<int> clo(ncoef0, nbps), chi(ncoef0, -1);
        int hsup = 0;
        for (int cl = 0; cl < ncoef0; cl++) {
            for (int bp = 0; bp < nbps; bp++) {
                const int k = cl - pb->hoff[bp];
                if (k >= 0 && k < ord0) { if (bp < clo[cl]) clo[cl] = bp; if (bp > chi[cl]) chi[cl] = bp; }
            }
            if (chi[cl] >= 0 && chi[cl] - clo[cl] > hsup) hsup = chi[cl] - clo[cl];
        }
        /* room for the halo breakpoints of K1c/H among the 224 breakpoint-threads of a CTA */
        int per_cta = 224 - 2 * hsup;
        if (per_cta < 64) per_cta = 224;
        int CL, bpc;
        ntgb_cluster_geometry(nbps, per_cta, &CL, &bpc);
        if ((long long)CL * bpc < nbps || bpc > 224) return fail(NTGB_ELIMIT, "internal: cluster geometry");
        T.band_tile = bpc; /* one tile per CTA of the cluster: each CTA streams one contiguous block */
        std::vector<int> ptr(ncoef0 + 1, 0);
        std::vector<int2> ent;
        for (int cl = 0; cl < ncoef0; cl++) {
            ptr[cl] = (int)ent.size();
            if (chi[cl] >= 0) {
                const int i0 = clo[cl] > 0 ? clo[cl] - 1 : 0;
                const int nend = (chi[cl] < nbps - 2 ? chi[cl] : nbps - 2) + 1;
                for (int n = i0; n <= nend; n++) {
                    const int k = cl - pb->hoff[n];
                    const int r = n / bpc, li = n - r * bpc;
                    const int o24 = (k >= 0 && k < ord0) ? k * bpc + li : 0xffffff;
                    ent.push_back(make_int2(n, (r << 24) | o24));
                }
            }
        }
        ptr[ncoef0] = (int)ent.size();
        if (ent.empty()) ent.push_back(make_int2(0, 0));
        const int plan_n = (int)ent.size();
        /* second plan (K1c/H, ntg_kernel_args.h): column cl belongs to rank own(cl) alone */
        auto own = [&](int cl) {
            int r = 0;
            while (r + 1 < CL && cl >= (int)(((long long)ncoef0 * (r + 1)) / CL)) r++;
            return r;
        };
        int halo = 0;
        for (int cl = 0; cl < ncoef0; cl++)
            if (chi[cl] >= 0) {
                const int r = own(cl), first = r * bpc, last = (first + bpc < nbps ? first + bpc : nbps) - 1;
                if (first - clo[cl] > halo) halo = first - clo[cl];
                if (chi[cl] - last > halo) halo = chi[cl] - last;
            }
        bool hot_ok = bpc + 2 * halo <= 224 && ncoef0 / CL >= ord0;
        const bool fast_pack = pb->pack_copy.exact == 0;
        std::vector<int> hptr(ncoef0 + 1, 0);
        std::vector<int2> hent;
        if (hot_ok) {
            const int pitch = bpc + 2 * halo;
            for (int cl = 0; cl < ncoef0; cl++) {
                hptr[cl] = plan_n + (int)hent.size();
                if (chi[cl] < 0) continue;
                const int r = own(cl);
                const int i0 = clo[cl] > 0 ? clo[cl] - 1 : 0;
                const int nend = (chi[cl] < nbps - 2 ? chi[cl] : nbps - 2) + 1;
                for (int n = i0; n <= nend; n++) {
                    const int k = cl - pb->hoff[n];
                    const bool in = k >= 0 && k < ord0;
                    if (!in && fast_pack) continue; /* node-weight quadrature: in-band terms only */
                    hent.push_back(make_int2(n, in ? k * pitch + (n - r * bpc + halo) : -1));
                }
            }
            hptr[ncoef0] = plan_n + (int)hent.size();
            T.plan_share = 0;
            for (int r = 0; r < CL; r++) {
                const int a = (int)(((long long)ncoef0 * r) / CL), b = (int)(((long long)ncoef0 * (r + 1)) / CL);
                if (hptr[b] - hptr[a] > T.plan_share) T.plan_share = hptr[b] - hptr[a];
            }
            ptr.insert(ptr.end(), hptr.begin(), hptr.end());
            ent.insert(ent.end(), hent.begin(), hent.end());
            T.plan_halo = halo;
        }
        int *dptr = nullptr; int2 *dent = nullptr;
        if ((rc = dev_upload(pb, &dptr, ptr.data(), ptr.size()))) return rc;
        if ((rc = dev_upload(pb, &dent, ent.data(), ent.size()))) return rc;
        T.plan_ptr = dptr; T.plan = dent; T.plan_cl = CL; T.plan_bpc = bpc;
        const int hw = T.plan_halo > 0 ? T.plan_halo : 0;
        int wmax = 0;
        for (int r = 0; r < CL; r++) { /* coefficient window of rank r's breakpoints (+ halo) */
            int lo = 0x7fffffff, hi = -1;
            for (int bp = r * bpc - hw; bp < (r + 1) * bpc + hw; bp++) {
                if (bp < 0 || bp >= nbps) continue;
                lo = pb->hoff[bp] < lo ? pb->hoff[bp] : lo;
                hi = pb->hoff[bp] > hi ? pb->hoff[bp] : hi;
            }
            if (hi >= 0 && hi + ord0 - lo > wmax) wmax = hi + ord0 - lo;
        }
        T.plan_cwin = wmax * nout;
        T.plan_n = plan_n;
    }

    /* Jacobian row pattern (reference src/colloc.c:243-316) */
    pb->col0.resize((size_t)(T.ncnln > 0 ? T.ncnln : 1) * nout);
    {
        int row = 0;
        for (int r = 0; r < s->nnlic; r++, row++)
            for (int j = 0; j < nout; j++) pb->col0[(size_t)row * nout + j] = T.iC[j];
        for (int m = 0; m < s->nnltc; m++)
            for (int bp = 0; bp < nbps; bp++, row++)
                for (int j = 0; j < nout; j++)
                    pb->col0[(size_t)row * nout + j] = T.iC[j] + pb->hoff[(size_t)j * nbps + bp];
        for (int r = 0; r < s->nnlfc; r++, row++)
            for (int j = 0; j < nout; j++)
                pb->col0[(size_t)row * nout + j] = T.iC[j] + pb->hoff[(size_t)j * nbps + nbps - 1];
    }

    /* bounds (compact), nonlinear part on the device for the violation epilogue */
    const int nlin_b = s->nlic + s->nltc + s->nlfc, nnl_b = s->nnlic + s->nnltc + s->nnlfc;
    pb->lowerb.assign((size_t)nlin_b + nnl_b, -DBL_MAX);
    pb->upperb.assign((size_t)nlin_b + nnl_b, DBL_MAX);
    if (s->lowerb) pb->lowerb.assign(s->lowerb, s->lowerb + nlin_b + nnl_b);
    if (s->upperb) pb->upperb.assign(s->upperb, s->upperb + nlin_b + nnl_b);
    {
        double *dlb = nullptr, *dub = nullptr;
        if ((rc = dev_upload(pb, &dlb, pb->lowerb.data() + nlin_b, (size_t)nnl_b))) return rc;
        if ((rc = dev_upload(pb, &dub, pb->upperb.data() + nlin_b, (size_t)nnl_b))) return rc;
        T.nl_lb = dlb; T.nl_ub = dub;
        T.nl_inline = nnl_b <= NTGB_MAXNLB;
        for (int i = 0; i < NTGB_MAXNLB; i++) {
            T.nl_lb_v[i] = (T.nl_inline && i < nnl_b) ? pb->lowerb[(size_t)nlin_b + i] : -DBL_MAX;
            T.nl_ub_v[i] = (T.nl_inline && i < nnl_b) ? pb->upperb[(size_t)nlin_b + i] : DBL_MAX;
        }
    }

    /* linear constraints: A (NPSOL layout, host) and band form (device) */
    auto copy_rows = [&](std::vector<double> &dst, const double *const *src, int n) {
        dst.assign((size_t)n * T.nz, 0.0);
        for (int r = 0; r < n; r++)
            for (int q = 0; q < T.nz; q++) dst[(size_t)r * T.nz + q] = src[r][q];
    };
    if (s->nlic) { if (!s->lic) return fail(NTGB_EINVAL, "nlic > 0 but lic == NULL"); copy_rows(pb->lic, s->lic, s->nlic); }
    if (s->nltc) { if (!s->ltc) return fail(NTGB_EINVAL, "nltc > 0 but ltc == NULL"); copy_rows(pb->ltc, s->ltc, s->nltc); }
    if (s->nlfc) { if (!s->lfc) return fail(NTGB_EINVAL, "nlfc > 0 but lfc == NULL"); copy_rows(pb->lfc, s->lfc, s->nlfc); }
    const int nclin = pb->dims.nclin;
    if (nclin > 0) {
        std::vector<double> band((size_t)nclin * T.S, 0.0), llb(nclin), lub(nclin);
        std::vector<int> acol0((size_t)nclin * nout);
        pb->A.assign((size_t)nclin * T.nC, 0.0);
        int row = 0, bsrc = 0;
        auto put = [&](const double *dz, int bp, bool initial, double lbv, double ubv) {
            double *b = band.data() + (size_t)row * T.S;
            host_band_row(pb, dz, bp, b);
            for (int j = 0; j < nout; j++) {
                const int c0 = T.iC[j] + (initial ? 0 : pb->hoff[(size_t)j * nbps + bp]);
                acol0[(size_t)row * nout + j] = c0;
                for (int k = 0; k < T.order[j]; k++) pb->A[(size_t)(c0 + k) * nclin + row] = b[T.jk0[j] + k];
            }
            llb[row] = lbv; lub[row] = ubv;
            row++;
        };
        for (int r = 0; r < s->nlic; r++, bsrc++) put(&pb->lic[(size_t)r * T.nz], 0, true, pb->lowerb[bsrc], pb->upperb[bsrc]);
        for (int r = 0; r < s->nltc; r++, bsrc++)
            for (int bp = 0; bp < nbps; bp++) put(&pb->ltc[(size_t)r * T.nz], bp, false, pb->lowerb[bsrc], pb->upperb[bsrc]);
        for (int r = 0; r < s->nlfc; r++, bsrc++) put(&pb->lfc[(size_t)r * T.nz], nbps - 1, false, pb->lowerb[bsrc], pb->upperb[bsrc]);
        if ((rc = dev_upload(pb, &pb->dAband, band.data(), band.size()))) return rc;
        if ((rc = dev_upload(pb, &pb->dAcol0, acol0.data(), acol0.size()))) return rc;
        pb->lin_lb = llb;
        pb->lin_ub = lub;
        if ((rc = dev_upload(pb, &pb->dlin_lb, llb.data(), llb.size()))) return rc;
        if ((rc = dev_upload(pb, &pb->dlin_ub, lub.data(), lub.size()))) return rc;
    }
    CUDA_TRY(cudaDeviceSynchronize());
    cleanup.p = nullptr;
    pb->dims.band_tile = T.band_tile;
    *out = pb;
    return 0;
}

int ntgb_get_dims(const ntgb_problem *pb, ntgb_dims *dims)
{
    if (!pb || !dims) return fail(NTGB_EINVAL, "ntgb_get_dims: null argument");
    *dims = pb->dims;
    return 0;
}

int ntgb_get_tables(const ntgb_problem *pb, double *B, int *offset, int *left)
{
    if (!pb) return fail(NTGB_EINVAL, "null problem");
    if (B) memcpy(B, pb->hB.data(), pb->hB.size() * sizeof(double));
    if (offset) memcpy(offset, pb->hoff.data(), pb->hoff.size() * sizeof(int));
    if (left) memcpy(left, pb->hleft.data(), pb->hleft.size() * sizeof(int));
    return 0;
}

int ntgb_get_augknots(const ntgb_problem *pb, int j, double *t, int *len)
{
    if (!pb || j < 0 || j >= pb->dims.nout) return fail(NTGB_EINVAL, "bad output index");
    if (len) *len = (int)pb->augknots[j].size();
    if (t) memcpy(t, pb->augknots[j].data(), pb->augknots[j].size() * sizeof(double));
    return 0;
}

int ntgb_get_pattern(const ntgb_problem *pb, int *col0, int *jk0)
{
    if (!pb) return fail(NTGB_EINVAL, "null problem");
    if (col0 && pb->dims.ncnln > 0) memcpy(col0, pb->col0.data(), sizeof(int) * (size_t)pb->dims.ncnln * pb->dims.nout);
    if (jk0) memcpy(jk0, pb->tab.jk0, sizeof(int) * pb->dims.nout);
    return 0;
}

int ntgb_get_linear(const ntgb_problem *pb, double *A)
{
    if (!pb || !A) return fail(NTGB_EINVAL, "null argument");
    if (pb->dims.nclin > 0) memcpy(A, pb->A.data(), pb->A.size() * sizeof(double));
    return 0;
}

/* bounds(), reference src/constraints.c:5-33 with bigbnd = +-DBL_MAX (src/ntg.c:226-229) */
int ntgb_get_bounds(const ntgb_problem *pb, double *bl, double *bu)
{
    if (!pb) return fail(NTGB_EINVAL, "null problem");
    const int nbps = pb->dims.nbps;
    for (int pass = 0; pass < 2; pass++) {
        double *dst = pass ? bu : bl;
        const std::vector<double> &b = pass ? pb->upperb : pb->lowerb;
        if (!dst) continue;
        size_t pos = 0, src = 0;
        for (int i = 0; i < pb->dims.nC; i++) dst[pos++] = pass ? DBL_MAX : -DBL_MAX;
        for (int i = 0; i < pb->nlic; i++) dst[pos++] = b[src++];
        for (int i = 0; i < pb->nltc; i++, src++) for (int j = 0; j < nbps; j++) dst[pos++] = b[src];
        for (int i = 0; i < pb->nlfc; i++) dst[pos++] = b[src++];
        for (int i = 0; i < pb->nnlic; i++) dst[pos++] = b[src++];
        for (int i = 0; i < pb->nnltc; i++, src++) for (int j = 0; j < nbps; j++) dst[pos++] = b[src];
        for (int i = 0; i < pb->nnlfc; i++) dst[pos++] = b[src++];
    }
    return 0;
}

int ntgb_eval(ntgb_problem *pb, const ntgb_eval_args *a)
{
    if (!pb || !a) return fail(NTGB_EINVAL, "ntgb_eval: null argument");
    if (a->P < 0) return fail(NTGB_EINVAL, "P = %d", a->P);
    if (a->P == 0) return 0;
    if (!a->C) return fail(NTGB_EINVAL, "ntgb_eval: C == NULL");
    if (a->mode_obj < -1 || a->mode_obj > 2 || a->mode_con < -1 || a->mode_con > 2)
        return fail(NTGB_EINVAL, "mode must be -1, 0, 1 or 2");
    if (a->jac_layout < NTGB_JAC_NONE || a->jac_layout > NTGB_JAC_BAND)
        return fail(NTGB_EINVAL, "unknown jac_layout %d", a->jac_layout);
    if (a->npeers < 0 || a->npeers > NTGB_MAXPEERS || a->peer_row0 < 0)
        return fail(NTGB_EINVAL, "npeers = %d outside [0,%d] or negative peer_row0", a->npeers, NTGB_MAXPEERS);
    if (a->npeers > 0 && !a->peer_result) return fail(NTGB_EINVAL, "npeers = %d but peer_result == NULL", a->npeers);
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    ntgb_launch L;
    L.abi = NTGB_KERNEL_ABI;
    L.tab = pb->tab;
    L.args = *a;
    L.sm_count = pb->sm_count;
    L.max_smem_optin = pb->max_smem_optin;
    const int rc = pb->pack->launch(&L);
    if (rc == -1000) return fail(NTGB_ELIMIT, "problem needs more shared memory than the device offers");
    if (rc != 0) return fail(NTGB_ECUDA, "kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
    return 0;
}

/* ntgb_eval_host for a handful of problems: everything through one mapped staging block */
static int eval_host_small(ntgb_problem *pb, const ntgb_eval_args *h, size_t jper)
{
    constexpr size_t kBlock = 512 << 10;
    const ntgb_dims &d = pb->dims;
    auto &z = pb->zc;
    if (!z.buf) {
        CUDA_TRY(cudaHostAlloc((void **)&z.buf, kBlock, cudaHostAllocMapped | cudaHostAllocPortable));
        memset(z.buf, 0, kBlock);
        z.bytes = kBlock;
    }
    auto &s0 = pb->hs[0];
    if (!s0.stream) CUDA_TRY(cudaStreamCreateWithFlags(&s0.stream, cudaStreamNonBlocking));
    const size_t P = (size_t)h->P, ncn = (size_t)(d.ncnln > 0 ? d.ncnln : 1);
    /* fixed carve-up for this P: abort flag, C, f, g, c, result, Z, J (J last: its size depends on the layout) */
    size_t off = 16;
    auto take = [&](size_t doubles) { const size_t o = off; off += (doubles * sizeof(double) + 15) & ~(size_t)15; return o; };
    const size_t oC = take(P * d.nC), of = take(P), og = take(P * d.nC), oc = take(P * ncn), orr = take(P * 2),
                 oZ = take(h->Z ? P * d.nZ : 0), oJ = take(h->J ? P * jper : 0);
    if (off > z.bytes) return 1; /* does not fit: the caller falls back to the copying path */
    if (P != z.lastP) { /* another carve-up: nothing that was written before means anything now */
        memset(z.buf, 0, z.bytes);
        z.j_bytes = 0; z.j_layout = NTGB_JAC_NONE; z.lastP = P;
    }
    const bool ov = h->mode_obj == 0 || h->mode_obj == 2, od = h->mode_obj == 1 || h->mode_obj == 2;
    const bool cv = h->mode_con == 0 || h->mode_con == 2, cd = h->mode_con == 1 || h->mode_con == 2;
    if (z.j_bytes && !(h->J && jper) && off > z.j_off) {
        /* a call WITHOUT a Jacobian whose carve-up reaches into the region the last Jacobian call
         * zeroed (Z sits where J used to start): whatever this call writes there would be taken for
         * out-of-band zeros by the next Jacobian call -- forget the region, it is cleared again then */
        memset(z.buf + z.j_off, 0, z.j_bytes);
        z.j_bytes = 0; z.j_layout = NTGB_JAC_NONE;
    }
    if (h->J && jper) {
        /* out-of-band entries are zeros written once (src/ntg.c:218); a different layout, batch size
         * or place in the block means different band positions: clear the old and the new region */
        if (z.j_layout != h->jac_layout || z.j_off != oJ || z.j_bytes != P * jper * sizeof(double)) {
            if (z.j_bytes) memset(z.buf + z.j_off, 0, z.j_bytes);
            memset(z.buf + oJ, 0, P * jper * sizeof(double));
            z.j_layout = h->jac_layout; z.j_off = oJ; z.j_bytes = P * jper * sizeof(double);
        }
    }
    if (h->Z) memset(z.buf + oZ, 0, P * d.nZ * sizeof(double)); /* entries outside the active-variable lists are 0 */
    *reinterpret_cast<int *>(z.buf) = 0;
    memcpy(z.buf + oC, h->C, P * d.nC * sizeof(double));
    ntgb_eval_args a = *h;
    a.C = reinterpret_cast<double *>(z.buf + oC);
    a.f = h->f ? reinterpret_cast<double *>(z.buf + of) : nullptr;
    a.g = h->g ? reinterpret_cast<double *>(z.buf + og) : nullptr;
    a.c = h->c ? reinterpret_cast<double *>(z.buf + oc) : nullptr;
    a.J = h->J ? reinterpret_cast<double *>(z.buf + oJ) : nullptr;
    a.Z = h->Z ? reinterpret_cast<double *>(z.buf + oZ) : nullptr;
    a.result = h->result ? reinterpret_cast<double *>(z.buf + orr) : nullptr;
    a.stream = s0.stream;
    a.abort_flag = reinterpret_cast<int *>(z.buf);
    const int rc = ntgb_eval(pb, &a);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(s0.stream));
    if (h->f && ov) memcpy(h->f, z.buf + of, P * sizeof(double));
    if (h->g && od) memcpy(h->g, z.buf + og, P * d.nC * sizeof(double));
    if (h->c && cv && d.ncnln) memcpy(h->c, z.buf + oc, P * d.ncnln * sizeof(double));
    if (h->J && cd && jper) memcpy(h->J, z.buf + oJ, P * jper * sizeof(double));
    if (h->Z) memcpy(h->Z, z.buf + oZ, P * d.nZ * sizeof(double));
    if (h->result) memcpy(h->result, z.buf + orr, P * 2 * sizeof(double));
    if (*reinterpret_cast<volatile int *>(z.buf)) return fail(NTGB_EABORT, "a callback set *mode = -1");
    return 0;
}

int ntgb_eval_host(ntgb_problem *pb, const ntgb_eval_args *h)
{
    if (!pb || !h) return fail(NTGB_EINVAL, "ntgb_eval_host: null argument");
    if (h->P <= 0) return h->P == 0 ? 0 : fail(NTGB_EINVAL, "P = %d", h->P);
    if (!h->C) return fail(NTGB_EINVAL, "ntgb_eval_host: C == NULL");
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    const ntgb_dims &d = pb->dims;
    const size_t jper = h->jac_layout == NTGB_JAC_DENSE ? (size_t)d.ncnln * d.nC
                      : h->jac_layout == NTGB_JAC_BAND  ? (size_t)d.ncnln * d.sorder : 0;
    /* chunking: one chunk for small batches (an NPSOL callback is P = 1); otherwise chunks of
     * >= 1024 problems and ~192 MB of results (measured on CFG-4, 747 MB per call: 32 MB chunks 13.9 ms,
     * 64 MB 13.5, 192 MB 13.3 = 0.98 of one plain pinned copy of the same bytes; every chunk costs five
     * device-to-host copies, the small ones mostly latency), alternating between the two buffer sets so
     * copies overlap compute.  Host buffers should be page-locked (cudaHostRegister / cudaMallocHost)
     * for the copies to be asynchronous; pageable memory works, without the overlap. */
    const size_t per = sizeof(double) * ((size_t)2 * d.nC + 3 + (size_t)(d.ncnln > 0 ? d.ncnln : 1) +
                                         (h->J ? jper : 0) + (h->Z ? (size_t)d.nZ : 0));
    if (per * (size_t)h->P <= (256u << 10) && getenv("NTG_B200_NO_ZEROCOPY") == nullptr) {
        const int rz = eval_host_small(pb, h, jper);
        if (rz != 1) return rz; /* 1: did not fit after all */
    }
    static const unsigned long long chunk_mb = getenv("NTG_B200_HOST_CHUNK_MB") ? strtoull(getenv("NTG_B200_HOST_CHUNK_MB"), nullptr, 10) : 192ull;
    long long chunk = (long long)(((chunk_mb ? chunk_mb : 192ull) << 20) / (per ? per : 1));
    if (chunk < 1024) chunk = 1024;
    if (chunk > h->P) chunk = h->P;
    const int nbuf = chunk < h->P ? 2 : 1;
    for (int b = 0; b < nbuf; b++) {
        auto &s = pb->hs[b];
        if (!s.stream) CUDA_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        const bool grow = chunk > s.cap || (h->J && (s.jac_layout != h->jac_layout || s.Jbytes < (size_t)chunk * jper * sizeof(double))) ||
                          (h->Z && !s.hasZ);
        if (!grow) continue;
        double **ptrs[] = {&s.C, &s.f, &s.g, &s.c, &s.J, &s.Z, &s.result};
        for (double **pp : ptrs) { if (*pp) cudaFree(*pp); *pp = nullptr; }
        /* nothing is allocated now: if one of the allocations below fails, the next call starts over */
        s.cap = 0; s.Jbytes = 0; s.hasZ = false; s.jac_layout = NTGB_JAC_NONE;
        const size_t cap = (size_t)chunk;
        CUDA_TRY(cudaMalloc((void **)&s.C, cap * d.nC * sizeof(double)));
        CUDA_TRY(cudaMalloc((void **)&s.f, cap * sizeof(double)));
        CUDA_TRY(cudaMalloc((void **)&s.g, cap * d.nC * sizeof(double)));
        CUDA_TRY(cudaMalloc((void **)&s.c, cap * (size_t)(d.ncnln > 0 ? d.ncnln : 1) * sizeof(double)));
        CUDA_TRY(cudaMalloc((void **)&s.result, cap * 2 * sizeof(double)));
        s.hasZ = false;
        if (h->Z) { CUDA_TRY(cudaMalloc((void **)&s.Z, cap * d.nZ * sizeof(double))); s.hasZ = true; }
        s.Jbytes = 0;
        if (h->J && jper) {
            s.Jbytes = cap * jper * sizeof(double);
            CUDA_TRY(cudaMalloc((void **)&s.J, s.Jbytes));
            /* out-of-band entries are zeroed once, as the reference's calloc does (src/ntg.c:218);
             * the band positions are the same for every problem, so reuse across chunks is safe */
            CUDA_TRY(cudaMemsetAsync(s.J, 0, s.Jbytes, s.stream));
        }
        s.cap = (int)cap;
        s.jac_layout = h->jac_layout;
    }
    const bool ov = h->mode_obj == 0 || h->mode_obj == 2, od = h->mode_obj == 1 || h->mode_obj == 2;
    const bool cv = h->mode_con == 0 || h->mode_con == 2, cd = h->mode_con == 1 || h->mode_con == 2;
    if (!pb->d_abort) { if (int rc0 = dev_alloc(pb, &pb->d_abort, 1)) return rc0; }
    CUDA_TRY(cudaMemsetAsync(pb->d_abort, 0, sizeof(int), pb->hs[0].stream));
    if (nbuf > 1) CUDA_TRY(cudaStreamSynchronize(pb->hs[0].stream)); /* the other stream must see the zero */
    int k = 0;
    for (long long lo = 0; lo < h->P; lo += chunk, k++) {
        auto &s = pb->hs[k % nbuf];
        const size_t n = (size_t)((h->P - lo) < chunk ? (h->P - lo) : chunk);
        cudaStream_t st = s.stream;
        CUDA_TRY(cudaMemcpyAsync(s.C, h->C + (size_t)lo * d.nC, n * d.nC * sizeof(double), cudaMemcpyHostToDevice, st));
        ntgb_eval_args a = *h;
        a.P = (int)n;
        a.C = s.C;
        a.f = h->f ? s.f : nullptr;
        a.g = h->g ? s.g : nullptr;
        a.c = h->c ? s.c : nullptr;
        a.J = h->J ? s.J : nullptr;
        a.Z = h->Z ? s.Z : nullptr;
        a.result = h->result ? s.result : nullptr;
        a.stream = st;
        a.abort_flag = pb->d_abort;
        const int rc = ntgb_eval(pb, &a);
        if (rc) return rc;
        if (h->f && ov) CUDA_TRY(cudaMemcpyAsync(h->f + lo, s.f, n * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (h->g && od) CUDA_TRY(cudaMemcpyAsync(h->g + (size_t)lo * d.nC, s.g, n * d.nC * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (h->c && cv && d.ncnln) CUDA_TRY(cudaMemcpyAsync(h->c + (size_t)lo * d.ncnln, s.c, n * d.ncnln * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (h->J && cd && jper) CUDA_TRY(cudaMemcpyAsync(h->J + (size_t)lo * jper, s.J, n * jper * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (h->Z) CUDA_TRY(cudaMemcpyAsync(h->Z + (size_t)lo * d.nZ, s.Z, n * d.nZ * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (h->result) CUDA_TRY(cudaMemcpyAsync(h->result + (size_t)lo * 2, s.result, n * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    int aborted = 0;
    CUDA_TRY(cudaMemcpyAsync(&aborted, pb->d_abort, sizeof(int), cudaMemcpyDeviceToHost, pb->hs[(k - 1) % nbuf].stream));
    for (int b = 0; b < nbuf; b++) CUDA_TRY(cudaStreamSynchronize(pb->hs[b].stream));
    if (nbuf > 1 && !aborted) { /* the flag copy ran on one stream; re-read after both finished */
        CUDA_TRY(cudaMemcpy(&aborted, pb->d_abort, sizeof(int), cudaMemcpyDeviceToHost));
    }
    if (aborted) return fail(NTGB_EABORT, "a callback set *mode = -1");
    return 0;
}

void *ntgb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        fail(NTGB_ENOMEM, "cudaMallocHost(%zu) failed", bytes);
        return nullptr;
    }
    return p;
}

void ntgb_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

int ntgb_host_register(void *p, size_t bytes)
{
    if (!p) return fail(NTGB_EINVAL, "ntgb_host_register: null pointer");
    CUDA_TRY(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
    return 0;
}

int ntgb_host_unregister(void *p)
{
    if (!p) return fail(NTGB_EINVAL, "ntgb_host_unregister: null pointer");
    CUDA_TRY(cudaHostUnregister(p));
    return 0;
}

int ntgb_eval_linear(ntgb_problem *pb, int P, const double *C, double *lin, double *viol, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_eval_linear: null argument");
    const int nclin = pb->dims.nclin;
    if (P <= 0 || nclin == 0) return 0;
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (viol) CUDA_TRY(cudaMemsetAsync(viol, 0, sizeof(double) * (size_t)P, st));
    const long long total = (long long)P * nclin;
    const int block = 256;
    const unsigned grid = (unsigned)((total + block - 1) / block);
    CUDA_TRY(launch(k_linear, grid, block, st, pb->dAband, pb->dAcol0, pb->dlin_lb, pb->dlin_ub, nclin,
                    pb->dims.nout, pb->dims.sorder, pb->tab, P, C, lin, viol));
    return 0;
}

int ntgb_linesearch(ntgb_problem *pb, int P, const double *C, const double *dC, int nalpha, const double *alpha,
                    double mu, double c1, const double *phi0, const double *dphi0, double *alpha_best,
                    double *phi_best, double *C_new, void *stream)
{
    if (!pb || !C || !dC || !alpha) return fail(NTGB_EINVAL, "ntgb_linesearch: null argument");
    if (P <= 0) return 0;
    if (nalpha < 1 || nalpha > 64) return fail(NTGB_EINVAL, "nalpha = %d outside [1,64]", nalpha);
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    const size_t n = (size_t)P * nalpha;
    if (n > 0x7fffffffull) return fail(NTGB_EINVAL, "P*nalpha too large");
    cudaStream_t st = (cudaStream_t)stream;
    LsArrays la;
    int rc;
    if ((rc = scratch_carve(pb->scratch.ls, st, [&](Carve &c) { la.take(c, n, pb->dims.nC); }))) return rc;
    return linesearch_run(pb, P, C, dC, nalpha, alpha, mu, c1, phi0, dphi0, alpha_best, phi_best, C_new, st, la);
}

int ntgb_solve_eq(ntgb_problem *pb, int P, double *C, double *f, int *iters, int *status,
                  const ntgb_solve_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_eq: null argument");
    return solve_eq_impl(pb, Run::Sync, P, C, nullptr, nullptr, f, iters, status, opts, stream);
}

int ntgb_solve_eq_bounds(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                         int *iters, int *status, const ntgb_solve_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_eq_bounds: null argument");
    if (bounds_layout(pb).nb() > 0 && (!lowerb || !upperb))
        return fail(NTGB_EINVAL, "ntgb_solve_eq_bounds: lowerb / upperb is NULL");
    return solve_eq_impl(pb, Run::Sync, P, C, lowerb, upperb, f, iters, status, opts, stream);
}

int ntgb_solve_eq_reserve(ntgb_problem *pb, int P_max)
{
    if (!pb) return fail(NTGB_EINVAL, "ntgb_solve_eq_reserve: null argument");
    if (P_max < 1) return fail(NTGB_EINVAL, "ntgb_solve_eq_reserve: P_max = %d", P_max);
    return solve_eq_impl(pb, Run::Reserve, P_max, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

int ntgb_solve_eq_async(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                        int *iters, int *status, const ntgb_solve_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_eq_async: null argument");
    if ((lowerb == nullptr) != (upperb == nullptr))
        return fail(NTGB_EINVAL, "ntgb_solve_eq_async: exactly one of lowerb / upperb is NULL");
    return solve_eq_impl(pb, Run::Async, P, C, lowerb, upperb, f, iters, status, opts, stream);
}

int ntgb_solve_eq_lbfgs(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                        int *iters, int *status, const ntgb_lbfgs_opts *opts, void *stream)
{
    /* the argument checks read nothing behind pb */
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_eq_lbfgs: null argument");
    if ((lowerb == nullptr) != (upperb == nullptr))
        return fail(NTGB_EINVAL, "ntgb_solve_eq_lbfgs: exactly one of lowerb / upperb is NULL");
    ntgb_lbfgs_opts o{500, 1e-9, 1e-4, 8, 4};
    if (opts) {
        if (opts->memory < 1 || opts->memory > ntgb::lbfgs::kMaxMemory)
            return fail(NTGB_EINVAL, "ntgb_solve_eq_lbfgs: memory = %d outside [1,%d]", opts->memory,
                        ntgb::lbfgs::kMaxMemory);
        o.memory = opts->memory;
        if (opts->max_iter > 0) o.max_iter = opts->max_iter;
        if (opts->gtol > 0.0) o.gtol = opts->gtol;
        if (opts->c1 > 0.0) o.c1 = opts->c1;
        if (opts->check_every > 0) o.check_every = opts->check_every;
    }
    if (P <= 0) return 0;
    return solve_lbfgs_impl(pb, P, C, lowerb, upperb, f, iters, status, o, stream);
}

int ntgb_solve_eq_newton(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                         int *iters, int *status, const ntgb_newton_opts *opts, void *stream)
{
    /* the argument checks read nothing behind pb */
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_eq_newton: null argument");
    if ((lowerb == nullptr) != (upperb == nullptr))
        return fail(NTGB_EINVAL, "ntgb_solve_eq_newton: exactly one of lowerb / upperb is NULL");
    ntgb_newton_opts o{100, 1e-9, 1e-4, 4};
    if (opts) {
        if (opts->max_iter > 0) o.max_iter = opts->max_iter;
        if (opts->gtol > 0.0) o.gtol = opts->gtol;
        if (opts->c1 > 0.0) o.c1 = opts->c1;
        if (opts->check_every > 0) o.check_every = opts->check_every;
    }
    if (P <= 0) return 0;
    return solve_newton_impl(pb, P, C, lowerb, upperb, f, iters, status, o, stream);
}

int ntgb_newton_structure(ntgb_problem *pb, int *ncolors, int *half_bandwidth, int *perm)
{
    if (!pb) return fail(NTGB_EINVAL, "ntgb_newton_structure: null argument");
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    int rc;
    if ((rc = newton_prepare(pb))) return rc;
    const auto &nw = pb->newton;
    if (ncolors) *ncolors = nw.K;
    if (half_bandwidth) *half_bandwidth = nw.w;
    if (perm) memcpy(perm, nw.hperm.data(), sizeof(int) * nw.hperm.size());
    return 0;
}

} /* extern "C" */

namespace {

/* ntgb_solve_eq, ntgb_solve_eq_bounds and their reserve / async entry points (Run): lowerb == nullptr = the
 * setup's bounds for every problem */
int solve_eq_impl(ntgb_problem *pb, Run run, int P, double *C, const double *lowerb, const double *upperb, double *f,
                  int *iters, int *status, const ntgb_solve_opts *opts, void *stream)
{
    if (P <= 0) return 0;
    AsyncWork &aw = pb->async.eq;
    if (run == Run::Async && P > aw.P)
        return fail(NTGB_EINVAL, "ntgb_solve_eq_async: P = %d above the %d problems reserved by ntgb_solve_eq_reserve", P,
                    aw.P);
    const ntgb_dims &dm = pb->dims;
    int rc;
    if ((rc = check_eq_only(pb, "ntgb_solve_eq"))) return rc;
    ntgb_solve_opts o{200, 1e-9, 1e-4, 4};
    if (opts) {
        if (opts->max_iter > 0) o.max_iter = opts->max_iter;
        if (opts->gtol > 0.0) o.gtol = opts->gtol;
        if (opts->c1 > 0.0) o.c1 = opts->c1;
        if (opts->check_every > 0) o.check_every = opts->check_every;
    }
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int nC = dm.nC;
    /* every linear row is an equality (the refusals above), so alm's reduced form eliminates all of them */
    if ((rc = alm_prepare(pb))) return rc;
    const auto &al = pb->alm;
    if (al.nr > kSolveMaxNr)
        return fail(NTGB_ELIMIT, "ntgb_solve_eq: %d free directions after eliminating the linear constraints (limit %d)",
                    al.nr, kSolveMaxNr);
    const int nr = al.nr;
    constexpr int kNalpha = 12;
    const size_t Pz = (size_t)P;
    double *y, *yp, *grp, *d, *H, *dC, *g, *fv, *phi0, *dphi0, *ab, *pbest, *alphas;
    int *state, *its, *fails, *count;
    /* be = the expanded linear bounds, row r of be is linear row r */
    const BoundsDesc B{bounds_layout(pb), nC, 0, 0, dm.nclin, nullptr, nullptr, al.M, al.Ae};
    BoundsArrays ba;
    LsArrays la;
    auto layout = [&](Carve &c) {
        c.take(Pz * nr, y, yp, grp, d);
        c.take(Pz * nr * nr, H);
        c.take(Pz * nC, dC, g);
        c.take(Pz, fv, phi0, dphi0, ab, pbest, state, its, fails);
        c.take(kNalpha, alphas);
        c.take(1, count);
        if (run != Run::Sync) { /* what the synchronous path takes from the bounds' and the line search's scratch */
            ba.take(c, Pz, B);
            la.take(c, Pz * kNalpha, nC);
        }
    };
    if (run == Run::Reserve) {
        if (Pz * kNalpha > 0x7fffffffull) return fail(NTGB_EINVAL, "P*nalpha too large"); /* ntgb_linesearch's check */
        return reserve_work(pb, aw, P, layout);
    }
    if ((rc = scratch_carve(run == Run::Sync ? pb->scratch.eq : aw.s, st, layout, run == Run::Sync))) return rc;
    if (run == Run::Sync) {
        if ((rc = upload_halving(alphas, kNalpha, st))) return rc;
    } else {
        alphas = pb->async.halving;
    }
    CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
    const double *Cpart = al.Cpart;
    int Cstride = 0;
    if (lowerb) {
        if (run == Run::Sync && (rc = scratch_carve(pb->scratch.bnd, st, [&](Carve &c) { ba.take(c, Pz, B); }))) return rc;
        if ((rc = bounds_prepare(P, lowerb, upperb, B, ba, st, state, its, count))) return rc;
        Cpart = ba.Cpart;
        Cstride = nC;
    }
    const unsigned grid = (unsigned)((P + 127) / 128);
    CUDA_TRY(launch(k_solve_init, grid, 128, st, P, nC, nr, al.N, Cpart, Cstride, C, y, H, state, its, fails));
    ntgb_eval_args a;
    memset(&a, 0, sizeof a);
    a.P = P; a.C = C; a.mode_obj = 2; a.mode_con = -1; a.f = fv; a.g = g; a.jac_layout = NTGB_JAC_NONE; a.stream = st;
    for (int it = 0; it < o.max_iter; it++) {
        if ((rc = ntgb_eval(pb, &a))) return rc;
        CUDA_TRY(launch(k_solve_dir, grid, 128, st, P, nC, nr, al.N, fv, g, o.gtol, y, yp, grp, H, d, dC, phi0,
                        dphi0, state, fails, count));
        if (run == Run::Sync && (it + 1) % o.check_every == 0 && (rc = all_finished(count, P, st)) != 0) {
            if (rc < 0) return rc;
            break;
        }
        if (run == Run::Sync)
            rc = ntgb_linesearch(pb, P, C, dC, kNalpha, alphas, 0.0, o.c1, phi0, dphi0, ab, pbest, nullptr, st);
        else
            rc = linesearch_run(pb, P, C, dC, kNalpha, alphas, 0.0, o.c1, phi0, dphi0, ab, pbest, nullptr, st, la);
        if (rc) return rc;
        CUDA_TRY(launch(k_solve_update, grid, 128, st, P, nC, nr, al.N, Cpart, Cstride, phi0, ab, pbest, d, y, H,
                        C, state, its, fails, count));
    }
    if (f) {
        a.mode_obj = 0; a.f = f; a.g = nullptr;
        if ((rc = ntgb_eval(pb, &a))) return rc;
    }
    if (iters) CUDA_TRY(cudaMemcpyAsync(iters, its, sizeof(int) * (size_t)P, cudaMemcpyDeviceToDevice, st));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, state, sizeof(int) * (size_t)P, cudaMemcpyDeviceToDevice, st));
    if (run == Run::Sync) CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}


/* ---- ntgb_solve_eq_lbfgs: projected L-BFGS, one CTA per problem running ntg_lbfgs.h --------------------- */
struct LbfgsDesc {
    const double *Q1; /* [r][nC] */
    int r, nC, mem;
};

/* per-problem state: the ring [P][mem][2][nC] of curvature pairs and what ntg_lbfgs.h keeps next to it */
struct LbfgsArrays {
    double *ring, *sv, *gp; /* [P][mem][2][nC], [P][nC], [P][nC] */
    double *rho;            /* [P][mem] */
    double *gamma;          /* [P] */
    int *state, *its, *head, *npair, *pend; /* [P] */

    void take(Carve &c, size_t P, int nC, int mem)
    {
        c.take(P * mem * 2 * nC, ring);
        c.take(P * nC, sv, gp);
        c.take(P * mem, rho);
        c.take(P, gamma);
        c.take(P, state, its, head, npair, pend);
    }
    __device__ ntgb::lbfgs::View view(const LbfgsDesc &D, int p) const
    {
        const size_t n = D.nC;
        return ntgb::lbfgs::View{D.Q1, D.r, D.nC, D.mem, ring + (size_t)p * D.mem * 2 * n, rho + (size_t)p * D.mem,
                                 sv + p * n, gp + p * n};
    }
    __device__ ntgb::lbfgs::State load(int p) const { return ntgb::lbfgs::State{head[p], npair[p], pend[p], gamma[p]}; }
    __device__ void store(int p, const ntgb::lbfgs::State &s) const
    {
        head[p] = s.head;
        npair[p] = s.npair;
        pend[p] = s.pend;
        gamma[p] = s.gamma;
    }
};

/* threads per problem: every step streams a handful of nC-vectors through a chain of block reductions.  Up to
 * a few thousand coefficients, 128 threads keep each reduction short and leave room for more resident CTAs;
 * at CFG-5 sizes (nC = 4824) 256 threads halve the elements each thread walks between two reductions, and
 * such batches are small, so the larger CTA costs no occupancy.  It depends on nC alone, so the reduction
 * order, and every result, does not depend on the batch. */
int lbfgs_threads(int nC) { return nC >= 2048 ? 256 : 128; }

/* the CTA as ntg_lbfgs.h's group; its reductions take one double of shared memory per warp */
__device__ __forceinline__ sqp::Coop lbfgs_group()
{
    return sqp::Coop{(int)threadIdx.x, (int)blockDim.x, (int)(threadIdx.x & 31), 32};
}

/* at entry: C onto problem p's affine set, fresh history.  Per-problem bounds (Cstride = nC): k_bounds_prep has
 * set state / iters, a rejected problem keeps its C.  No free direction (r == nC): C = Cpart and status 1, as
 * ntgb_solve_eq gives */
__global__ void k_lbfgs_init(int P, LbfgsDesc D, LbfgsArrays S, const double *Cpart, int Cstride, double *C)
{
    __shared__ double red[8];
    const int p = blockIdx.x;
    if (Cstride != 0 && S.state[p] == NTGB_STATUS_BAD_BOUNDS) return;
    Cpart += (size_t)p * Cstride;
    double *Cp = C + (size_t)p * D.nC;
    if (D.r == D.nC) {
        for (int e = threadIdx.x; e < D.nC; e += blockDim.x) Cp[e] = Cpart[e];
    } else {
        ntgb::lbfgs::affine_step(lbfgs_group(), red, S.view(D, p), Cpart, Cp, nullptr, 0.0);
    }
    if (threadIdx.x == 0) {
        S.state[p] = D.r == D.nC ? 1 : 0;
        S.its[p] = 0;
        S.store(p, ntgb::lbfgs::State{0, 0, 0, 1.0});
    }
}

/* projected gradient, convergence test, pair update, two-loop direction dC and its slope; a finished problem
 * gets dC = 0 and slope 0, which keeps it where it is through the search */
__global__ void k_lbfgs_dir(int P, LbfgsDesc D, LbfgsArrays S, const double *f, const double *g, double gtol, double *dC,
                            double *phi0, double *dphi0, int *count)
{
    __shared__ double red[8];
    const int p = blockIdx.x;
    const size_t n = D.nC;
    double *d = dC + p * n;
    int st = S.state[p];
    double dg = 0.0;
    if (st == 0) {
        ntgb::lbfgs::State s = S.load(p);
        st = ntgb::lbfgs::direction(lbfgs_group(), red, S.view(D, p), s, f[p], g + p * n, gtol, d, dg);
        if (threadIdx.x == 0) {
            S.store(p, s);
            if (st != 0) {
                S.state[p] = st;
                atomicAdd(count, 1);
            }
        }
    }
    if (st != 0) {
        for (size_t e = threadIdx.x; e < n; e += blockDim.x) d[e] = 0.0;
        dg = 0.0;
    }
    if (threadIdx.x == 0) {
        phi0[p] = f[p];
        dphi0[p] = dg;
    }
}

/* the step the search chose, or what a failed search means (ntg_lbfgs.h accept) */
__global__ void k_lbfgs_update(int P, LbfgsDesc D, LbfgsArrays S, const double *Cpart, int Cstride, const double *phi0,
                               const double *alpha_best, const double *phi_best, const double *dC, double *C, int *count)
{
    __shared__ double red[8];
    const int p = blockIdx.x;
    if (S.state[p] != 0) return;
    const size_t n = D.nC;
    ntgb::lbfgs::State s = S.load(p);
    const int st = ntgb::lbfgs::accept(lbfgs_group(), red, S.view(D, p), s, Cpart + (size_t)p * Cstride, C + p * n,
                                       dC + p * n, alpha_best[p], phi0[p], phi_best[p]);
    if (threadIdx.x == 0) {
        S.its[p] += 1;
        S.store(p, s);
        if (st != 0) {
            S.state[p] = st;
            atomicAdd(count, 1);
        }
    }
}

/* merit of the L-BFGS search: the plain cost, where two_stage_search's pick kernels read it */
__global__ void k_cost_merit(int Q, const double *f, double *res)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < Q) res[2 * (size_t)q] = f[q];
}

/* ntgb_solve_eq_lbfgs.  The search is two_stage_search on the plain cost: L-BFGS accepts the unit step most of
 * the time, so the 4 coarse steps evaluated for every problem usually decide, and the 12 fine ones are
 * evaluated only for the few problems that need them (ntgb_linesearch would evaluate 12 for every problem). */
int solve_lbfgs_impl(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                     int *iters, int *status, const ntgb_lbfgs_opts &o, void *stream)
{
    const ntgb_dims &dm = pb->dims;
    const int nC = dm.nC;
    int rc;
    if ((rc = check_eq_only(pb, "ntgb_solve_eq_lbfgs"))) return rc;
    if ((rc = TwoStage::check_size(P))) return rc;
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = reduced_form(pb, false, true))) return rc;
    const auto &al = pb->alm;
    const size_t Pz = (size_t)P;
    const LbfgsDesc D{al.Q1, al.r, nC, o.memory};
    /* be = the expanded linear bounds, row r of be is linear row r (every linear row is eliminated) */
    const BoundsDesc B{bounds_layout(pb), nC, 0, 0, dm.nclin, nullptr, nullptr, al.M, al.Ae};
    LbfgsArrays S;
    TwoStage ts;
    BoundsArrays ba;
    double *g, *dC, *fv, *phi0, *dphi0;
    int *count;
    if ((rc = scratch_carve(pb->scratch.lbfgs, st, [&](Carve &c) {
             S.take(c, Pz, nC, o.memory);
             c.take(Pz * nC, g, dC);
             c.take(Pz, fv, phi0, dphi0);
             c.take(1, count);
             ts.take(c, Pz, dm);
             if (lowerb) ba.take(c, Pz, B);
         })))
        return rc;
    if ((rc = ts.start(P, st))) return rc;
    CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
    const double *Cpart = al.Cpart;
    int Cstride = 0;
    if (lowerb) {
        if ((rc = bounds_prepare(P, lowerb, upperb, B, ba, st, S.state, S.its, count))) return rc;
        Cpart = ba.Cpart;
        Cstride = nC;
    }
    const int nt = lbfgs_threads(nC);
    CUDA_TRY(launch(k_lbfgs_init, (unsigned)P, nt, st, P, D, S, Cpart, Cstride, C));
    ntgb_eval_args a;
    memset(&a, 0, sizeof a);
    a.P = P; a.C = C; a.mode_obj = 2; a.mode_con = -1; a.f = fv; a.g = g; a.jac_layout = NTGB_JAC_NONE; a.stream = st;
    auto merit = [&](int n, int, const int *) -> int {
        CUDA_TRY(launch(k_cost_merit, (unsigned)((n + 255) / 256), 256, st, n, (const double *)ts.ft, ts.res));
        return 0;
    };
    const int max_iter = al.nr > 0 ? o.max_iter : 0; /* no free direction: k_lbfgs_init has finished every problem */
    for (int it = 0; it < max_iter; it++) {
        if ((rc = ntgb_eval(pb, &a))) return rc;
        CUDA_TRY(launch(k_lbfgs_dir, (unsigned)P, nt, st, P, D, S, (const double *)fv, (const double *)g, o.gtol, dC, phi0,
                        dphi0, count));
        if ((it + 1) % o.check_every == 0 && (rc = all_finished(count, P, st)) != 0) {
            if (rc < 0) return rc;
            break;
        }
        if ((rc = two_stage_search(pb, P, C, dC, o.c1, phi0, dphi0, S.state, ts, st, merit))) return rc;
        CUDA_TRY(launch(k_lbfgs_update, (unsigned)P, nt, st, P, D, S, Cpart, Cstride, phi0, ts.ab, ts.pbest, dC, C, count));
    }
    if (f) {
        a.mode_obj = 0; a.f = f; a.g = nullptr;
        if ((rc = ntgb_eval(pb, &a))) return rc;
    }
    if (iters) CUDA_TRY(cudaMemcpyAsync(iters, S.its, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, S.state, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

/* ---- ntgb_solve_eq_newton: banded Newton, one CTA per problem running ntg_newton.h ----------------------- */

/* threads of the factor and direction CTAs: fixed, so that no result depends on the batch.  The window update
 * of the factor has w (w+1) / 2 entries per column (91 at the lane change's w = 13), the direction walks r + 1
 * right-hand sides, one per thread (r <= kMaxRows). */
constexpr int kNewtonThreads = 128;

struct NewtonArrays {
    double *Xp, *Gp, *fp;                  /* [P][2K][nC] difference points and their gradients, [P][2K] costs */
    double *band;                          /* [P][nC][w+1] H + rho A'A + tau I, then its factor */
    double *Y, *S, *lam;                   /* [P][r+1][nC], [P][r][r], [P][r] of the range-space step */
    double *pg, *sv;                       /* [P][nC] projected gradient, the last step */
    double *tau, *beta;                    /* [P] */
    int *state, *its, *stall, *factored;   /* [P] */

    void take(Carve &c, size_t P, int nC, int K, int w, int r)
    {
        c.take(P * 2 * K * nC, Xp, Gp);
        c.take(P * 2 * K, fp);
        c.take(P * nC * (w + 1), band);
        c.take(P * (r + 1) * nC, Y);
        c.take(P * std::max(r * r, 1), S);
        c.take(P * std::max(r, 1), lam);
        c.take(P * nC, pg, sv);
        c.take(P, tau, beta);
        c.take(P, state, its, stall, factored);
    }
    __device__ ntgb::lbfgs::View proj(const ntgb::newton::Desc &D, int p) const
    {
        return ntgb::lbfgs::View{D.Q1, D.r, D.nC, 0, nullptr, nullptr, sv + (size_t)p * D.nC, nullptr};
    }
};

/* at entry: C onto problem p's affine set, no shift.  Per-problem bounds (Cstride = nC): k_bounds_prep has set
 * state / iters, a rejected problem keeps its C.  No free direction (r == nC): C = Cpart and status 1 */
__global__ void k_newton_init(int P, ntgb::newton::Desc D, NewtonArrays S, const double *Cpart, int Cstride, double *C)
{
    __shared__ double red[kNewtonThreads / 32];
    const int p = blockIdx.x;
    if (Cstride != 0 && S.state[p] == NTGB_STATUS_BAD_BOUNDS) return;
    Cpart += (size_t)p * Cstride;
    double *Cp = C + (size_t)p * D.nC;
    if (D.r == D.nC) {
        for (int e = threadIdx.x; e < D.nC; e += blockDim.x) Cp[e] = Cpart[e];
    } else {
        ntgb::lbfgs::affine_step(lbfgs_group(), red, S.proj(D, p), Cpart, Cp, nullptr, 0.0);
    }
    if (threadIdx.x == 0) {
        S.state[p] = D.r == D.nC ? 1 : 0;
        S.its[p] = 0;
        S.tau[p] = 0.0;
        S.beta[p] = 0.0;
        S.stall[p] = 0;
    }
}

/* P g and the convergence test: |P g|_inf <= gtol max(1, |f|) is status 1, a NaN gradient status 2 */
__global__ void k_newton_check(int P, ntgb::newton::Desc D, NewtonArrays S, const double *f, const double *g, double gtol,
                               int *count)
{
    __shared__ double red[kNewtonThreads / 32];
    const int p = blockIdx.x;
    if (S.state[p] != 0) return;
    const size_t n = D.nC;
    double *pg = S.pg + p * n;
    const sqp::Coop cg = lbfgs_group();
    for (size_t e = threadIdx.x; e < n; e += blockDim.x) pg[e] = g[p * n + e];
    ntgb::lbfgs::project(cg, red, D.Q1, D.r, D.nC, pg);
    double gmax = 0.0, gg = 0.0;
    for (size_t e = threadIdx.x; e < n; e += blockDim.x) {
        gmax = fmax(gmax, fabs(pg[e]));
        gg += pg[e] * pg[e];
    }
    gmax = cg.reduce<true>(gmax, red);
    gg = cg.reduce<false>(gg, red);
    const double fa = fabs(f[p]);
    const int st = gg != gg ? 2 : (!(gmax > gtol * (fa > 1.0 ? fa : 1.0)) ? 1 : 0);
    if (threadIdx.x == 0 && st != 0) {
        S.state[p] = st;
        atomicAdd(count, 1);
    }
}

/* the 2K difference points of every problem: point 2k = C + h on the columns of colour k, 2k + 1 = C - h */
__global__ void k_newton_points(int P, int nC, int K, const int *color, const double *C, double *Xp)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (long long)P * 2 * K * nC) return;
    const int e = (int)(q % nC);
    const long long pk = q / nC;
    const int k2 = (int)(pk % (2 * K));
    const long long p = pk / (2 * K);
    const double x = C[p * nC + e], h = ntgb::newton::fd_step(x);
    Xp[q] = color[e] == (k2 >> 1) ? ((k2 & 1) ? x - h : x + h) : x;
}

/* M = H + rho A'A + tau I from the differences and its banded Cholesky; a nonpositive pivot raises tau to
 * max(4 tau, beta) and refactors, up to kMaxShift times.  The window is dynamic shared memory. */
__global__ void k_newton_factor(int P, ntgb::newton::Desc D, NewtonArrays S, const double *C)
{
    extern __shared__ double win[];
    __shared__ double red[kNewtonThreads / 32];
    const int p = blockIdx.x;
    if (S.state[p] != 0) return;
    const size_t n = D.nC;
    const sqp::Coop cg = lbfgs_group();
    double *band = S.band + p * n * (D.w + 1);
    double tau = S.tau[p], beta = 0.0;
    bool ok = false;
    for (int a = 0; a <= ntgb::newton::kMaxShift && !ok; a++) {
        if (a > 0) tau = fmax(4.0 * tau, beta);
        double dmax = 0.0;
        ntgb::newton::assemble(cg, red, D, C + p * n, S.Gp + p * 2 * D.K * n, tau, band, dmax);
        beta = ntgb::newton::kBetaRel * (dmax > 0.0 ? dmax : 1.0);
        ok = ntgb::newton::band_cholesky(cg, D.nC, D.w, band, win);
    }
    if (threadIdx.x == 0) {
        S.tau[p] = tau;
        S.beta[p] = beta;
        S.factored[p] = ok ? 1 : 0;
    }
}

/* the range-space Newton step, or d = -P g after a failed factorization, a singular S or a slope d'g >= 0;
 * phi0 = f + 8 eps |f| (the search's rounding allowance), dphi0 = d'g.  A finished problem gets d = 0. */
__global__ void k_newton_dir(int P, ntgb::newton::Desc D, NewtonArrays S, const double *f, const double *g, double *dC,
                             double *phi0, double *dphi0)
{
    __shared__ double red[kNewtonThreads / 32];
    const int p = blockIdx.x;
    const size_t n = D.nC;
    double *d = dC + p * n;
    const sqp::Coop cg = lbfgs_group();
    double dg = 0.0;
    if (S.state[p] == 0) {
        const size_t r = D.r, rr = r > 0 ? r * r : 1, r1 = r > 0 ? r : 1; /* NewtonArrays::take */
        bool ok = S.factored[p] && ntgb::newton::range_step(cg, D, S.band + p * n * (D.w + 1), g + p * n,
                                                             S.Y + p * (r + 1) * n, S.S + p * rr, S.lam + p * r1, d);
        if (ok) {
            dg = ntgb::lbfgs::dot(cg, red, d, g + p * n, D.nC);
            ok = dg < 0.0;
        }
        if (!ok) {
            const double *pg = S.pg + p * n;
            double gg = 0.0;
            for (size_t e = threadIdx.x; e < n; e += blockDim.x) {
                d[e] = -pg[e];
                gg += pg[e] * pg[e];
            }
            dg = -cg.reduce<false>(gg, red);
        }
    } else {
        for (size_t e = threadIdx.x; e < n; e += blockDim.x) d[e] = 0.0;
    }
    if (threadIdx.x == 0) {
        const double fa = fabs(f[p]);
        phi0[p] = S.state[p] == 0 ? f[p] + 8.0 * DBL_EPSILON * fa : f[p];
        dphi0[p] = dg;
    }
}

/* the step the search chose, the shift and the stopping rule (ntg_newton.h after_search) */
__global__ void k_newton_update(int P, ntgb::newton::Desc D, NewtonArrays S, const double *Cpart, int Cstride, double c1,
                                const double *f, const double *phi0, const double *dphi0, const double *alpha_best,
                                const double *phi_best, const double *dC, double *C, int *count)
{
    __shared__ double red[kNewtonThreads / 32];
    const int p = blockIdx.x;
    if (S.state[p] != 0) return;
    const size_t n = D.nC;
    const double a = alpha_best[p];
    /* the test of k_alm_pick1 / k_alm_pick2, on the same operands */
    const bool armijo = phi_best[p] <= phi0[p] + c1 * a * dphi0[p];
    if (armijo) ntgb::lbfgs::affine_step(lbfgs_group(), red, S.proj(D, p), Cpart + (size_t)p * Cstride, C + p * n, dC + p * n, a);
    if (threadIdx.x == 0) {
        ntgb::newton::State s{S.tau[p], S.beta[p], S.stall[p]};
        int done = 0;
        ntgb::newton::after_search(s, armijo, a, phi_best[p], f[p], &done);
        S.tau[p] = s.tau;
        S.stall[p] = s.stall;
        S.its[p] += 1;
        if (done != 0) {
            S.state[p] = done;
            atomicAdd(count, 1);
        }
    }
}

/* the structure of ntg_newton.h for this setup, once: the pattern of the cost from the K0 offsets and the
 * cost's active variables, and of A'A from the equality rows */
int newton_prepare(ntgb_problem *pb)
{
    auto &nw = pb->newton;
    if (nw.ready) return 0;
    const ntgb_dims &dm = pb->dims;
    const int nC = dm.nC, nclin = dm.nclin;
    std::vector<double> A;
    int m = 0;
    for (int i = 0; i < nclin; i++)
        if (pb->lin_lb[i] == pb->lin_ub[i]) {
            for (int c = 0; c < nC; c++) A.push_back(pb->A[i + (size_t)c * nclin]);
            m++;
        }
    if (A.empty()) A.push_back(0.0);
    ntgb::newton::Structure S;
    ntgb::newton::build_structure(dm.nout, dm.nbps, pb->order.data(), pb->ncoef.data(), pb->hoff.data(), pb->cost_out,
                                  A.data(), m, S);
    if (S.w > ntgb::newton::kMaxHalfBand)
        return fail(NTGB_ELIMIT, "ntgb_solve_eq_newton: the Hessian's half-bandwidth %d is above the limit of %d", S.w,
                    ntgb::newton::kMaxHalfBand);
    int rc;
    if ((rc = dev_upload(pb, &nw.perm, S.perm.data(), S.perm.size())) ||
        (rc = dev_upload(pb, &nw.color, S.color.data(), S.color.size())) ||
        (rc = dev_upload(pb, &nw.hmask, S.hmask.data(), S.hmask.size())) ||
        (rc = dev_upload(pb, &nw.ata, S.ata.data(), S.ata.size())))
        return rc;
    nw.ata_max = 0.0;
    for (int i = 0; i < nC; i++) nw.ata_max = std::max(nw.ata_max, S.ata[(size_t)i * (S.w + 1)]);
    nw.K = S.K;
    nw.w = S.w;
    nw.hperm = S.perm;
    nw.ready = true;
    return 0;
}

/* ntgb_solve_eq_newton.  Per iteration: one evaluation at C, the convergence test, one evaluation of the 2K
 * difference points of every problem, the factor, the direction, two_stage_search on the cost and the update. */
int solve_newton_impl(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                      int *iters, int *status, const ntgb_newton_opts &o, void *stream)
{
    const ntgb_dims &dm = pb->dims;
    const int nC = dm.nC;
    int rc;
    if ((rc = check_eq_only(pb, "ntgb_solve_eq_newton"))) return rc;
    if ((rc = TwoStage::check_size(P))) return rc;
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = reduced_form(pb, false, true))) return rc;
    const auto &al = pb->alm;
    if (al.nr > 0 && al.r > ntgb::newton::kMaxRows)
        return fail(NTGB_ELIMIT,
                    "ntgb_solve_eq_newton: the equality rows span %d dimensions, above the limit of %d of the range-space "
                    "step (trajectory equality rows at many breakpoints exceed it)",
                    al.r, ntgb::newton::kMaxRows);
    if ((rc = newton_prepare(pb))) return rc;
    const auto &nw = pb->newton;
    if ((size_t)P * 2 * nw.K > 0x7fffffffull) return fail(NTGB_EINVAL, "P*2*ncolors too large");
    const size_t Pz = (size_t)P;
    const ntgb::newton::Desc D{nw.perm, nw.color, nw.hmask, nw.ata, al.Q1, nC, nw.w, nw.K, al.r, nw.ata_max};
    const BoundsDesc B{bounds_layout(pb), nC, 0, 0, dm.nclin, nullptr, nullptr, al.M, al.Ae};
    NewtonArrays S;
    TwoStage ts;
    BoundsArrays ba;
    double *g, *dC, *fv, *phi0, *dphi0;
    int *count;
    if ((rc = scratch_carve(pb->scratch.newton, st, [&](Carve &c) {
             S.take(c, Pz, nC, nw.K, nw.w, al.r);
             c.take(Pz * nC, g, dC);
             c.take(Pz, fv, phi0, dphi0);
             c.take(1, count);
             ts.take(c, Pz, dm);
             if (lowerb) ba.take(c, Pz, B);
         })))
        return rc;
    if ((rc = ts.start(P, st))) return rc;
    CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
    const double *Cpart = al.Cpart;
    int Cstride = 0;
    if (lowerb) {
        if ((rc = bounds_prepare(P, lowerb, upperb, B, ba, st, S.state, S.its, count))) return rc;
        Cpart = ba.Cpart;
        Cstride = nC;
    }
    const int nt = kNewtonThreads;
    const size_t win = sizeof(double) * (nw.w + 1) * (nw.w + 1);
    CUDA_TRY(launch(k_newton_init, (unsigned)P, nt, st, P, D, S, Cpart, Cstride, C));
    ntgb_eval_args a, ad;
    memset(&a, 0, sizeof a);
    a.P = P; a.C = C; a.mode_obj = 2; a.mode_con = -1; a.f = fv; a.g = g; a.jac_layout = NTGB_JAC_NONE; a.stream = st;
    ad = a;
    ad.P = P * 2 * nw.K; ad.C = S.Xp; ad.f = S.fp; ad.g = S.Gp;
    const long long npts = (long long)ad.P * nC;
    auto merit = [&](int n, int, const int *) -> int {
        CUDA_TRY(launch(k_cost_merit, (unsigned)((n + 255) / 256), 256, st, n, (const double *)ts.ft, ts.res));
        return 0;
    };
    const int max_iter = al.nr > 0 ? o.max_iter : 0; /* no free direction: k_newton_init has finished every problem */
    for (int it = 0; it < max_iter; it++) {
        if ((rc = ntgb_eval(pb, &a))) return rc;
        CUDA_TRY(launch(k_newton_check, (unsigned)P, nt, st, P, D, S, (const double *)fv, (const double *)g, o.gtol, count));
        if ((it + 1) % o.check_every == 0 && (rc = all_finished(count, P, st)) != 0) {
            if (rc < 0) return rc;
            break;
        }
        CUDA_TRY(launch(k_newton_points, (unsigned)((npts + 255) / 256), 256, st, P, nC, nw.K, (const int *)nw.color,
                        (const double *)C, S.Xp));
        if ((rc = ntgb_eval(pb, &ad))) return rc;
        {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)P);
            cfg.blockDim = dim3(nt);
            cfg.dynamicSmemBytes = win;
            cfg.stream = st;
            CUDA_TRY(cudaLaunchKernelEx(&cfg, k_newton_factor, P, D, S, (const double *)C));
        }
        CUDA_TRY(launch(k_newton_dir, (unsigned)P, nt, st, P, D, S, (const double *)fv, (const double *)g, dC, phi0, dphi0));
        if ((rc = two_stage_search(pb, P, C, dC, o.c1, phi0, dphi0, S.state, ts, st, merit))) return rc;
        CUDA_TRY(launch(k_newton_update, (unsigned)P, nt, st, P, D, S, Cpart, Cstride, o.c1, (const double *)fv,
                        (const double *)phi0, (const double *)dphi0, (const double *)ts.ab, (const double *)ts.pbest,
                        (const double *)dC, C, count));
    }
    if (f) {
        a.mode_obj = 0; a.f = f; a.g = nullptr;
        if ((rc = ntgb_eval(pb, &a))) return rc;
    }
    if (iters) CUDA_TRY(cudaMemcpyAsync(iters, S.its, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, S.state, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

} /* namespace */

extern "C" {

int ntgb_solve_nlp(ntgb_problem *pb, int P, double *C, double *f, double *viol_out, int *iters, int *status,
                   const ntgb_nlp_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_nlp: null argument");
    if (P <= 0) return 0;
    const ntgb_dims &dm = pb->dims;
    ntgb_nlp_opts o{40, 80, 1e-6, 1e-6, 10.0, 10.0, 1e4, 1e-4, 4};
    if (opts) {
        if (opts->max_outer > 0) o.max_outer = opts->max_outer;
        if (opts->max_inner > 0) o.max_inner = opts->max_inner;
        if (opts->gtol > 0.0) o.gtol = opts->gtol;
        if (opts->ctol > 0.0) o.ctol = opts->ctol;
        if (opts->rho0 > 0.0) o.rho0 = opts->rho0;
        if (opts->rho_mul > 1.0) o.rho_mul = opts->rho_mul;
        if (opts->rho_max > 0.0) o.rho_max = opts->rho_max;
        if (opts->c1 > 0.0) o.c1 = opts->c1;
        if (opts->check_every > 0) o.check_every = opts->check_every;
    }
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int nC = dm.nC, nclin = dm.nclin, ncnln = dm.ncnln;
    int rc;
    if ((rc = alm_prepare(pb))) return rc;
    auto &al = pb->alm;
    if (al.nr > kSolveMaxNr)
        return fail(NTGB_ELIMIT, "ntgb_solve_nlp: %d free directions after eliminating the linear equalities (limit %d)",
                    al.nr, kSolveMaxNr);
    const int nr = al.nr, m = al.m, n_li = al.n_li;
    if ((rc = TwoStage::check_size(P))) return rc;
    const size_t Pz = (size_t)P;
    const size_t mz = (size_t)std::max(m, 1), ncz = (size_t)std::max(ncnln, 1), nlz = (size_t)std::max(nclin, 1);
    double *y, *yp, *grp, *d, *H, *dC, *g, *gA, *lam, *mu, *cc, *J, *lin, *fv, *LA, *viol, *violp, *rho, *phi0, *dphi0;
    int *state, *its, *fails, *fin, *count;
    TwoStage ts;
    if ((rc = scratch_carve(pb->scratch.nlp, st, [&](Carve &c) {
             c.take(Pz * nr, y, yp, grp, d);
             c.take(Pz * nr * nr, H);
             c.take(Pz * nC, dC, g, gA);
             c.take(Pz * mz, lam, mu);
             c.take(Pz * ncz, cc);
             c.take(Pz * ncz * dm.sorder, J);
             c.take(Pz * nlz, lin);
             c.take(Pz, fv, LA, viol, violp, rho, phi0, dphi0, state, its, fails, fin);
             c.take(1, count);
             ts.take(c, Pz, dm);
         })))
        return rc;

    if ((rc = ts.start(P, st))) return rc;
    const unsigned grid = (unsigned)((P + 127) / 128);
    CUDA_TRY(launch(k_solve_init, grid, 128, st, P, nC, nr, al.N, al.Cpart, 0, C, y, H, state, its, fails));
    CUDA_TRY(launch(k_alm_prep, grid, 128, st, P, m, o.rho0, lam, rho, violp, fin));
    CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));

    ntgb_eval_args ea;
    memset(&ea, 0, sizeof ea);
    ea.P = P; ea.C = C; ea.mode_obj = 2; ea.mode_con = ncnln > 0 ? 2 : -1; ea.f = fv; ea.g = g; ea.c = cc; ea.J = J;
    ea.jac_layout = ncnln > 0 ? NTGB_JAC_BAND : NTGB_JAC_NONE; ea.stream = st;
    /* the search's merit: the augmented Lagrangian at the trial points */
    auto merit = [&](int n, int nalpha, const int *pidx) -> int {
        CUDA_TRY(launch(k_alm_mu, (unsigned)(((long long)n * 32 + 127) / 128), 128, st, n, nalpha, ncnln, nclin, n_li,
                        al.li_idx, al.hl, al.hu, lam, rho, ts.ft, ts.ct, ts.lint, (double *)nullptr, ts.res,
                        (double *)nullptr, 2, pidx));
        return 0;
    };

    auto assemble = [&]() -> int { /* f, g, c, J, lin at C -> mu, L_A, violation, grad L_A */
        int r2;
        if ((r2 = ntgb_eval(pb, &ea))) return r2;
        if (n_li > 0 && (r2 = ntgb_eval_linear(pb, P, C, lin, nullptr, st))) return r2;
        const unsigned gw = (unsigned)(((long long)P * 32 + 127) / 128);
        CUDA_TRY(launch(k_alm_mu, gw, 128, st, P, 1, ncnln, nclin, n_li, al.li_idx, al.hl, al.hu, lam, rho, fv, cc, lin, mu,
                        LA, viol, 1, (const int *)nullptr));
        const long long tot = (long long)P * nC;
        CUDA_TRY(launch(k_alm_grad, (unsigned)((tot + 127) / 128), 128, st, P, pb->tab, nclin, n_li, al.li_idx, al.A, g, J,
                        mu, gA));
        return 0;
    };

    for (int outer = 0; outer < o.max_outer; outer++) {
        for (int it = 0; it < o.max_inner; it++) {
            if ((rc = assemble())) return rc;
            CUDA_TRY(launch(k_solve_dir, grid, 128, st, P, nC, nr, al.N, LA, gA, o.gtol, y, yp, grp, H, d, dC, phi0, dphi0,
                            state, fails, count));
            if ((it + 1) % o.check_every == 0 && (rc = all_finished(count, P, st)) != 0) {
                if (rc < 0) return rc;
                break;
            }
            if ((rc = two_stage_search(pb, P, C, dC, o.c1, phi0, dphi0, state, ts, st, merit))) return rc;
            CUDA_TRY(launch(k_solve_update, grid, 128, st, P, nC, nr, al.N, al.Cpart, 0, phi0, ts.ab, ts.pbest, d, y, H, C,
                            state, its, fails, count));
        }
        /* round finished: fresh multipliers at the point reached, then the outer update */
        if ((rc = assemble())) return rc;
        CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
        CUDA_TRY(launch(k_alm_outer, grid, 128, st, P, m, nr, mu, lam, rho, viol, violp, o.ctol, o.rho_mul, o.rho_max,
                        outer + 1 == o.max_outer ? 1 : 0, H, state, fails, fin, count));
        if ((rc = all_finished(count, P, st)) != 0) {
            if (rc < 0) return rc;
            break;
        }
    }
    if (f) CUDA_TRY(cudaMemcpyAsync(f, fv, sizeof(double) * Pz, cudaMemcpyDeviceToDevice, st));
    if (viol_out) CUDA_TRY(cudaMemcpyAsync(viol_out, viol, sizeof(double) * Pz, cudaMemcpyDeviceToDevice, st));
    if (iters) CUDA_TRY(cudaMemcpyAsync(iters, its, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, fin, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

int ntgb_solve_sqp(ntgb_problem *pb, int P, double *C, double *f, double *viol_out, int *iters, int *status,
                   double *lambda, int *istate, const ntgb_sqp_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_sqp: null argument");
    return solve_sqp_impl(pb, Run::Sync, P, C, nullptr, nullptr, nullptr, f, viol_out, iters, status, lambda, istate, opts,
                          stream);
}

int ntgb_solve_sqp_bounds(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *f,
                          double *viol_out, int *iters, int *status, double *lambda, int *istate,
                          const ntgb_sqp_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_sqp_bounds: null argument");
    if (bounds_layout(pb).nb() > 0 && (!lowerb || !upperb))
        return fail(NTGB_EINVAL, "ntgb_solve_sqp_bounds: lowerb / upperb is NULL");
    return solve_sqp_impl(pb, Run::Sync, P, C, lowerb, upperb, nullptr, f, viol_out, iters, status, lambda, istate, opts,
                          stream);
}

int ntgb_sqp_warm_doubles(ntgb_problem *pb, size_t *n)
{
    if (!pb || !n) return fail(NTGB_EINVAL, "ntgb_sqp_warm_doubles: null argument");
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    int rc;
    if ((rc = sqp_prepare(pb, "ntgb_sqp_warm_doubles"))) return rc;
    *n = ntgb::warm_doubles(pb->alm.nr);
    return 0;
}

int ntgb_solve_sqp_warm(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *warm,
                        double *f, double *viol_out, int *iters, int *status, double *lambda, int *istate,
                        const ntgb_sqp_opts *opts, void *stream)
{
    if (!pb || !C || !warm) return fail(NTGB_EINVAL, "ntgb_solve_sqp_warm: null argument");
    if ((lowerb == nullptr) != (upperb == nullptr))
        return fail(NTGB_EINVAL, "ntgb_solve_sqp_warm: exactly one of lowerb / upperb is NULL");
    return solve_sqp_impl(pb, Run::Sync, P, C, lowerb, upperb, warm, f, viol_out, iters, status, lambda, istate, opts,
                          stream);
}

int ntgb_solve_sqp_reserve(ntgb_problem *pb, int P_max)
{
    if (!pb) return fail(NTGB_EINVAL, "ntgb_solve_sqp_reserve: null argument");
    if (P_max < 1) return fail(NTGB_EINVAL, "ntgb_solve_sqp_reserve: P_max = %d", P_max);
    return solve_sqp_impl(pb, Run::Reserve, P_max, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                          nullptr, nullptr, nullptr, nullptr);
}

int ntgb_solve_sqp_async(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb, double *warm,
                         double *f, double *viol_out, int *iters, int *status, double *lambda, int *istate,
                         const ntgb_sqp_opts *opts, void *stream)
{
    if (!pb || !C) return fail(NTGB_EINVAL, "ntgb_solve_sqp_async: null argument");
    if ((lowerb == nullptr) != (upperb == nullptr))
        return fail(NTGB_EINVAL, "ntgb_solve_sqp_async: exactly one of lowerb / upperb is NULL");
    return solve_sqp_impl(pb, Run::Async, P, C, lowerb, upperb, warm, f, viol_out, iters, status, lambda, istate, opts,
                          stream);
}

} /* extern "C" */

namespace {

/* ntgb_solve_sqp, ntgb_solve_sqp_bounds, ntgb_solve_sqp_warm and the reserve / async entry points (Run):
 * lowerb == nullptr = the setup's bounds for every problem; warm == nullptr = cold start, no state written back */
int solve_sqp_impl(ntgb_problem *pb, Run run, int P, double *C, const double *lowerb, const double *upperb, double *warm,
                   double *f, double *viol_out, int *iters, int *status, double *lambda, int *istate,
                   const ntgb_sqp_opts *opts, void *stream)
{
    if (P <= 0) return 0;
    AsyncWork &aw = pb->async.sqp;
    if (run == Run::Async && P > aw.P)
        return fail(NTGB_EINVAL, "ntgb_solve_sqp_async: P = %d above the %d problems reserved by ntgb_solve_sqp_reserve", P,
                    aw.P);
    const ntgb_dims &dm = pb->dims;
    ntgb_sqp_opts o{100, 1e-6, 1e-8, 1e4, 1e-4, 4};
    if (opts) {
        if (opts->max_iter > 0) o.max_iter = opts->max_iter;
        if (opts->gtol > 0.0) o.gtol = opts->gtol;
        if (opts->ctol > 0.0) o.ctol = opts->ctol;
        if (opts->rho_pen > 0.0) o.rho_pen = opts->rho_pen;
        if (opts->c1 > 0.0) o.c1 = opts->c1;
        if (opts->check_every > 0) o.check_every = opts->check_every;
    }
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int nC = dm.nC, nclin = dm.nclin, ncnln = dm.ncnln;
    int rc;
    if ((rc = sqp_prepare(pb, "ntgb_solve_sqp"))) return rc;
    const auto &al = pb->alm;
    const auto &sq = pb->sqp;
    const int nr = al.nr, m = al.m, n_li = al.n_li;
    /* one CTA per problem: 32 threads up to 31 reduced variables, 64 beyond */
    const int nt = nr < 32 ? 32 : 64;
    const size_t smem = sqp::sqp_smem_doubles(nr, m, nt) * sizeof(double) + sqp::sqp_smem_ints(nr, m, nt) * sizeof(int);
    if (smem > (size_t)pb->max_smem_optin)
        return fail(NTGB_ELIMIT,
                    "ntgb_solve_sqp: %d reduced variables x %d rows need %zu bytes of shared memory per problem (limit %d): "
                    "the dense reduced-space QP is meant for short horizons",
                    nr, m, smem, pb->max_smem_optin);
    if ((rc = TwoStage::check_size(P))) return rc;
    const size_t Pz = (size_t)P;
    const size_t mz = (size_t)std::max(m, 1), ncz = (size_t)std::max(ncnln, 1), nlz = (size_t)std::max(nclin, 1);
    SqpArrays S;
    double *dC, *g, *gL, *mu, *cc, *J, *lin, *fv, *phi0, *dphi0;
    int *state, *its, *count;
    TwoStage ts;
    const BoundsDesc B{bounds_layout(pb), nC, n_li, m, sq.me, al.li_idx, sq.eq_idx, al.M, al.Ae};
    BoundsArrays ba;
    auto layout = [&](Carve &c) {
        c.take(Pz * nr, S.y, S.sprev, S.grLold, S.grold, S.d);
        c.take(Pz * nr * nr, S.B);
        c.take(Pz * nC, dC, g, gL);
        c.take(Pz * mz, S.lam, mu, S.istate);
        c.take(Pz * ncz, cc);
        c.take(Pz * ncz * dm.sorder, J);
        c.take(Pz * nlz, lin);
        c.take(Pz * 8, S.scal, S.flag);
        c.take(Pz, fv, phi0, dphi0, state, its);
        c.take(1, count);
        ts.take(c, Pz, dm);
        if (run != Run::Sync) ba.take(c, Pz, B); /* the synchronous path takes these from the bounds' scratch */
    };
    if (run == Run::Reserve) {
        /* the limit every launch of k_sqp_step needs, raised to what the device offers: a reserve for a smaller
         * QP on another ntgb_problem cannot lower it below this one's */
        if (smem > 48 * 1024) {
            cudaFuncAttributes fa;
            CUDA_TRY(cudaFuncGetAttributes(&fa, k_sqp_step));
            CUDA_TRY(cudaFuncSetAttribute(k_sqp_step, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          pb->max_smem_optin - (int)fa.sharedSizeBytes));
        }
        return reserve_work(pb, aw, P, layout);
    }
    if ((rc = scratch_carve(run == Run::Sync ? pb->scratch.sqp : aw.s, st, layout, run == Run::Sync))) return rc;
    if (run == Run::Async) ts.alphas = pb->async.halving;

    SqpDesc D;
    D.nC = nC; D.nr = nr; D.m = m; D.n_li = n_li; D.nclin = nclin; D.ncnln = ncnln;
    D.N = al.N; D.ArN = sq.ArN; D.li_idx = al.li_idx; D.hl = al.hl; D.hu = al.hu;
    D.Cstride = 0; D.hstride = 0;
    D.gtol = o.gtol; D.ctol = o.ctol; D.rho_pen = o.rho_pen;
    const double *Cpart = al.Cpart;

    if ((rc = ts.start(P, st, run == Run::Sync))) return rc;
    CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
    if (lowerb) {
        if (run == Run::Sync && (rc = scratch_carve(pb->scratch.bnd, st, [&](Carve &c) { ba.take(c, Pz, B); }))) return rc;
        if ((rc = bounds_prepare(P, lowerb, upperb, B, ba, st, state, its, count))) return rc;
        Cpart = ba.Cpart;
        D.hl = ba.hl; D.hu = ba.hu;
        D.Cstride = nC; D.hstride = m;
    }
    const unsigned grid = (unsigned)((P + 127) / 128);
    const ntgb::WarmKey wk{nr, m, al.digest};
    CUDA_TRY(launch(k_sqp_init, grid, 128, st, P, D, S, Cpart, C, state, its, (const double *)warm, wk));
    if (run == Run::Sync && smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(k_sqp_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    ntgb_eval_args ea;
    memset(&ea, 0, sizeof ea);
    ea.P = P; ea.C = C; ea.mode_obj = 2; ea.mode_con = ncnln > 0 ? 2 : -1; ea.f = fv; ea.g = g; ea.c = cc; ea.J = J;
    ea.jac_layout = ncnln > 0 ? NTGB_JAC_BAND : NTGB_JAC_NONE; ea.stream = st;
    /* the search's merit: the L1 merit at the trial points */
    auto merit = [&](int n, int nalpha, const int *pidx) -> int {
        CUDA_TRY(launch(k_sqp_merit, (unsigned)(((long long)n * 32 + 127) / 128), 128, st, n, nalpha, D, S.scal, ts.ft,
                        ts.ct, ts.lint, ts.res, pidx));
        return 0;
    };

    auto direction = [&]() -> int { /* f, g, c, J, lin at C -> QP -> d, dC, merit and slope; finished problems counted */
        int r2;
        if ((r2 = ntgb_eval(pb, &ea))) return r2;
        if (n_li > 0 && (r2 = ntgb_eval_linear(pb, P, C, lin, nullptr, st))) return r2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)P);
        cfg.blockDim = dim3((unsigned)nt);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, k_sqp_step, P, pb->tab, D, S, (const double *)fv, (const double *)g, (const double *)cc,
                                    (const double *)J, (const double *)lin, dC, phi0, dphi0, state, count));
        return 0;
    };

    for (int it = 0; it <= o.max_iter; it++) {
        if ((rc = direction())) return rc;
        if (it == o.max_iter) break; /* the last pass only evaluates and tests convergence at the final point */
        if (run == Run::Sync && (it + 1) % o.check_every == 0 && (rc = all_finished(count, P, st)) != 0) {
            if (rc < 0) return rc;
            break;
        }
        if ((rc = two_stage_search(pb, P, C, dC, o.c1, phi0, dphi0, state, ts, st, merit, run == Run::Async))) return rc;
        CUDA_TRY(launch(k_sqp_update, grid, 128, st, P, D, S, Cpart, phi0, ts.ab, ts.pbest, C, state, its, count));
    }
    if (warm)
        CUDA_TRY(launch(k_sqp_warm_store, (unsigned)(((long long)P * 32 + 127) / 128), 128, st, P, S, wk, (const int *)state,
                        warm));
    if (lambda || istate) {
        /* gL = g - A_in' l_in - J' l_nl in the full space (k_alm_grad adds dh' mu: mu = -lambda) */
        const long long totm = (long long)P * mz;
        CUDA_TRY(launch(k_scale_copy, (unsigned)((totm + 255) / 256), 256, st, totm, -1.0, (const double *)S.lam, mu));
        const long long tot = (long long)P * nC;
        CUDA_TRY(launch(k_alm_grad, (unsigned)((tot + 127) / 128), 128, st, P, pb->tab, nclin, n_li, al.li_idx, al.A, g, J, mu, gL));
        CUDA_TRY(launch(k_sqp_outputs, grid, 128, st, P, D, S, sq.me, sq.eq_idx, sq.W, gL, (const int *)state, lambda, istate));
    }
    if (f) CUDA_TRY(cudaMemcpyAsync(f, fv, sizeof(double) * Pz, cudaMemcpyDeviceToDevice, st));
    if (viol_out) CUDA_TRY(cudaMemcpy2DAsync(viol_out, sizeof(double), S.scal + 3, 8 * sizeof(double), sizeof(double), Pz,
                                             cudaMemcpyDeviceToDevice, st));
    if (iters) CUDA_TRY(cudaMemcpyAsync(iters, its, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, state, sizeof(int) * Pz, cudaMemcpyDeviceToDevice, st));
    if (run == Run::Sync) CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

} /* namespace */

extern "C" {

int ntgb_peer_table_alloc(ntgb_problem *pb, size_t rows, double **table, unsigned char handle[64])
{
    if (!pb || !table || !handle || rows == 0) return fail(NTGB_EINVAL, "ntgb_peer_table_alloc: bad argument");
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    double *p = nullptr;
    CUDA_TRY(cudaMalloc((void **)&p, rows * 2 * sizeof(double)));
    CUDA_TRY(cudaMemset(p, 0, rows * 2 * sizeof(double)));
    cudaIpcMemHandle_t h;
    static_assert(sizeof(h) == 64, "CUDA IPC handles are 64 bytes");
    const cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(NTGB_ECUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(handle, &h, 64);
    *table = p;
    return 0;
}

int ntgb_peer_table_open(ntgb_problem *pb, const unsigned char handle[64], double **table)
{
    if (!pb || !table || !handle) return fail(NTGB_EINVAL, "ntgb_peer_table_open: null argument");
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void *p = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *table = static_cast<double *>(p);
    return 0;
}

int ntgb_peer_table_close(ntgb_problem *pb, double *table)
{
    if (!pb || !table) return 0;
    DeviceGuard dg(pb->device);
    CUDA_TRY(cudaIpcCloseMemHandle(table));
    return 0;
}

int ntgb_peer_table_free(ntgb_problem *pb, double *table)
{
    if (!pb || !table) return 0;
    DeviceGuard dg(pb->device);
    CUDA_TRY(cudaFree(table));
    return 0;
}

int ntgb_integrate(int rule, long long nchain, int n, const double *f, const double *t, double *I, void *stream)
{
    if (rule != NTGB_QUAD_FEULER && rule != NTGB_QUAD_BEULER && rule != NTGB_QUAD_TRAPEZOID)
        return fail(NTGB_EINVAL, "ntgb_integrate: unknown rule %d", rule);
    if (nchain <= 0) return 0;
    if (!f || !t || !I || n < 1) return fail(NTGB_EINVAL, "ntgb_integrate: null argument or n < 1");
    CUDA_TRY(launch(k_integrate, (unsigned)((nchain + 127) / 128), 128, (cudaStream_t)stream, rule, nchain, n, f, t, I));
    return 0;
}

int ntgb_spline_interp(ntgb_problem *pb, int P, const double *C, int nt, const double *t, double *out, void *stream)
{
    if (!pb || !C || !t || !out) return fail(NTGB_EINVAL, "ntgb_spline_interp: null argument");
    if (P <= 0 || nt <= 0) return 0;
    DeviceGuard dg(pb->device);
    if (!dg.ok) return fail(NTGB_ECUDA, "cannot select device %d", pb->device);
    InterpDesc D;
    D.nout = pb->dims.nout; D.nC = pb->dims.nC; D.nz = pb->dims.nz;
    for (int j = 0; j < D.nout; j++) {
        D.order[j] = pb->order[j]; D.mult[j] = pb->mult[j]; D.md[j] = pb->maxderiv[j];
        D.ninterv[j] = pb->ninterv[j]; D.ncoef[j] = pb->ncoef[j];
        D.iC[j] = pb->tab.iC[j]; D.iz[j] = pb->tab.iz[j];
        D.aug[j] = pb->daug[j]; D.knots[j] = pb->dknots[j];
    }
    const long long total = (long long)P * nt * D.nout;
    const int block = 128;
    CUDA_TRY(launch(k_spline_interp, (unsigned)((total + block - 1) / block), block, (cudaStream_t)stream, D, P, C, nt,
                    t, out));
    return 0;
}

} /* extern "C" */
