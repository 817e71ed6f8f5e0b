/*
 * ntg_b200.h -- C ABI of the B200-native batched collocation evaluator.
 *
 * This is the drop-in boundary for NTG's per-iterate hot path: everything
 * NPSOL's funobj/funcon callbacks compute in the reference
 * (src/ntg.c:274-371 and the cost/constraint/colloc/integrator/matrix code
 * under them), for P independent coefficient vectors in one launch.
 *
 * Plain C: pointers and sizes only, no torch / C++ types.  Device pointers are
 * ordinary CUDA device addresses; `stream` is a cudaStream_t passed as void*.
 *
 * Every entry point returns 0 on success or a negative NTGB_E* code;
 * ntgb_last_error() gives the message of the last failure on this thread.
 * There is no CPU fallback: without a CUDA device every compute entry fails
 * with NTGB_ECUDA.
 */
#ifndef NTG_B200_H_
#define NTG_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- active variables: identical to reference src/av.h:18-26 ------------- */
#ifndef _AV_H_
#define _AV_H_
#define AVINITIAL    0
#define AVTRAJECTORY 1
#define AVFINAL      2
typedef struct AVStruct {
    int output;
    int deriv;
} AV;
#endif

/* ---- callback surface: reference src/ntg.c:34-41, src/ntg.h:81-92 -------- */
typedef void (*ntg_nlicf_t)(int *mode, int *nstate, double *f, double **df, double **zp);
typedef void (*ntg_nltcf_t)(int *mode, int *nstate, int *i, double *f, double **df, double **zp);
typedef void (*ntg_nlfcf_t)(int *mode, int *nstate, double *f, double **df, double **zp);
typedef void (*ntg_icf_t)(int *mode, int *nstate, double *f, double *df, double **zp);
typedef void (*ntg_ucf_t)(int *mode, int *nstate, int *i, double *f, double *df, double **zp);
typedef void (*ntg_fcf_t)(int *mode, int *nstate, double *f, double *df, double **zp);

/*
 * Problem description = the setup subset of ntg()'s arguments, same names,
 * same meaning, same order (reference src/ntg.h:72-99, src/ntg.c:54-83).
 * Callbacks are the HOST addresses of functions that were also compiled as
 * device code in a registered callback pack (see ntgb_register_pack).
 */
typedef struct ntgb_setup {
    int nout;
    const double *bps;
    int nbps;
    const int *kninterv;
    const double *const *knots;
    const int *order;
    const int *mult;
    const int *maxderiv;

    int nlic; const double *const *lic;
    int nltc; const double *const *ltc;
    int nlfc; const double *const *lfc;

    int nnlic; ntg_nlicf_t nlicf;
    int nnltc; ntg_nltcf_t nltcf;
    int nnlfc; ntg_nlfcf_t nlfcf;

    int ninitialconstrav;    const AV *initialconstrav;
    int ntrajectoryconstrav; const AV *trajectoryconstrav;
    int nfinalconstrav;      const AV *finalconstrav;

    const double *lowerb; /* [nlic+nltc+nlfc+nnlic+nnltc+nnlfc], may be NULL */
    const double *upperb;

    int nicf; ntg_icf_t icf;
    int nucf; ntg_ucf_t ucf;
    int nfcf; ntg_fcf_t fcf;

    int ninitialcostav;    const AV *initialcostav;
    int ntrajectorycostav; const AV *trajectorycostav;
    int nfinalcostav;      const AV *finalcostav;
} ntgb_setup;

typedef struct ntgb_problem ntgb_problem; /* opaque */

/* sizes derived at create time (reference src/colloc.c:34-52, src/ntg.c:155-157) */
typedef struct ntgb_dims {
    int nout, nbps;
    int nC;      /* number of coefficients = NPSOL n                     */
    int nz;      /* sum_j maxderiv_j                                     */
    int nZ;      /* nz * nbps                                            */
    int nclin;   /* nlic + nltc*nbps + nlfc                              */
    int ncnln;   /* nnlic + nnltc*nbps + nnlfc                           */
    int sorder;  /* S = sum_j order_j = band width of one Jacobian row   */
    int device;  /* CUDA device ordinal the tables live on               */
    int band_tile; /* TB: breakpoints per tile of the band-compact Jacobian
                    * layout (NTGB_JAC_BAND); TB = nbps unless the horizon
                    * is split over a thread-block cluster                 */
} ntgb_dims;

/* Jacobian layouts for ntgb_eval */
#define NTGB_JAC_NONE  0
/* NPSOL layout: per problem column-major ncnln x nC, ldJ = ncnln
 * (reference src/ntg.c:217-220).  Only band entries are written; the caller
 * zeroes the buffer once, exactly as the reference's one-time calloc does. */
#define NTGB_JAC_DENSE 1
/* Band-compact: per problem ncnln x S values.  Trajectory rows are stored
 * breakpoint-fastest, in tiles of TB = ntgb_dims.band_tile breakpoints: with
 * t = bp / TB, n_t = min(TB, nbps - t*TB) breakpoints in tile t, the value of
 * (row = nnlic + m*nbps + bp, band slot s) is at
 *   Jb[p*ncnln*S + nnlic*S + t*nnltc*S*TB + (m*S + s)*n_t + (bp - t*TB)];
 * TB = nbps (one tile, Jb[... + (m*S + s)*nbps + bp]) for every horizon one CTA
 * covers; long horizons that a thread-block cluster splits use one tile per
 * CTA, so that each CTA streams ONE contiguous block of the problem's
 * Jacobian (DRAM and copy-engine efficiency, DESIGN.md section 4).
 * ntgb_band_index() below is the index function.
 * Initial rows r at Jb[p*ncnln*S + r*S + s]; final rows r at
 *   Jb[p*ncnln*S + (nnlic + nnltc*nbps)*S + r*S + s].
 * Band slot s = jk0[j] + k maps to column col0[row][j] + k (ntgb_pattern). */
#define NTGB_JAC_BAND  2

/* offset (in doubles, inside one problem's ncnln*S block) of band slot s of trajectory row
 * (constraint m, breakpoint bp) in the NTGB_JAC_BAND layout */
#ifdef __CUDACC__
__host__ __device__
#endif
static inline size_t ntgb_band_index(int nnlic, int nnltc, int S, int nbps, int band_tile, int m, int s, int bp)
{
    const int t = bp / band_tile;
    const int nt = nbps - t * band_tile < band_tile ? nbps - t * band_tile : band_tile;
    return (size_t)nnlic * S + (size_t)t * nnltc * S * band_tile + ((size_t)m * S + s) * nt + (size_t)(bp - t * band_tile);
}

/*
 * One batched evaluation.  All pointers are DEVICE pointers (or NULL to skip
 * an output).  mode_obj / mode_con follow NPSOL: 0 values, 1 derivatives,
 * 2 both, -1 skip that half entirely.
 */
typedef struct ntgb_eval_args {
    int P;               /* number of problems in the batch                    */
    const double *C;     /* [P][nC] coefficients, problem-major                */
    int mode_obj;
    int mode_con;
    int nstate;          /* forwarded to callbacks (NPSOL: 1 on first call)    */
    double *f;           /* [P]           objective (modes 0,2)                */
    double *g;           /* [P][nC]       objective gradient (modes 1,2)       */
    double *c;           /* [P][ncnln]    nonlinear constraints (modes 0,2)    */
    double *J;           /* Jacobian, layout jac_layout (modes 1,2)            */
    int jac_layout;
    double *Z;           /* [P][nZ] flat outputs and derivatives, or NULL      */
    double *result;      /* [P][2] = (objective, max nonlinear violation), or NULL */
    void *stream;        /* cudaStream_t                                       */
    int *abort_flag;     /* optional device int: set to 1 when any callback asks to stop by
                          * writing *mode = -1 (reference src/ntg.c:369: NPSOL then terminates);
                          * the caller zeroes it.  ntgb_eval_host manages its own and returns
                          * NTGB_EABORT.                                        */
    /* Fused multi-GPU gather (optional; npeers = 0 turns it off).  Problems are sharded over the
     * GPUs of a node and the only thing the ranks exchange is the 16 B/problem (objective,
     * violation) table.  Instead of a collective after the kernel, the evaluator's epilogue stores
     * each pair into EVERY rank's copy of the gathered table -- peer_result[r] (an array in device
     * memory) is rank r's table
     * [total problems][2], mapped into this process (ntgb_peer_table_open: CUDA IPC, NVLink peer
     * stores); this rank's rows start at peer_row0.  No NCCL kernel competes with the persistent
     * evaluator for SMs.  A rank may read its table once every rank's stream has been
     * synchronised (a barrier), exactly when it could have waited for an asynchronous collective. */
    int npeers;                   /* <= NTGB_MAXPEERS */
    int peer_row0;
    double *const *peer_result;   /* DEVICE array [npeers] of table pointers (kept out of the kernel
                                   * parameters: the evaluators are sensitive to their size) */
} ntgb_eval_args;
#define NTGB_MAXPEERS 8

/* error codes */
#define NTGB_OK        0
#define NTGB_EINVAL   -1  /* bad argument / shape contract violated            */
#define NTGB_ENOPACK  -2  /* callbacks not found in any registered device pack */
#define NTGB_ECUDA    -3  /* CUDA runtime failure (includes: no device)        */
#define NTGB_ELIMIT   -4  /* problem exceeds the pack's compile-time bounds    */
#define NTGB_ENOMEM   -5
#define NTGB_EABORT   -6  /* a callback set *mode = -1 (only from ntgb_eval_host)  */

const char *ntgb_last_error(void);
const char *ntgb_version(void);

int  ntgb_create(ntgb_problem **out, const ntgb_setup *setup, int device);
void ntgb_destroy(ntgb_problem *pb);
int  ntgb_get_dims(const ntgb_problem *pb, ntgb_dims *dims);

/* device buffers in, device buffers out, asynchronous on args->stream */
int  ntgb_eval(ntgb_problem *pb, const ntgb_eval_args *args);
/* same call with HOST buffers: H2D of C, launch, D2H of the requested outputs,
 * synchronous.  This is what ntg()'s funobj/funcon trampolines use.  Large batches are chunked
 * over two streams so copies overlap the kernels; calls that move less than 256 KB (an NPSOL
 * callback is P = 1) skip the copies: the kernel reads and writes one page-locked, device-mapped
 * staging block (NTG_B200_NO_ZEROCOPY=1 forces the copying path). */
int  ntgb_eval_host(ntgb_problem *pb, const ntgb_eval_args *host_args);

/* Page-locked host memory for ntgb_eval_host (so its copies are asynchronous and overlap the
 * kernels) without pulling CUDA headers into a C program; ntgb_host_register pins memory the
 * caller already owns. */
void *ntgb_host_alloc(size_t bytes);
void  ntgb_host_free(void *p);
int   ntgb_host_register(void *p, size_t bytes);
int   ntgb_host_unregister(void *p);

/*
 * One-time tables built on the device by K0 (replaces CollocMatrix + PGS,
 * reference src/colloc.c:57-117), copied back for inspection / parity:
 *   B      [sum_j nbps*order_j*maxderiv_j]  per output contiguous,
 *          index (bp*order_j + k)*maxderiv_j + d   (reference block layout)
 *   offset [nout*nbps]    block[bp].offset            (src/colloc.c:108)
 *   left   [nout*nbps]    interv() result on the augmented knots, 1-based
 * Any pointer may be NULL.
 */
int  ntgb_get_tables(const ntgb_problem *pb, double *B, int *offset, int *left);
/* augmented knot vector of output j (length n_j + order_j), host copy */
int  ntgb_get_augknots(const ntgb_problem *pb, int j, double *t, int *len);

/* Jacobian sparsity: col0[row*nout + j] = first column of output j's band in
 * that row (reference src/colloc.c:243-316); jk0[j] = band slot of (j,k=0). */
int  ntgb_get_pattern(const ntgb_problem *pb, int *col0, int *jk0);

/* Linear constraints (reference src/constraints.c:198-261, src/ntg.c:162-206):
 * A is nclin x nC column-major (ldA = nclin), host memory. */
int  ntgb_get_linear(const ntgb_problem *pb, double *A);
/* NPSOL bound vectors bl/bu of length nC+nclin+ncnln (src/constraints.c:5-33) */
int  ntgb_get_bounds(const ntgb_problem *pb, double *bl, double *bu);
/* batched A*C and linear violation on the device: lin [P][nclin], viol [P] */
int  ntgb_eval_linear(ntgb_problem *pb, int P, const double *C, double *lin,
                      double *viol, void *stream);

/* Batched SplineInterp (reference src/colloc.c:449-484): for every problem p
 * and time t[i], out[(p*nt + i)*nz + iz_j + d].  Device pointers. */
/*
 * Batched IntegrateVector / IntegrateFMatrixCols (/root/reference/src/integrator.c:16-62) with the
 * reference's three rules (src/integrator.h:19-21).  f holds nchain sample vectors of n values
 * ([nchain][n], e.g. nchain = P columns), t the n sample times; I[q] = the rule's sum over vector q,
 * accumulated in the reference's order with the reference's expression (bit-identical to it).  The
 * evaluator itself only ever integrates with TRAPEZOID, as every call site of the reference does
 * (src/cost.c:61,96,111,134); the other two rules are here for callers of the public helper.
 * Device pointers; runs on the current device.
 */
#define NTGB_QUAD_FEULER    0
#define NTGB_QUAD_BEULER    1
#define NTGB_QUAD_TRAPEZOID 2
int  ntgb_integrate(int rule, long long nchain, int n, const double *f, const double *t, double *I, void *stream);

int  ntgb_spline_interp(ntgb_problem *pb, int P, const double *C, int nt,
                        const double *t, double *out, void *stream);

/*
 * Batched merit line search -- first step towards a batched SQP consumer
 * (SURVEY.md section 8(f) rank 3; NPSOL's line search is serial and proprietary).
 * For every problem p and every trial step alpha[a] (device array, tried in the
 * given order) evaluates x = C[p] + alpha[a]*dC[p] in values-only mode, P*nalpha
 * evaluations in ONE launch of the evaluator, and the L-infinity merit
 *     phi = f + mu * max(max nonlinear violation, max linear violation).
 * Per problem it selects the first alpha with phi <= phi0[p] + c1*alpha*dphi0[p]
 * (Armijo; phi0/dphi0 device arrays, dphi0 may be NULL = plain decrease), else
 * the alpha of smallest phi.  Outputs (device, any may be NULL): alpha_best[P],
 * phi_best[P], C_new[P][nC] = C + alpha_best*dC.  Asynchronous on `stream`.
 */
int  ntgb_linesearch(ntgb_problem *pb, int P, const double *C, const double *dC, int nalpha,
                     const double *alpha, double mu, double c1, const double *phi0, const double *dphi0,
                     double *alpha_best, double *phi_best, double *C_new, void *stream);

/*
 * Batched solve for the class of problems both shipped examples belong to: no nonlinear
 * constraints and only EQUALITY linear constraints (examples/vanderpol.c:159-169,
 * examples/kincar.c:322-339).  Second step towards a batched SQP consumer (SURVEY.md
 * section 8(f) rank 3): every problem of the batch is minimised independently, entirely on the
 * GPU, by a reduced-space BFGS -- the linear constraints A*C = b are eliminated once on the host
 * (C = C_part + N*y with N an orthonormal null-space basis of A), each iteration is one batched
 * evaluation (cost + gradient), one tiny per-problem BFGS kernel and one batched Armijo line
 * search (ntgb_linesearch).  C [P][nC] (device) holds the initial guesses on entry and the
 * solutions on return; f [P], iters [P], status [P] (device, may be NULL) receive the final cost,
 * the iteration count and 1 = reduced gradient below gtol, 2 = no further decrease, 0 = max_iter.
 * Synchronous.  NTGB_EINVAL if the problem has nonlinear or inequality constraints.
 */
typedef struct ntgb_solve_opts {
    int max_iter;     /* default 200 */
    double gtol;      /* |reduced gradient|_inf <= gtol * max(1, |f|), default 1e-9 */
    double c1;        /* Armijo constant, default 1e-4 */
    int check_every;  /* host looks at the convergence counter every this many iterations, default 4 */
} ntgb_solve_opts;
int  ntgb_solve_eq(ntgb_problem *pb, int P, double *C, double *f, int *iters, int *status,
                   const ntgb_solve_opts *opts, void *stream);

/*
 * Batched solve of the GENERAL problem ntg() poses (src/ntg.c:162-253): linear equalities are
 * eliminated as in ntgb_solve_eq; linear inequalities and the nonlinear constraints
 * bl <= c(C) <= bu go into an augmented Lagrangian (Powell-Hestenes-Rockafellar form for two-sided
 * bounds) that is minimised per problem by the same reduced-space BFGS, multipliers and penalty
 * updated between rounds.  Every step is a batched kernel: evaluation with the band Jacobian,
 * multiplier / merit kernel, J^T*mu gather per gradient column, BFGS direction, batched Armijo line
 * search on the augmented Lagrangian (steps 1 .. 1/8 for every problem in one evaluation, steps
 * 2^-4 .. 2^-15 in a second one for the compacted list of problems that need them).  C [P][nC] (device): guesses in, solutions out.  f, viol
 * (maximum violation of any constraint), iters (evaluations of the inner loop), status
 * (1 = violation <= ctol and reduced gradient <= gtol, 2 = violation <= ctol and no further
 * decrease of the merit function possible, 0 = not converged) are optional device outputs.
 * Synchronous.  A local method with no globalisation beyond the line search: it returns a KKT
 * point near the guess, like the SQP solver it stands in for.
 */
typedef struct ntgb_nlp_opts {
    int max_outer;    /* multiplier updates, default 40 */
    int max_inner;    /* BFGS iterations per round, default 80 */
    double gtol;      /* reduced gradient of the augmented Lagrangian, relative to max(1,|L|); default 1e-6 */
    double ctol;      /* constraint violation, relative to max(1, |bound|); default 1e-6 */
    double rho0;      /* initial penalty, default 10 */
    double rho_mul;   /* penalty growth when the violation does not drop by 4x, default 10 */
    double rho_max;   /* penalty cap, default 1e4 (larger values make the inner problems ill-conditioned) */
    double c1;        /* Armijo constant, default 1e-4 */
    int check_every;  /* host reads the done counter every this many inner iterations, default 4 */
} ntgb_nlp_opts;
int  ntgb_solve_nlp(ntgb_problem *pb, int P, double *C, double *f, double *viol, int *iters, int *status,
                    const ntgb_nlp_opts *opts, void *stream);

/*
 * Batched SQP solver: what NPSOL does for the reference (/root/reference/src/ntg.c:250-253), for P
 * problems at once.  Linear equality rows are eliminated (C = C_part + N y); per iteration ONE
 * batched evaluation (cost, gradient, constraints, band Jacobian), then one CTA per problem solves
 * the dense QP subproblem on the reduced space in shared memory (Goldfarb-Idnani dual active set;
 * a Gauss-Newton step on the violated rows when the linearised rows are inconsistent), damped BFGS
 * on the reduced Lagrangian, Armijo search on the L1 merit (two batched values-only evaluations).
 * Outputs as NPSOL's (/root/reference/src/ntg.h:64-68): lambda / istate over the general
 * constraints in NPSOL's order [nclin linear rows ; ncnln nonlinear rows] (lambda > 0 at a lower
 * bound, < 0 at an upper one; istate 0 inactive, 1 lower, 2 upper, 3 equality); either may be NULL.
 * status: 1 converged (violation <= ctol, reduced Lagrangian gradient <= gtol*max(1,|f|)), 2 no
 * decrease of the merit function even from B = I, 4 stationary point of the violation (locally
 * infeasible), 0 iteration limit.  Limit: the per-problem work space (about 4 nr^2 + m nr doubles for
 * nr free directions and m rows) must fit in shared memory -- short horizons; NTGB_ELIMIT otherwise.
 */
typedef struct ntgb_sqp_opts {
    int max_iter;     /* SQP iterations, default 100 */
    double gtol;      /* default 1e-6 */
    double ctol;      /* default 1e-8 */
    double rho_pen;   /* Gauss-Newton weight of inconsistent rows, relative to trace(B)/nr / max |a_i|^2; default 1e4 */
    double c1;        /* Armijo constant, default 1e-4 */
    int check_every;  /* host reads the done counter every this many iterations, default 4 */
} ntgb_sqp_opts;
int  ntgb_solve_sqp(ntgb_problem *pb, int P, double *C, double *f, double *viol, int *iters, int *status,
                    double *lambda, int *istate, const ntgb_sqp_opts *opts, void *stream);

/*
 * Per-problem constraint bounds: one call solves P problems that share the setup's functions and
 * constraint rows but each have their own bounds -- e.g. a batch of MPC problems that start from
 * different states (the initial state is a linear equality row: lowerb == upperb == x0).
 *
 * lowerb / upperb are DEVICE arrays [P][nb], nb = nlic+nltc+nlfc+nnlic+nnltc+nnlfc: row p is problem
 * p's version of ntgb_setup.lowerb / upperb, compact like them (one value per trajectory constraint,
 * expanded over the breakpoints as ntgb_get_bounds does); |b| >= 1e19 means "no bound".  NULL with
 * nb > 0 is NTGB_EINVAL, returned before any CUDA call.  Everything else is as in ntgb_solve_eq /
 * ntgb_solve_sqp.
 *
 * The SETUP's bounds decide the structure: the linear rows with lower == upper there are the equality
 * rows that get eliminated (ntgb_solve_eq_bounds, like ntgb_solve_eq, refuses nonlinear and inequality
 * rows).  Each problem's bounds are checked on the device, per problem; the call does not fail for
 * them.  A problem is rejected when it has a NaN bound or lower > upper, when a row the setup
 * eliminates has lower != upper, or when its equality right-hand sides are inconsistent (possible only
 * if the setup's equality rows are dependent; residual > 1e-8 (1 + |b|_inf)).  A rejected problem gets
 * status NTGB_STATUS_BAD_BOUNDS, its C is left untouched bit for bit, iters is 0, viol is NaN and its
 * lambda / istate rows are 0; the other problems are solved as if it were absent.
 *
 * viol, status, lambda and istate (3 on eliminated rows, 1 / 2 on active rows) are measured against
 * each problem's own bounds.  Not so ntgb_eval's result[p][1] (max nonlinear violation), which keeps
 * using the setup's bounds.
 *
 * Cost: one extra kernel per call (k_bounds_prep, one warp per problem) and P*nC doubles of
 * per-problem C_part read by the solver kernels instead of one shared vector.
 */
#define NTGB_STATUS_BAD_BOUNDS 5
int  ntgb_solve_eq_bounds(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                          double *f, int *iters, int *status, const ntgb_solve_opts *opts, void *stream);
int  ntgb_solve_sqp_bounds(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                           double *f, double *viol, int *iters, int *status, double *lambda, int *istate,
                           const ntgb_sqp_opts *opts, void *stream);

/*
 * SQP warm start: solver state carried from one call to the next, for receding-horizon MPC (each step
 * re-solves nearly the same problem with its initial state moved) and real-time iteration (a fixed
 * small max_iter per control step).  The reduced space C = C_part + N y depends on the setup's linear
 * rows, not on the bounds, so the quasi-Newton Hessian B of the reduced Lagrangian in y stays
 * meaningful from one call to the next, with or without per-problem bounds.
 *
 * ntgb_sqp_warm_doubles: n, the doubles in one problem's row of warm-start state for this setup
 * (prepares the reduced form if needed).
 *
 * ntgb_solve_sqp_warm: ntgb_solve_sqp (lowerb == upperb == NULL) or ntgb_solve_sqp_bounds (both
 * non-NULL, as there) with solver state carried in warm (DEVICE, [P][n], in and out).  Exactly one of
 * lowerb / upperb NULL, or warm NULL, is NTGB_EINVAL before any CUDA call.
 *
 * One row of warm:
 *   - Rows are independent: row p belongs to problem p and nothing else.  Between calls rows may be
 *     copied, permuted, gathered or dropped with their problems (problems joining or leaving the
 *     fleet), and moved to another ntgb_problem created from the same setup (e.g. on another GPU).
 *   - Content: a header (format tag, nr, m, a 64-bit digest of the reduced form), then the merit
 *     weight nu and B as nr x nr (layout: ntg_b200/csrc/ntg_warm.h).
 *   - A row is used only if tag, nr, m and digest all match this setup.  Any other row -- all zeros,
 *     another setup's, garbage -- is a cold start: B = I, nu = 0, every output bit-identical to
 *     ntgb_solve_sqp / ntgb_solve_sqp_bounds.  From a matching row a NaN, infinite or negative nu is
 *     taken as 0 and B is read from its lower triangle; a B that is not positive definite is replaced
 *     by I.  No content of warm makes a call fail.
 *   - Warm start: B and nu from the row, no previous step.  If no step from it decreases the merit
 *     function, the solver restarts once from B = I as it does mid-solve.  The QP's working set is not
 *     warm-started; lambda / istate are outputs only.
 *   - On return every problem's row holds its B and nu of the last iteration, for status 0 (iteration
 *     limit), 1, 2 and 4.  Rows of problems with rejected bounds (NTGB_STATUS_BAD_BOUNDS) are left
 *     untouched bit for bit, like their C.  A call that fails before the end leaves warm unchanged.
 * Cost: nr^2 + 6 doubles per problem read once and written once per call.
 */
int  ntgb_sqp_warm_doubles(ntgb_problem *pb, size_t *n);
int  ntgb_solve_sqp_warm(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                         double *warm, double *f, double *viol, int *iters, int *status, double *lambda,
                         int *istate, const ntgb_sqp_opts *opts, void *stream);

/*
 * Stream-ordered solvers, for a fixed small number of iterations per control step (real-time iteration):
 * the call queues its work on `stream` and returns.  It synchronizes nothing, copies nothing to or from
 * the host, allocates nothing and sets no kernel attribute, so a whole control step can be recorded in
 * a CUDA graph (cudaStreamBeginCapture ... cudaStreamEndCapture) and replayed, or queued behind and
 * beside other GPU work.  Full solves stay with the synchronous entry points.
 *
 * ntgb_solve_eq_reserve / ntgb_solve_sqp_reserve: the one-time host work (the reduced form, the step
 * table and, for SQP, the QP kernel's shared-memory limit) and a work space for up to P_max problems.
 * They refuse what ntgb_solve_eq / ntgb_solve_sqp refuse, with the same code and message (nonlinear or
 * inequality rows for eq, too many free directions, QP work space above the shared memory: NTGB_ELIMIT,
 * no free direction).  They may synchronize the device and allocate.  Reserving again with a larger
 * P_max replaces the work space: graphs captured before must be captured again.  The work space
 * belongs to the async entry point alone, apart from what the synchronous calls use, so no synchronous
 * call on the same ntgb_problem -- one that grows its own scratch included -- invalidates a graph.
 * A synchronous ntgb_solve_sqp* call sets the QP kernel's shared-memory limit to what its own problem
 * needs: after one on ANOTHER ntgb_problem, call ntgb_solve_sqp_reserve again before the next async
 * call or replay.
 *
 * ntgb_solve_eq_async / ntgb_solve_sqp_async: arguments and outputs as in the synchronous entry points.
 * lowerb and upperb are both NULL (the setup's bounds) or both set (per-problem bounds, as in
 * ntgb_solve_*_bounds); warm is NULL (no state carried) or a [P][ntgb_sqp_warm_doubles] array (as in
 * ntgb_solve_sqp_warm); lambda, istate and the other outputs may be NULL.  The call runs EXACTLY
 * opts->max_iter iterations (default 100 for SQP, 200 for eq); check_every is ignored.  A finished
 * problem is inert in every solver kernel, so each output -- C, f, viol, iters, status, lambda, istate,
 * the warm rows, and problems with rejected bounds left untouched -- is bit-identical to the synchronous
 * call with the same arguments.  That call stops once every problem has finished; an async call pays for
 * all max_iter iterations even then.  The SQP line search evaluates the 16 steps 1 .. 2^-15 of every
 * problem in one batch (the synchronous one evaluates 4 steps, then 12 more only for the problems that
 * need them), and picks the same step.
 *
 * P above the reserved P_max, or no reserve yet, is NTGB_EINVAL before any CUDA call; so is exactly
 * one of lowerb / upperb NULL.  P == 0 returns 0.  An ntgb_problem runs one async call per solver at a
 * time: async calls on different streams must be ordered by the caller (an event), since they share
 * the work space.
 */
int  ntgb_solve_eq_reserve(ntgb_problem *pb, int P_max);
int  ntgb_solve_eq_async(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                         double *f, int *iters, int *status, const ntgb_solve_opts *opts, void *stream);
int  ntgb_solve_sqp_reserve(ntgb_problem *pb, int P_max);
int  ntgb_solve_sqp_async(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                          double *warm, double *f, double *viol, int *iters, int *status, double *lambda,
                          int *istate, const ntgb_sqp_opts *opts, void *stream);

/*
 * Long horizons: the problem class of ntgb_solve_eq (a smooth cost, only EQUALITY linear constraints, no
 * nonlinear ones) with any number of free directions.  Projected L-BFGS: no null-space basis is formed.
 * The projector onto null(A) is P v = v - Q1 (Q1' v), Q1 the nC x r orthonormal basis of the equality
 * rows' span from the same pivoted QR that ntgb_solve_eq uses.  C is projected onto each problem's affine
 * set at entry and after every accepted step, so A C = b holds to rounding throughout.  Per iteration:
 * one batched evaluation (cost + gradient), one CTA per problem for the projected gradient, the curvature
 * pair (s = the step taken, u = the change of P g; skipped when s'u <= 1e-10 |s| |u|), the two-loop
 * recursion with H0 = (s'u / u'u) I of the newest pair, and d = -P (H P g) (the history is dropped and
 * d = -P g when d'g >= 0), then the two-stage Armijo search of ntgb_solve_sqp on the cost (steps 1 .. 1/8
 * for every problem, 2^-4 .. 2^-15 for the rest).  Each reduction has a fixed order that depends on nC
 * alone: results do not depend on the batch size or order.
 *
 * Arguments and outputs as in ntgb_solve_eq_bounds: lowerb / upperb both NULL (the setup's bounds) or both
 * set (DEVICE [P][nb] per-problem bounds); exactly one NULL is NTGB_EINVAL before any CUDA call, and so is
 * opts->memory outside 1..32.  opts may be NULL (every default); in a non-NULL opts, a max_iter, gtol, c1
 * or check_every <= 0 takes its default.  status: 1 |P g|_inf <= gtol max(1, |f|), 2 no further decrease
 * (also from steepest descent) or a NaN gradient, 0 iteration limit, NTGB_STATUS_BAD_BOUNDS rejected bounds
 * (C left untouched bit for bit, iters 0).  Refusals as in ntgb_solve_eq (nonlinear or inequality rows:
 * NTGB_EINVAL).  Linear equalities that leave no free direction give C = C_part, status 1 and iters 0, as
 * ntgb_solve_eq does.  There is no limit on free directions.  Synchronous.
 *
 * Work space (device, kept between calls, freed by ntgb_destroy): about
 *     P (2 memory + 16 + 4) nC + r nC  doubles
 * (the curvature pairs, the 16 trial points of the search, the gradient, direction, last step and last
 * projected gradient; Q1), plus nC per problem with per-problem bounds.  Nothing of size nC x nC or
 * nC x (nC - r) is on the device.  The host builds the dense nC x nC Q of the QR once per setup.
 */
typedef struct ntgb_lbfgs_opts {
    int max_iter;     /* default 500 */
    double gtol;      /* |P g|_inf <= gtol * max(1, |f|), default 1e-9 */
    double c1;        /* Armijo constant, default 1e-4 */
    int memory;       /* curvature pairs kept per problem, 1..32, default 8 */
    int check_every;  /* host reads the done counter every this many iterations, default 4 */
} ntgb_lbfgs_opts;
int  ntgb_solve_eq_lbfgs(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                         double *f, int *iters, int *status, const ntgb_lbfgs_opts *opts, void *stream);

/*
 * Long horizons with a Newton method: the problem class of ntgb_solve_eq_lbfgs (a smooth cost, only EQUALITY
 * linear constraints, no nonlinear ones, any number of free directions), with an iteration count that does not
 * grow with the horizon.
 *
 * Structure (host, once per setup; ntgb_newton_structure reports it).  A breakpoint touches only order_j
 * coefficients of each output, so the cost's Hessian H couples exactly the coefficients of the outputs in its
 * active-variable lists that share a breakpoint.  The columns are ordered by the first breakpoint that touches
 * them (ties by output): then H + A'A is a band of half-bandwidth w, independent of the horizon.  A greedy
 * distance-2 colouring of H's pattern (no two columns of one colour share a row) gives K colours.
 *
 * Per iteration: one batched evaluation (cost + gradient) and the test |P g|_inf <= gtol max(1, |f|), P the
 * projector onto null(A) (as in ntgb_solve_eq_lbfgs); then ONE batched gradient evaluation of the 2K points
 * C +- h e_k (central differences on colour k, h_c = eps^(1/3) max(1, |C_c|)), from which each problem's band of
 * H is recovered; M = H + rho A'A + tau I with rho = max diag H / max diag A'A and tau a per-problem
 * Levenberg-Marquardt shift; a banded Cholesky of M (O(nC w^2)); the range-space step
 * d = -M^-1 (g + Q1' lam), S lam = -Q1 M^-1 g, S = Q1 M^-1 Q1' (r x r, Q1 the orthonormal basis of the equality
 * rows' span, r its dimension); the two-stage Armijo search on the cost with a rounding allowance of
 * 8 eps |f|; the step projected onto the affine set again.  The shift: tau = tau / 4 after a unit step,
 * max(4 tau, beta) after a step below 1/4, a failed search or a nonpositive pivot (then refactored, up to 8
 * times, before the direction falls back to -P g), beta = 1e-3 max diag (H + rho A'A); tau starts at 0.
 * Stopping: status 1 by the gradient test; status 2 after two consecutive iterations without a strict decrease
 * of the cost (the cost no longer resolves a decrease: the rounding floor) or at a NaN gradient; status 0 at
 * max_iter.  Each reduction has a fixed order: results do not depend on the batch size or order.
 *
 * Arguments, outputs and refusals as in ntgb_solve_eq_lbfgs: lowerb / upperb both NULL or both DEVICE [P][nb];
 * exactly one NULL is NTGB_EINVAL before any CUDA call; opts may be NULL (every default), a field <= 0 takes its
 * default; status 1, 2, 0 or NTGB_STATUS_BAD_BOUNDS (C left untouched bit for bit, iters 0); nonlinear or
 * inequality rows are NTGB_EINVAL; no free direction gives C = C_part, status 1 and iters 0.  Limits
 * (NTGB_ELIMIT): r <= 128 (trajectory equality rows at many breakpoints can exceed it) and w <= 64.
 * Synchronous.
 *
 * Work space (device, kept between calls, freed by ntgb_destroy): about
 *     P (4K + w + r + 24) nC + P r^2  doubles
 * (the 2K difference points and their gradients, the band, M^-1 [g, Q1'], the 16 trial points of the search and
 * a handful of vectors; S), plus r nC for Q1 and nC per problem with per-problem bounds.  Nothing of size
 * nC x nC is on the device.
 */
typedef struct ntgb_newton_opts {
    int max_iter;     /* default 100 */
    double gtol;      /* |P g|_inf <= gtol * max(1, |f|), default 1e-9 */
    double c1;        /* Armijo constant, default 1e-4 */
    int check_every;  /* host reads the done counter every this many iterations, default 4 */
} ntgb_newton_opts;
int  ntgb_solve_eq_newton(ntgb_problem *pb, int P, double *C, const double *lowerb, const double *upperb,
                          double *f, int *iters, int *status, const ntgb_newton_opts *opts, void *stream);
/* the structure ntgb_solve_eq_newton uses for this setup: K colours (2K gradient evaluations per Hessian), the
 * half-bandwidth w and perm [nC] (perm[i] = the column at band position i; may be NULL).  NTGB_ELIMIT when
 * w > 64.  Use K, w and r (nC minus the free directions) to size the work space above. */
int  ntgb_newton_structure(ntgb_problem *pb, int *ncolors, int *half_bandwidth, int *perm);

/* Gathered result tables for the fused multi-GPU gather (ntgb_eval_args.peer_result): alloc creates
 * this rank's table (rows x 2 doubles, zeroed) and the 64-byte CUDA IPC handle the other ranks
 * need; open maps another rank's table into this process (peer access over NVLink is enabled on
 * first use); close unmaps it; free releases an own table. */
int  ntgb_peer_table_alloc(ntgb_problem *pb, size_t rows, double **table, unsigned char handle[64]);
int  ntgb_peer_table_open(ntgb_problem *pb, const unsigned char handle[64], double **table);
int  ntgb_peer_table_close(ntgb_problem *pb, double *table);
int  ntgb_peer_table_free(ntgb_problem *pb, double *table);

/* ---- callback packs ------------------------------------------------------ */
/*
 * A pack is a shared object produced by tools/ntg_pack.py from a user's
 * UNMODIFIED C file: the callbacks are compiled a second time as __device__
 * code and the fused evaluator is instantiated on them.  Its static
 * initialiser calls ntgb_register_pack().  Lookup is by the callbacks' host
 * addresses, so an unchanged ntg(..., ucf, ...) call finds its kernel.
 */
struct ntgb_launch; /* internal, see ntg_b200/csrc/ntg_kernel_args.h */
typedef struct ntgb_pack {
    const char *name;
    ntg_icf_t   icf;
    ntg_ucf_t   ucf;
    ntg_fcf_t   fcf;
    ntg_nlicf_t nlicf;
    ntg_nltcf_t nltcf;
    ntg_nlfcf_t nlfcf;
    /* compile-time shape of the kernel: nout and maxderiv[] are EXACT (the
     * callbacks hard-code zp[j][d] and the df index layout), order is a bound,
     * constraint counts are exact when the kind is enabled */
    int max_nout, max_maxderiv, max_order;
    int max_nnlic, max_nnltc, max_nnlfc;
    int maxderiv[8];
    int exact;  /* 1: reference operation order, no FMA contraction */
    int (*launch)(const struct ntgb_launch *);
    int abi;    /* NTGB_KERNEL_ABI the pack was built against (ntg_kernel_args.h): a pack built
                 * from an older header is refused at registration */
} ntgb_pack;

int ntgb_register_pack(const ntgb_pack *pack);
const ntgb_pack *ntgb_find_pack(const char *name);
int ntgb_num_packs(void);

#ifdef __cplusplus
}
#endif
#endif /* NTG_B200_H_ */
