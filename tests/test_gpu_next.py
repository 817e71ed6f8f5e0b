"""GPU tests for the rows SURVEY.md section 8(f) marks "next": linear constraints
(A*C, bounds, violation), batched SplineInterp, and the ntg() drop-in driven by
the same fake NPSOL that drives the reference."""
import ctypes as C
import os

import numpy as np
import pytest

from common import GOLDEN, assert_bitexact, assert_close, golden_module, golden_spec, load_golden
from ntg_b200 import configs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["cfg2_vanderpol", "cfg3_kincar", "endpoint"])
def test_linear_constraints_batched(port, name):
    """A*C per problem equals the oracle's A (reference LinearConstraintsMatrix,
    src/constraints.c:198-261) applied on the host; violation against bounds()"""
    import torch
    from ntg_b200 import Problem
    spec, X = golden_spec(name)
    o = port.eval(spec, X, dense=False, band=False, linear=True)
    pb = Problem(spec, 0)
    lin, viol = pb.eval_linear(torch.from_numpy(X).cuda())
    want = X @ o["A"].T
    assert_close(lin.cpu().numpy(), want, "A*C")
    lb, ub = o["bl"][spec.nC:spec.nC + spec.nclin], o["bu"][spec.nC:spec.nC + spec.nclin]
    lin_h = lin.cpu().numpy()
    v = np.maximum(np.maximum(lb - lin_h, lin_h - ub), 0).max(axis=1)
    assert_bitexact(viol.cpu().numpy(), v, "linear violation")
    pb.close()


def test_spline_interp_batched(port):
    """reference SplineInterp (src/colloc.c:449-484) at arbitrary times, incl. both ends,
    interior knots and a point past the last knot"""
    import torch
    from ntg_b200 import Problem
    spec = configs.endpoint()
    rng = np.random.default_rng(9)
    X = rng.uniform(-2, 2, (5, spec.nC))
    t = np.concatenate([[0.0, 0.5, 0.8, 1.25, 2.0, 2.0000000000000004], rng.uniform(0, 2, 20)])
    pb = Problem(spec, 0)
    out = pb.spline_interp(torch.from_numpy(X).cuda(), torch.from_numpy(t).cuda()).cpu().numpy()
    iC = np.concatenate([[0], np.cumsum(spec.ncoef)])
    iz = np.concatenate([[0], np.cumsum(spec.maxderiv)])
    for p in range(X.shape[0]):
        for i, ti in enumerate(t):
            for j in range(spec.nout):
                f = port.spline_interp(ti, spec.knots[j], X[p, iC[j]:iC[j + 1]], spec.order[j],
                                       spec.mult[j], spec.maxderiv[j])
                assert_bitexact(out[p, i, iz[j]:iz[j + 1]], f, f"p={p} t={ti} output {j}")
    pb.close()


def test_single_point_SplineInterp_dropin(port):
    from ntg_b200 import build
    lib = C.CDLL(build.CORE_SO)
    dp = C.POINTER(C.c_double)
    knots = np.array([0.0, 2.5, 5.0])
    coefs = np.random.default_rng(4).uniform(-1, 1, 7)
    for x in (0.0, 1.7, 2.5, 5.0):
        f = np.zeros(3)
        lib.SplineInterp(f.ctypes.data_as(dp), C.c_double(x), knots.ctypes.data_as(dp), 2,
                         coefs.ctypes.data_as(dp), 7, 5, 3, 3)
        assert_bitexact(f, port.spline_interp(x, knots, coefs, 5, 3, 3), f"x={x}")


@pytest.mark.parametrize("example", ["vanderpol", "kincar"])
def test_reference_examples_drop_in(example):
    """examples/vanderpol.c and examples/kincar.c, UNMODIFIED, compiled against
    include/ntg.h with their callbacks as __device__ functions, linked against
    libntg_b200.so: main() runs, calls ntg(), which hands NPSOL (here: the same
    fake npsol_ that drives the reference) GPU-backed funobj/funcon.  Outputs must
    match the fixture produced by the reference's own build of the same program."""
    from ntg_b200 import build, problem
    from oracle import oracle
    so = build.pack_so(f"ref_{example}")
    if not os.path.exists(so):
        pytest.skip("drop-in example packs are built where /root/reference exists")
    lib = problem.load_pack(f"ref_{example}")
    main = C.cast(getattr(lib, f"ntg_example_{example}_main"), C.c_void_p).value
    g = load_golden(f"example_{example}")
    cwd = os.getcwd()
    import tempfile
    with tempfile.TemporaryDirectory() as td:   # vanderpol.c writes its solution to ./coef1
        os.chdir(td)
        try:
            r = oracle.run_product_main(main, g["X"])
        finally:
            os.chdir(cwd)
    assert r["calls"] == 1, "ntg() did not reach npsol_"
    assert [r["n"], r["nclin"], r["ncnln"]] == list(g["dims"])
    assert_bitexact(r["A"], g["A"], "linear constraint matrix handed to NPSOL")
    assert_bitexact(r["bl"], g["bl"], "bl")
    assert_bitexact(r["bu"], g["bu"], "bu")
    # vanderpol's ucf calls pow(); device pow is within 2 ulp of glibc's
    assert_close(r["f"], g["f"], "objective")
    assert_close(r["g"], g["g"], "gradient")


def test_ntg_dropin_with_constraints_dense_jacobian(port):
    """ntg() with nonlinear constraints: NPSOL's funcon gets c and the dense column-major
    Jacobian (ldJ = ncnln) exactly as the reference's NPfuncon fills it."""
    from ntg_b200 import build, problem
    from ntg_b200.abi import BuiltSetup
    from oracle import oracle
    spec, X = golden_spec("endpoint")
    o = port.eval(spec, X, dense=True, band=False, linear=True)
    lib = problem.load_pack("endpt")
    bs = BuiltSetup(spec, lambda role, sym: C.cast(getattr(lib, sym), C.c_void_p).value)
    s = bs.struct
    core = problem.core()
    shim = C.CDLL(oracle.SHIM_SO, mode=C.RTLD_GLOBAL)

    # a main() that forwards the prepared setup to ntg()
    n = spec.nC
    istate = (C.c_int * (n + spec.nclin + spec.ncnln))()
    clambda = (C.c_double * (n + spec.nclin + spec.ncnln))()
    R = (C.c_double * ((n + 1) * (n + 1)))()
    inform, obj = C.c_int(0), C.c_double(0.0)
    x0 = (C.c_double * n)()

    @C.CFUNCTYPE(C.c_int, C.c_int, C.POINTER(C.c_char_p))
    def main(argc, argv):
        core.ntg.restype = None
        core.ntg(s.nout, s.bps, s.nbps, s.kninterv, s.knots, s.order, s.mult, s.maxderiv, x0,
                 s.nlic, s.lic, s.nltc, s.ltc, s.nlfc, s.lfc,
                 s.nnlic, C.c_void_p(s.nlicf), s.nnltc, C.c_void_p(s.nltcf), s.nnlfc, C.c_void_p(s.nlfcf),
                 s.ninitialconstrav, s.initialconstrav, s.ntrajectoryconstrav, s.trajectoryconstrav,
                 s.nfinalconstrav, s.finalconstrav, s.lowerb, s.upperb,
                 s.nicf, C.c_void_p(s.icf), s.nucf, C.c_void_p(s.ucf), s.nfcf, C.c_void_p(s.fcf),
                 s.ninitialcostav, s.initialcostav, s.ntrajectorycostav, s.trajectorycostav,
                 s.nfinalcostav, s.finalcostav, istate, clambda, R, C.byref(inform), C.byref(obj))
        return 0

    r = oracle.run_product_main(C.cast(main, C.c_void_p).value, X, ncnln=spec.ncnln)
    assert r["calls"] == 1 and (r["n"], r["nclin"], r["ncnln"]) == (spec.nC, spec.nclin, spec.ncnln)
    assert_close(r["f"], o["f"], "f")
    assert_close(r["g"], o["g"], "g")
    assert_close(r["c"], o["c"], "c")
    assert_close(r["Jdense"], np.nan_to_num(o["Jdense"], nan=0.0), "dense Jacobian as NPSOL sees it")
    assert_bitexact(r["A"], o["A"], "A")


_NTG_NO_NPSOL_CODE = r"""
import ctypes as C, sys
sys.path.insert(0, %r)
from ntg_b200 import problem, configs
from ntg_b200.abi import BuiltSetup
spec = configs.vanderpol(20, constraints=%s)
lib = problem.load_pack("vdp")
s = BuiltSetup(spec, lambda role, sym: C.cast(getattr(lib, sym), C.c_void_p).value).struct
core = problem.core()
n = spec.nC
inform, obj = C.c_int(0), C.c_double(0.0)
x0 = (C.c_double * n)(*([1.0] * n))
ntot = n + spec.nclin + spec.ncnln
istate, clambda = (C.c_int * ntot)(*([-99] * ntot)), (C.c_double * ntot)()
core.ntg.restype = None
core.ntg(s.nout, s.bps, s.nbps, s.kninterv, s.knots, s.order, s.mult, s.maxderiv, x0,
         s.nlic, s.lic, s.nltc, s.ltc, s.nlfc, s.lfc, 0, None, s.nnltc, C.c_void_p(s.nltcf), 0, None,
         0, None, s.ntrajectoryconstrav, s.trajectoryconstrav, 0, None,
         s.lowerb, s.upperb, 0, None, 1, C.c_void_p(s.ucf), 0, None, 0, None,
         s.ntrajectorycostav, s.trajectorycostav, 0, None,
         istate, clambda, (C.c_double * ((n + 1) ** 2))(),
         C.byref(inform), C.byref(obj))
print("INFORM", inform.value)
print("ISTATE", " ".join(str(v) for v in istate))
print("CLAMBDA", " ".join("%%.17g" %% v for v in clambda))
print("OBJ %%.17g" %% obj.value)
print("X", " ".join("%%.17g" %% v for v in x0))
"""


def _run_ntg_no_npsol(constraints, env=None):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, "-c", _NTG_NO_NPSOL_CODE % (root, constraints)], capture_output=True,
                       text=True, timeout=300, env=e)
    return p.stdout, p.stderr


def test_ntg_without_npsol_reports_it():
    """NPSOL absent and the built-in solvers switched off -> ntg() sets up on the GPU, says so,
    sets inform, solves nothing."""
    for constraints in (True, False):
        out, err = _run_ntg_no_npsol(constraints, {"NTG_B200_NO_BUILTIN_SOLVER": "1"})
        assert "INFORM -1000" in out, out + err
        assert "NPSOL" in err


def test_ntg_without_npsol_solves_constrained_problems(port):
    """NPSOL absent, van der Pol with the nonlinear input constraint |u| <= 2 (pack VDP-C): ntg()
    falls back to the built-in SQP solver and returns a KKT point -- feasible, and stationary by the
    ORACLE's gradient and Jacobian with the multipliers ntg() hands back in NPSOL's clambda / istate
    layout (/root/reference/src/ntg.h:64-68)."""
    out, err = _run_ntg_no_npsol(True)
    lines = dict(l.split(" ", 1) for l in out.strip().splitlines() if " " in l)
    assert int(lines["INFORM"]) == 0, out + err
    assert "SQP solver" in err and "istate and clambda are set" in err
    x = np.array([float(v) for v in lines["X"].split()])
    spec = configs.vanderpol(20, constraints=True)
    o = port.eval(spec, x[None, :], mode_obj=2, mode_con=2, dense=False, band=False, linear=True)
    nC = spec.nC
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    assert np.abs(A @ x - b).max() < 1e-9
    lb, ub = o["bl"][nC + spec.nclin:], o["bu"][nC + spec.nclin:]
    assert (o["c"][0] >= lb - 2e-6).all() and (o["c"][0] <= ub + 2e-6).all()
    assert abs(float(lines["OBJ"]) - o["f"][0]) <= 1e-12 * abs(o["f"][0])
    ist = np.array([int(v) for v in lines["ISTATE"].split()])
    lam = np.array([float(v) for v in lines["CLAMBDA"].split()])
    assert ist.size == nC + spec.nclin + spec.ncnln and (ist[:nC] == 0).all() and (lam[:nC] == 0).all()
    assert (ist[nC:nC + spec.nclin] == 3).all(), "the linear rows of van der Pol are equalities"
    d = port.eval(spec, x[None, :], mode_obj=2, mode_con=2, dense=True, band=False)
    Jd = np.nan_to_num(d["Jdense"][0], nan=0.0)
    Jd = Jd.T if Jd.shape[0] == nC and Jd.shape[1] != nC else Jd
    r = o["g"][0] - A.T @ lam[nC:nC + spec.nclin] - Jd.T @ lam[nC + spec.nclin:]
    assert np.abs(r).max() <= 1e-5 * max(1.0, np.abs(o["g"][0]).max()), np.abs(r).max()
    sn, ln = ist[nC + spec.nclin:], lam[nC + spec.nclin:]
    assert set(np.unique(sn)) <= {0, 1, 2}
    assert (np.abs(o["c"][0] - lb)[sn == 1] <= 1e-6).all() and (np.abs(o["c"][0] - ub)[sn == 2] <= 1e-6).all()
    assert (ln[sn == 1] >= 0).all() and (ln[sn == 2] <= 0).all() and (ln[sn == 0] == 0).all()


def test_ntg_without_npsol_solves_equality_problems(port):
    """NPSOL absent, van der Pol as shipped (linear equalities only, examples/vanderpol.c:159-169):
    ntg() falls back to the built-in reduced-space BFGS and returns a feasible stationary point."""
    out, err = _run_ntg_no_npsol(False)
    lines = dict(l.split(" ", 1) for l in out.strip().splitlines() if " " in l)
    assert int(lines["INFORM"]) in (0, 1), out + err
    assert "built-in" in err
    x = np.array([float(v) for v in lines["X"].split()])
    spec = configs.vanderpol(20, constraints=False)
    o = port.eval(spec, x[None, :], mode_obj=2, mode_con=-1, dense=False, band=False, linear=True)
    nC = spec.nC
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    assert np.abs(A @ x - b).max() < 1e-10
    assert abs(float(lines["OBJ"]) - o["f"][0]) <= 1e-12 * abs(o["f"][0])
    N = _null_basis(A)
    assert np.abs(o["g"][0] @ N).max() < 1e-6
    f1 = port.eval(spec, np.ones((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0]
    assert o["f"][0] < f1


@pytest.mark.parametrize("name", ["cfg3_kincar", "endpoint"])
def test_batched_merit_linesearch(port, name):
    """ntgb_linesearch: P*nalpha values-only evaluations in one launch + per-problem Armijo /
    argmin selection, against the CPU oracle evaluated at the same trial points."""
    import torch
    from ntg_b200 import Problem
    from common import violation
    spec, X = golden_spec(name)
    rng = np.random.default_rng(21)
    P, nC = X.shape
    D = rng.uniform(-1, 1, (P, nC))
    alphas = np.array([1.0, 0.5, 0.25, 0.125, 0.0625])
    mu, c1 = 3.0, 1e-4
    o = port.eval(spec, X, dense=False, band=False, linear=True)
    def merit(Xe):
        r = port.eval(spec, Xe, mode_obj=0, mode_con=0, dense=False, band=False)
        v = violation(spec, r["c"])
        lin = Xe @ o["A"].T
        lb, ub = o["bl"][nC:nC + spec.nclin], o["bu"][nC:nC + spec.nclin]
        vl = np.maximum(np.maximum(lb - lin, lin - ub), 0).max(axis=1) if spec.nclin else np.zeros(len(Xe))
        return r["f"] + mu * np.maximum(v, vl)
    phi0 = merit(X)
    dphi0 = -np.abs(rng.uniform(0.1, 1.0, P)) * np.abs(phi0)
    trial = np.stack([merit(X + a * D) for a in alphas], axis=1)          # [P][nalpha]
    want_a, want_phi = np.zeros(P), np.zeros(P)
    for p in range(P):
        ok = [i for i, a in enumerate(alphas) if trial[p, i] <= phi0[p] + c1 * a * dphi0[p]]
        i = ok[0] if ok else int(np.argmin(trial[p]))
        want_a[p], want_phi[p] = alphas[i], trial[p, i]
    pb = Problem(spec, 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    ab, pbest, Cn = pb.linesearch(t(X), t(D), t(alphas), mu, c1, t(phi0), t(dphi0))
    torch.cuda.synchronize()
    assert_close(pbest.cpu().numpy(), want_phi, "merit at the chosen step")
    assert np.array_equal(ab.cpu().numpy(), want_a), "chosen step sizes"
    assert_bitexact(Cn.cpu().numpy(), X + want_a[:, None] * D, "updated coefficients")
    pb.close()


def _null_basis(A):
    """orthonormal null-space basis of A by SVD (independent of the library's Householder QR)"""
    if A.shape[0] == 0:
        return np.eye(A.shape[1])
    u, s, vt = np.linalg.svd(A)
    r = int((s > 1e-11 * s[0]).sum())
    return vt[r:].T


def test_batched_solve_quadratic_kkt(port):
    """ntgb_solve_eq on the kinematic-car lane change without nonlinear constraints (the shipped
    example's problem class, examples/kincar.c:319-339): the cost is a convex quadratic in C and
    the constraints are linear equalities, so every initial guess must reach THE solution of the
    KKT system assembled on the host from the oracle's gradient and A."""
    import torch
    from ntg_b200 import Problem
    spec = configs.kincar(20, constraints=False, name="solve_kincar")
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    Q = port.eval(spec, np.eye(nC), mode_obj=2, mode_con=-1, dense=False, band=False)["g"]   # g(e_i) = Q e_i
    m = A.shape[0]
    K = np.block([[Q, A.T], [A, np.zeros((m, m))]])
    sol = np.linalg.lstsq(K, np.concatenate([np.zeros(nC), b]), rcond=None)[0]
    Cstar = sol[:nC]
    fstar = 0.5 * Cstar @ Q @ Cstar
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=5)
    pb = Problem(spec, 0)
    Cd = torch.from_numpy(X).cuda()
    f, it, st = pb.solve_eq(Cd, max_iter=100, gtol=1e-10)
    Cs = Cd.cpu().numpy()
    assert (st.cpu().numpy() >= 1).all(), "every problem must terminate before the iteration limit"
    assert np.abs(Cs @ A.T - b).max() <= 1e-9 * (1 + np.abs(b).max()), "A*C = b"
    np.testing.assert_allclose(f.cpu().numpy(), fstar, rtol=1e-9)
    # the minimiser is unique in the null space directions the cost sees; compare the gradient-relevant part
    N = _null_basis(A)
    gr = (Cs @ Q) @ N
    assert np.abs(gr).max() <= 1e-6 * max(1.0, abs(fstar))
    assert it.cpu().numpy().max() <= 100
    pb.close()


def test_batched_solve_vanderpol_vs_scipy(port):
    """ntgb_solve_eq on the van der Pol problem of examples/vanderpol.c:159-169 (3 linear equality
    constraints, no nonlinear ones) from 256 random initial guesses: feasibility, first-order
    optimality checked with the ORACLE's gradient, and the cost against scipy's SLSQP started from
    the same guesses (it may stop in a different local minimum: ours must not be worse by more than
    rounding when both stop at the same point, and a few are compared point-wise)."""
    import torch
    from scipy.optimize import minimize
    from ntg_b200 import Problem
    spec = configs.vanderpol(20, constraints=False, name="solve_vdp")
    nC = spec.nC
    o = port.eval(spec, np.zeros((1, nC)), dense=False, band=False, linear=True)
    A, b = o["A"], o["bl"][nC:nC + spec.nclin]
    P = 256
    X = configs.coefficients("cfg2", P, spec, seed=9)
    pb = Problem(spec, 0)
    Cd = torch.from_numpy(X).cuda()
    f, it, st = pb.solve_eq(Cd, max_iter=300, gtol=1e-9)
    Cs, fs, sts = Cd.cpu().numpy(), f.cpu().numpy(), st.cpu().numpy()
    assert (sts >= 1).mean() > 0.98
    assert np.abs(Cs @ A.T - b).max() <= 1e-9
    r = port.eval(spec, Cs, mode_obj=2, mode_con=-1, dense=False, band=False)
    assert_close(fs, r["f"], "final cost equals the oracle's at the returned point")
    N = _null_basis(A)
    gr = np.abs(r["g"] @ N).max(axis=1)
    ok = sts == 1
    assert (gr[ok] <= 1e-6 * np.maximum(1.0, np.abs(fs[ok]))).all(), gr[ok].max()
    # feasible start of each problem = projection of X onto A*C = b; the cost must not rise from it
    y0 = (X - Cs) @ N
    f0 = port.eval(spec, Cs + y0 @ N.T, mode_obj=0, mode_con=-1, dense=False, band=False)["f"]
    assert (fs <= f0 + 1e-12 * np.abs(f0)).all(), "descent from the projected initial guess"

    def fun(c):
        e = port.eval(spec, c[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        return float(e["f"][0]), e["g"][0]
    same = 0
    for p in range(8):
        res = minimize(fun, X[p], jac=True, method="SLSQP",
                       constraints=[{"type": "eq", "fun": lambda c: A @ c - b, "jac": lambda c: A}],
                       options={"ftol": 1e-14, "maxiter": 500})
        if np.abs(res.x - Cs[p]).max() < 1e-3:
            same += 1
            assert abs(res.fun - fs[p]) <= 1e-7 * max(1.0, abs(fs[p]))
    assert same >= 4, "most starts should reach the same local minimum as SLSQP"
    pb.close()


def test_solve_refuses_inequalities_and_nonlinear():
    import torch
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    spec = configs.kincar(20, constraints=True, name="solve_refuse")
    pb = Problem(spec, 0)
    with pytest.raises(NtgError):
        pb.solve_eq(torch.zeros((4, spec.nC), dtype=torch.float64, device="cuda"))
    pb.close()


def _kincar_active_constraints(nbps=40, ninterv=4):
    """lane change with enough freedom (nC = 22, 10 free directions) and nonlinear bounds that are
    ACTIVE at the solution: speed^2 <= 66.2 (66.5 unconstrained), |curvature numerator| <= 7.2 (7.66)"""
    import dataclasses
    base = configs.kincar(nbps, constraints=True, name="nlp_kincar")
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    kw.update(ninterv=[ninterv, ninterv], knots=None, bps=None)
    spec = type(base)(**kw)
    lo, up = spec.lowerb.copy(), spec.upperb.copy()
    lo[-2], up[-2] = 0.0, 66.2
    lo[-1], up[-1] = -7.2, 7.2
    spec.lowerb, spec.upperb = lo, up
    return spec


def test_batched_nlp_solver_vs_slsqp(port):
    """ntgb_solve_nlp (augmented Lagrangian + reduced-space BFGS, every step a batched kernel) on 512
    lane-change problems with active nonlinear constraints, from random starts: feasibility and the
    linear equalities checked with the ORACLE, the cost against scipy SLSQP (started next to the
    GPU's answer so that it converges -- from the random starts it fails on most of them)."""
    import torch
    from scipy.optimize import minimize
    from ntg_b200 import Problem
    spec = _kincar_active_constraints()
    nC = spec.nC
    P = 512
    X = configs.coefficients("cfg3", P, spec, seed=5)
    pb = Problem(spec, 0)
    Cd = torch.from_numpy(X).cuda()
    f, v, it, st = pb.solve_nlp(Cd)
    Cs, f, v, st = Cd.cpu().numpy(), f.cpu().numpy(), v.cpu().numpy(), st.cpu().numpy()
    ok = st >= 1
    assert ok.mean() >= 0.9, f"only {ok.mean():.2f} of the problems converged"
    o = port.eval(spec, Cs, mode_obj=0, mode_con=0, dense=False, band=False, linear=True)
    A, bl, bu = o["A"], o["bl"], o["bu"]
    b = bl[nC:nC + spec.nclin]
    assert np.abs(Cs @ A.T - b).max() <= 1e-8 * (1 + np.abs(b).max()), "linear equalities"
    lb, ub = bl[nC + spec.nclin:], bu[nC + spec.nclin:]
    viol = np.maximum(np.maximum(lb - o["c"], o["c"] - ub), 0).max(axis=1)
    assert (viol[ok] <= 1e-4).all(), viol[ok].max()
    assert_close(f, o["f"], "reported cost equals the oracle's at the returned point")
    assert (o["c"][ok].max(axis=1) > 7.19).all(), "the curvature bound is active at the solution"

    def fun(c):
        e = port.eval(spec, c[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        return float(e["f"][0]), e["g"][0]

    def con(c):
        e = port.eval(spec, c[None, :], mode_obj=-1, mode_con=2, dense=True, band=False)
        Jd = np.nan_to_num(e["Jdense"][0], nan=0.0)
        return e["c"][0], (Jd.T if Jd.shape[0] == nC else Jd)

    cons = [{"type": "eq", "fun": lambda c: A @ c - b, "jac": lambda c: A},
            {"type": "ineq", "fun": lambda c: con(c)[0] - lb, "jac": lambda c: con(c)[1]},
            {"type": "ineq", "fun": lambda c: ub - con(c)[0], "jac": lambda c: -con(c)[1]}]
    idx = np.flatnonzero(ok)[:3]
    for p in idx:
        r = minimize(fun, Cs[p] + 1e-3, jac=True, method="SLSQP", constraints=cons, options={"ftol": 1e-13, "maxiter": 300})
        assert r.success, r.message
        assert abs(r.fun - f[p]) <= 2e-5 * abs(r.fun), (r.fun, f[p])
        assert np.abs(r.x - Cs[p]).max() <= 1e-2
    pb.close()


_EXAMPLE_MAIN_CODE = r"""
import ctypes as C, os, sys
sys.path.insert(0, %r)
from ntg_b200 import problem
lib = problem.load_pack("ref_%s")
os.chdir(%r)
main = getattr(lib, "ntg_example_%s_main")
main.restype = C.c_int
if %r == "kincar":
    argv = (C.c_char_p * 2)(b"kincar", None)
    rc = main(1, argv)
else:
    rc = main()
sys.stdout.flush()
print("MAIN_RC", rc)
"""


@pytest.mark.parametrize("example", ["vanderpol", "kincar"])
def test_reference_examples_end_to_end_without_npsol(port, example, tmp_path):
    """examples/vanderpol.c and examples/kincar.c, UNMODIFIED, as whole programs with NO NPSOL in
    the process: main() calls ntg(), ntg() solves with the built-in reduced-space BFGS, the program
    prints / stores its result as it would after NPSOL (examples/vanderpol.c:192 writes ./coef1,
    examples/kincar.c:393-406 prints the interpolated trajectory)."""
    import subprocess
    import sys
    from ntg_b200 import build
    if not os.path.exists(build.pack_so(f"ref_{example}")):
        pytest.skip("drop-in example packs are built where /root/reference exists")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = _EXAMPLE_MAIN_CODE % (root, example, str(tmp_path), example, example)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert "MAIN_RC 0" in p.stdout, p.stdout[-2000:] + p.stderr[-2000:]
    assert "built-in" in p.stderr and "reduced-space BFGS" in p.stderr
    if example == "vanderpol":
        coef = np.array(open(tmp_path / "coef1").read().split(), dtype=np.float64)
        spec = configs.vanderpol(20, constraints=False)
        assert coef.shape == (spec.nC,)
        o = port.eval(spec, coef[None, :], mode_obj=2, mode_con=-1, dense=False, band=False, linear=True)
        nC = spec.nC
        A, b = o["A"], o["bl"][nC:nC + spec.nclin]
        assert np.abs(A @ coef - b).max() < 1e-4          # %g keeps 6 significant digits
        N = _null_basis(A)
        assert np.abs(o["g"][0] @ N).max() < 1e-3, "coef1 is a stationary point of the problem the example poses"
        f1 = port.eval(spec, np.ones((1, nC)), mode_obj=0, mode_con=-1, dense=False, band=False)["f"][0]
        assert o["f"][0] < f1                              # better than the example's initial guess of ones
    else:
        rows = [l.split() for l in p.stdout.splitlines() if len(l.split()) == 6]
        T = np.array(rows[-30:], dtype=np.float64)         # time x y theta v delta
        assert T.shape == (30, 6)
        np.testing.assert_allclose(T[0, :3], [0.0, 0.0, -2.0], atol=1e-3)
        np.testing.assert_allclose(T[-1, :3], [5.0, 40.0, 2.0], atol=1e-3)
        np.testing.assert_allclose(T[[0, -1], 4], [8.0, 8.0], rtol=1e-3)   # speed at both ends
        assert (np.diff(T[:, 1]) > 0).all() and (np.diff(T[:, 2]) >= -1e-6).all()   # a lane change


def test_batched_nlp_solver_all_constraint_kinds(port):
    """ntgb_solve_nlp on the test problem that has EVERY kind of row (packs/endpt.c: initial /
    trajectory / final cost, nonlinear initial / trajectory / final constraints, linear inequality
    rows of all three kinds, two outputs with different splines): the assembly of grad L_A from the
    band Jacobian (k_alm_grad) is only right if the points it stops at are KKT points -- checked by
    starting scipy SLSQP AT the returned point with the oracle's f, g, c, J: it must stay there."""
    import torch
    from scipy.optimize import minimize
    from ntg_b200 import Problem
    spec = configs.endpoint()
    nC = spec.nC
    P = 64
    X = np.random.default_rng(3).uniform(-0.5, 0.5, (P, nC))
    pb = Problem(spec, 0)
    Cd = torch.from_numpy(X).cuda()
    f, v, it, st = pb.solve_nlp(Cd, max_outer=60, max_inner=100)
    Cs, f, v, st = Cd.cpu().numpy(), f.cpu().numpy(), v.cpu().numpy(), st.cpu().numpy()
    ok = st >= 1
    assert ok.mean() >= 0.6, f"only {ok.mean():.2f} of the problems converged"
    o = port.eval(spec, Cs, dense=False, band=False, linear=True)
    A, bl, bu = o["A"], o["bl"], o["bu"]
    lbl, ubl = bl[nC:nC + spec.nclin], bu[nC:nC + spec.nclin]
    lbn, ubn = bl[nC + spec.nclin:], bu[nC + spec.nclin:]
    lin = Cs @ A.T
    vl = np.maximum(np.maximum(lbl - lin, lin - ubl), 0).max(axis=1)
    vn = np.maximum(np.maximum(lbn - o["c"], o["c"] - ubn), 0).max(axis=1)
    assert (vl[ok] <= 1e-4).all() and (vn[ok] <= 1e-4).all(), (vl[ok].max(), vn[ok].max())

    def fun(c):
        e = port.eval(spec, c[None, :], mode_obj=2, mode_con=-1, dense=False, band=False)
        return float(e["f"][0]), e["g"][0]

    def con(c):
        e = port.eval(spec, c[None, :], mode_obj=-1, mode_con=2, dense=True, band=False)
        Jd = np.nan_to_num(e["Jdense"][0], nan=0.0)
        return e["c"][0], (Jd.T if Jd.shape[0] == nC else Jd)

    cons = [{"type": "ineq", "fun": lambda c: A @ c - lbl, "jac": lambda c: A},
            {"type": "ineq", "fun": lambda c: ubl - A @ c, "jac": lambda c: -A},
            {"type": "ineq", "fun": lambda c: con(c)[0] - lbn, "jac": lambda c: con(c)[1]},
            {"type": "ineq", "fun": lambda c: ubn - con(c)[0], "jac": lambda c: -con(c)[1]}]
    for p in np.flatnonzero(ok)[:3]:
        r = minimize(fun, Cs[p], jac=True, method="SLSQP", constraints=cons, options={"ftol": 1e-13, "maxiter": 300})
        assert abs(r.fun - f[p]) <= 1e-4 * max(1.0, abs(f[p])), (r.fun, f[p])
        assert np.abs(r.x - Cs[p]).max() <= 1e-2, "SLSQP moved away: the returned point was not a KKT point"
    pb.close()


def test_solver_edge_cases(port):
    """P = 1; a problem without any linear constraint (nothing to eliminate: N is the identity);
    a problem beyond the solvers' limit of 32 free directions is refused, not mangled."""
    import torch
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError
    # P = 1 through both solvers
    spec = configs.vanderpol(20, constraints=False, name="solve_vdp1")
    pb = Problem(spec, 0)
    C1 = torch.ones((1, spec.nC), dtype=torch.float64, device="cuda")
    f, it, st = pb.solve_eq(C1)
    assert int(st[0]) >= 1
    C2 = torch.ones((1, spec.nC), dtype=torch.float64, device="cuda")
    f2, v2, it2, st2 = pb.solve_nlp(C2)
    assert int(st2[0]) >= 1 and abs(float(f2[0]) - float(f[0])) <= 1e-6 * abs(float(f[0]))
    pb.close()
    # no linear constraints at all, one nonlinear trajectory constraint with bounds [-1, 1]
    spec = configs.high_order(order=6, mult=3, ninterv=4, nbps=33, name="solve_hi")
    assert spec.nclin == 0
    pb = Problem(spec, 0)
    X = np.random.default_rng(8).uniform(-0.5, 0.5, (32, spec.nC))
    Cd = torch.from_numpy(X).cuda()
    f, v, it, st = pb.solve_nlp(Cd)
    Cs = Cd.cpu().numpy()
    o = port.eval(spec, Cs, mode_obj=2, mode_con=0, dense=False, band=False)
    assert_close(f.cpu().numpy(), o["f"], "cost at the returned point")
    ok = st.cpu().numpy() >= 1
    assert ok.mean() >= 0.9
    assert (np.abs(o["c"][ok]).max(axis=1) <= 1.0 + 1e-5).all()
    # the cost is a positive definite quadratic and C = 0 is feasible: the minimum is f = 0 at C = 0
    assert (f.cpu().numpy()[ok] <= 1e-8).all()
    pb.close()
    # too many free directions
    spec, _ = configs.get("cfg5")
    pb = Problem(spec, 0)
    with pytest.raises(NtgError):
        pb.solve_nlp(torch.zeros((2, spec.nC), dtype=torch.float64, device="cuda"))
    pb.close()


@pytest.mark.gpu
def test_batched_integrate_all_three_rules():
    """ntgb_integrate against the UNMODIFIED reference's IntegrateVector (src/integrator.c:16-38) for
    FEULER / BEULER / TRAPEZOID: bit-identical sums on non-uniform times (tests/golden/integrate.npz)."""
    import ctypes as C
    import torch
    from ntg_b200 import problem
    core = problem.core()
    core.ntgb_integrate.argtypes = [C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    core.ntgb_integrate.restype = C.c_int
    gm = golden_module()
    want = np.load(os.path.join(GOLDEN, "integrate.npz"))
    rows = gm.INTEGRATE_ROWS
    for t, f in gm.integrate_inputs():
        n = t.size
        assert_bitexact(t, want[f"t{n}"], "seeded inputs reproduce")
        fd, td = torch.from_numpy(f).cuda(), torch.from_numpy(t).cuda()
        for rule in (0, 1, 2):
            out = torch.full((rows,), np.nan, dtype=torch.float64, device="cuda")
            assert core.ntgb_integrate(rule, rows, n, fd.data_ptr(), td.data_ptr(), out.data_ptr(), None) == 0
            torch.cuda.synchronize()
            assert_bitexact(out.cpu().numpy(), want[f"I{n}_rule{rule}"], f"rule {rule}, n {n}")
    assert core.ntgb_integrate(7, 1, 2, fd.data_ptr(), td.data_ptr(), out.data_ptr(), None) != 0
