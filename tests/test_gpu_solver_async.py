"""GPU tests of the stream-ordered solvers (ntgb_solve_eq_async, ntgb_solve_sqp_async and their reserve calls):
every output is bit-identical to the synchronous entry point with the same arguments; the call returns while
the stream is still busy; it can be captured in a CUDA graph right after the reserve, alone or as a whole
receding-horizon control step, and the graph keeps working when synchronous calls grow the Problem's own
scratch; refusals match the synchronous ones; two Problems solve side by side on two streams."""
import numpy as np
import pytest

from ntg_b200 import configs
from ntg_b200.abi import STATUS_BAD_BOUNDS

pytestmark = pytest.mark.gpu

P_SQP, P_EQ = 512, 4096


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(ts):
    return [None if t is None else t.cpu().numpy() for t in ts]


def _assert_same_bits(got, want):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        assert a.shape == b.shape and a.dtype == b.dtype, i
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"output {i} differs"


def _sqp_setup(P, seed):
    from test_gpu_mpc import _active_specs
    spec, lo, up = _active_specs(P, seed)
    X = configs.coefficients("cfg3", P, spec, seed=seed + 1)
    return spec, X, lo, up


def _reject(lo, up):
    """three problems whose bounds k_bounds_prep rejects: lower > upper on the speed row, an eliminated row with
    lower != upper, a NaN"""
    lo, up = lo.copy(), up.copy()
    lo[3, 12], up[3, 12] = 70.0, 60.0
    up[17, 4] = lo[17, 4] + 1e-9
    lo[40, 13] = np.nan
    return lo, up, [3, 17, 40]


def _warm_rows(spec, X, lo, up):
    """matching warm rows, from a synchronous solve on another Problem of the same setup"""
    import torch
    from ntg_b200 import Problem
    q = Problem(spec, 0)
    W = q.sqp_warm_state(X.shape[0])
    q.solve_sqp(_cuda(X), lowerb=_cuda(lo), upperb=_cuda(up), warm=W)
    torch.cuda.synchronize()
    q.close()
    return W.cpu().numpy()


def _sqp_call(pb, X, sync, lo=None, up=None, W=None, **kw):
    """-> [C, f, viol, iters, status, (lambda, istate), (warm)] as numpy, after a device synchronize"""
    import torch
    Cd = _cuda(X)
    b = {} if lo is None else {"lowerb": _cuda(lo), "upperb": _cuda(up)}
    Wd = None if W is None else _cuda(W)
    res = pb.solve_sqp(Cd, warm=Wd, sync=sync, **b, **kw)
    torch.cuda.synchronize()
    return _host([Cd, *res] + ([] if Wd is None else [Wd]))


def _eq_setup(P, seed):
    from test_gpu_mpc import _lane_changes
    spec = configs.kincar(64, constraints=False, name="async_eq")
    b = _lane_changes(P, seed)
    X = configs.coefficients("cfg4", P, spec, seed=seed + 1)
    return spec, X, b


def _eq_call(pb, X, sync, lo=None, up=None, **kw):
    import torch
    Cd = _cuda(X)
    b = {} if lo is None else {"lowerb": _cuda(lo), "upperb": _cuda(up)}
    res = pb.solve_eq(Cd, sync=sync, **b, **kw)
    torch.cuda.synchronize()
    return _host([Cd, *res])


# ---- 1. the same answers, bit for bit --------------------------------------------------------------------

@pytest.mark.parametrize("max_iter", [1, 2, 0])
def test_sqp_async_matches_sync(max_iter):
    from ntg_b200 import Problem
    spec, X, lo, up = _sqp_setup(P_SQP, seed=3)
    lor, upr, bad = _reject(lo, up)
    W = _warm_rows(spec, configs.coefficients("cfg3", P_SQP, spec, seed=11), lo, up)
    pb = Problem(spec, 0)
    pb.solver_reserve("sqp", P_SQP)
    cases = {
        "shared": dict(multipliers=True),
        "bounds": dict(multipliers=True, lo=lo, up=up),
        "bounds, no multipliers": dict(lo=lo, up=up),
        "rejected bounds": dict(multipliers=True, lo=lor, up=upr),
        "zero warm rows": dict(multipliers=True, lo=lo, up=up, W=np.zeros_like(W)),
        "carried warm rows": dict(multipliers=True, lo=lo, up=up, W=W),
        "carried warm rows, rejected bounds": dict(multipliers=True, lo=lor, up=upr, W=W),
        "carried warm rows, shared bounds": dict(multipliers=True, W=W),
    }
    for name, kw in cases.items():
        want = _sqp_call(pb, X, True, max_iter=max_iter, **kw)
        got = _sqp_call(pb, X, False, max_iter=max_iter, **kw)
        try:
            _assert_same_bits(got, want)
        except AssertionError as e:
            raise AssertionError(f"{name}: {e}") from None
        if kw.get("lo") is lor:
            st = got[4]
            assert (st[bad] == STATUS_BAD_BOUNDS).all()
            assert np.array_equal(got[0][bad].view(np.int64), X[bad].view(np.int64))
            if "W" in kw:
                assert np.array_equal(got[-1][bad].view(np.int64), W[bad].view(np.int64))
    pb.close()


@pytest.mark.parametrize("max_iter", [2, 0])
def test_eq_async_matches_sync(max_iter):
    from ntg_b200 import Problem
    spec, X, b = _eq_setup(P_EQ, seed=7)
    lo, up = b.copy(), b.copy()
    bad = [5, P_EQ // 2]
    lo[5, 1] = up[5, 1] + 1.0
    lo[P_EQ // 2, 3] = np.nan
    pb = Problem(spec, 0)
    pb.solver_reserve("eq", P_EQ)
    for kw in ({}, {"lo": lo, "up": up}):
        want = _eq_call(pb, X, True, max_iter=max_iter, **kw)
        got = _eq_call(pb, X, False, max_iter=max_iter, **kw)
        _assert_same_bits(got, want)
        if kw:
            assert (got[3][bad] == STATUS_BAD_BOUNDS).all()
            assert np.array_equal(got[0][bad].view(np.int64), X[bad].view(np.int64))
    if max_iter == 0:
        assert (want[3][np.setdiff1d(np.arange(P_EQ), bad)] == 1).all()
    pb.close()


# ---- 2. the host does not wait -----------------------------------------------------------------------------

def test_async_returns_before_the_stream_is_done():
    import torch
    from ntg_b200 import Problem
    spec, X, lo, up = _sqp_setup(256, seed=21)
    W = _warm_rows(spec, X, lo, up)
    pb = Problem(spec, 0)
    pb.solver_reserve("sqp", 256)
    _sqp_call(pb, X, False, lo=lo, up=up, W=W, max_iter=2)   # kernels loaded
    want = _sqp_call(pb, X, True, lo=lo, up=up, W=W, max_iter=2, multipliers=True)
    Cd, lod, upd, Wd = _cuda(X), _cuda(lo), _cuda(up), _cuda(W)
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)                           # about 0.1 s at the B200's clock
    res = pb.solve_sqp(Cd, max_iter=2, multipliers=True, lowerb=lod, upperb=upd, warm=Wd, sync=False)
    assert not torch.cuda.current_stream().query(), "the async call waited for the stream"
    torch.cuda.synchronize()
    _assert_same_bits(_host([Cd, *res, Wd]), want)

    spec, X, b = _eq_setup(1024, seed=22)
    q = Problem(spec, 0)
    q.solver_reserve("eq", 1024)
    _eq_call(q, X, False, lo=b, up=b, max_iter=4)
    want = _eq_call(q, X, True, lo=b, up=b, max_iter=4)
    Cd, bd = _cuda(X), _cuda(b)
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)
    res = q.solve_eq(Cd, max_iter=4, lowerb=bd, upperb=bd, sync=False)
    assert not torch.cuda.current_stream().query(), "the async call waited for the stream"
    torch.cuda.synchronize()
    _assert_same_bits(_host([Cd, *res]), want)
    pb.close()
    q.close()


# ---- 3. capturable right after the reserve ------------------------------------------------------------------

def _replays(g, restore, outputs):
    import torch
    got = []
    for _ in range(2):
        restore()
        g.replay()
        torch.cuda.synchronize()
        got.append(_host(outputs))
    return got


def test_sqp_async_captured_in_a_graph():
    import torch
    from ntg_b200 import Problem
    P = 256
    spec, X, lo, up = _sqp_setup(P, seed=31)
    W = _warm_rows(spec, X, lo, up)
    pb = Problem(spec, 0)
    pb.solver_reserve("sqp", P)
    C0, W0, lod, upd = _cuda(X), _cuda(W), _cuda(lo), _cuda(up)
    Cs, Ws = C0.clone(), W0.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):           # capture_error_mode "global": a synchronizing call fails the capture
        res = pb.solve_sqp(Cs, max_iter=3, multipliers=True, lowerb=lod, upperb=upd, warm=Ws, sync=False)
    Ce, We = C0.clone(), W0.clone()
    ref = pb.solve_sqp(Ce, max_iter=3, multipliers=True, lowerb=lod, upperb=upd, warm=We, sync=False)
    torch.cuda.synchronize()
    want = _host([Ce, *ref, We])

    def restore():
        Cs.copy_(C0)
        Ws.copy_(W0)

    for got in _replays(g, restore, [Cs, *res, Ws]):
        _assert_same_bits(got, want)
    assert not np.array_equal(want[0], X), "the solve moved C"
    pb.close()


def test_eq_async_captured_in_a_graph():
    import torch
    from ntg_b200 import Problem
    P = 1024
    spec, X, b = _eq_setup(P, seed=32)
    pb = Problem(spec, 0)
    pb.solver_reserve("eq", P)
    C0, bd = _cuda(X), _cuda(b)
    Cs = C0.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res = pb.solve_eq(Cs, max_iter=5, lowerb=bd, upperb=bd, sync=False)
    Ce = C0.clone()
    ref = pb.solve_eq(Ce, max_iter=5, lowerb=bd, upperb=bd, sync=False)
    torch.cuda.synchronize()
    want = _host([Ce, *ref])
    for got in _replays(g, lambda: Cs.copy_(C0), [Cs, *res]):
        _assert_same_bits(got, want)
    pb.close()


# ---- 4. a real-time-iteration control step as one graph --------------------------------------------------

def test_control_step_as_one_graph():
    import torch
    from ntg_b200 import Problem
    P, steps, dt = 512, 10, 0.1
    spec, X, lo, up = _sqp_setup(P, seed=41)
    pb = Problem(spec, 0)
    pb.solver_reserve("sqp", P)
    tq = torch.tensor([dt], dtype=torch.float64, device="cuda")

    def step(C, lo_, up_, W, sync):
        f, v, it, st = pb.solve_sqp(C, max_iter=2, lowerb=lo_, upperb=up_, warm=W, sync=sync)
        z = pb.spline_interp(C, tq)[:, 0, :]
        lo_[:, :6] = z
        up_[:, :6] = z
        return f, it, st

    Cg, log, upg, Wg = _cuda(X), _cuda(lo), _cuda(up), pb.sqp_warm_state(P)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fg, itg, stg = step(Cg, log, upg, Wg, False)
    Cr, lor, upr, Wr = _cuda(X), _cuda(lo), _cuda(up), pb.sqp_warm_state(P)
    for k in range(steps):
        want = _host([Cr, Wr, *step(Cr, lor, upr, Wr, True), lor, upr])
        g.replay()
        torch.cuda.synchronize()
        got = _host([Cg, Wg, fg, itg, stg, log, upg])
        try:
            _assert_same_bits(got, want)
        except AssertionError as e:
            raise AssertionError(f"step {k + 1}: {e}") from None
    # not vacuous: the steps moved C, filled every warm row and made their two iterations (real-time iteration
    # from random starts is not expected to converge within ten steps)
    assert not np.array_equal(want[0], X)
    assert (want[1][:, 0] == float(0x4E545731)).all()
    assert (want[3][want[4] == 0] == 2).all() and (want[4] == 0).any()
    pb.close()


# ---- 5. the async work space is apart from the synchronous scratch ------------------------------------------

def test_graph_survives_a_larger_synchronous_solve():
    import torch
    from ntg_b200 import Problem
    P, Pbig = 128, 2048
    spec, X, lo, up = _sqp_setup(Pbig, seed=51)
    pb = Problem(spec, 0)
    _sqp_call(pb, X[:8], True, lo=lo[:8], up=up[:8], max_iter=2)          # a small synchronous scratch
    pb.solver_reserve("sqp", P)
    C0, lod, upd = _cuda(X[:P]), _cuda(lo[:P]), _cuda(up[:P])
    Cs, Ws = C0.clone(), pb.sqp_warm_state(P)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res = pb.solve_sqp(Cs, max_iter=4, multipliers=True, lowerb=lod, upperb=upd, warm=Ws, sync=False)
    want = _sqp_call(pb, X[:P], True, lo=lo[:P], up=up[:P], W=np.zeros((P, Ws.shape[1])), max_iter=4,
                     multipliers=True)
    _sqp_call(pb, X, True, lo=lo, up=up, W=np.zeros((Pbig, Ws.shape[1])), max_iter=3, multipliers=True)  # grows it
    _sqp_call(pb, X, True, max_iter=3)

    def restore():
        Cs.copy_(C0)
        Ws.zero_()

    for got in _replays(g, restore, [Cs, *res, Ws]):
        _assert_same_bits(got, want)
    pb.close()


# ---- 6. refusals ------------------------------------------------------------------------------------------

def test_async_refusals():
    import torch
    from ntg_b200 import Problem
    from ntg_b200.problem import NtgError, core
    spec, X, lo, up = _sqp_setup(16, seed=61)
    pb = Problem(spec, 0)
    Cd = _cuda(X)
    with pytest.raises(NtgError, match="error -1: .*reserved"):
        pb.solve_sqp(Cd, sync=False)                                     # no reserve yet
    pb.solver_reserve("sqp", 8)
    with pytest.raises(NtgError, match=r"error -1: .*P = 16 above the 8 problems reserved"):
        pb.solve_sqp(Cd, max_iter=2, sync=False)
    torch.cuda.synchronize()
    assert np.array_equal(Cd.cpu().numpy(), X), "a refused call queued work"
    lod = _cuda(lo[:8])
    assert core().ntgb_solve_sqp_async(pb._h, 8, Cd.data_ptr(), lod.data_ptr(), None, *([None] * 9)) == -1
    assert core().ntgb_solve_sqp_async(pb._h, 8, Cd.data_ptr(), None, lod.data_ptr(), *([None] * 9)) == -1
    assert core().ntgb_solve_sqp_async(pb._h, 0, Cd.data_ptr(), *([None] * 11)) == 0
    with pytest.raises(NtgError):
        pb.solver_reserve("eq", 8)                                        # nonlinear rows
    with pytest.raises(ValueError):
        pb.solver_reserve("nlp", 8)

    def message(fn):
        with pytest.raises(NtgError) as e:
            fn()
        return str(e.value)

    # the synchronous entry point's code and message
    assert message(lambda: pb.solver_reserve("eq", 8)) == message(lambda: pb.solve_eq(Cd))
    from test_gpu_sqp_lockstep import _hi_eq
    wide = Problem(_hi_eq(5, 2, 11, "async_eq33"), 0)
    C33 = _cuda(np.zeros((2, wide.spec.nC)))
    m = message(lambda: wide.solver_reserve("eq", 2))
    assert "33 free directions" in m and m == message(lambda: wide.solve_eq(C33))
    with pytest.raises(NtgError, match="error -1: .*reserved"):
        wide.solve_eq(C33, sync=False)
    wide.close()

    espec, EX, b = _eq_setup(8, seed=62)
    q = Problem(espec, 0)
    q.solver_reserve("eq", 8)
    Ce, bd = _cuda(EX), _cuda(b)
    assert core().ntgb_solve_eq_async(q._h, 8, Ce.data_ptr(), bd.data_ptr(), None, *([None] * 5)) == -1
    assert core().ntgb_solve_eq_async(q._h, 8, Ce.data_ptr(), None, bd.data_ptr(), *([None] * 5)) == -1
    with pytest.raises(NtgError, match=r"error -1: .*P = 9 above the 8 problems reserved"):
        q.solve_eq(_cuda(configs.coefficients("cfg4", 9, espec, seed=1)), sync=False)
    pb.close()
    q.close()


# ---- 7. two Problems on two streams ----------------------------------------------------------------------

def test_two_problems_on_two_streams():
    import torch
    from ntg_b200 import Problem
    sspec, SX, lo, up = _sqp_setup(512, seed=71)
    espec, EX, b = _eq_setup(4096, seed=72)
    ps, pe = Problem(sspec, 0), Problem(espec, 0)
    ps.solver_reserve("sqp", 512)
    pe.solver_reserve("eq", 4096)
    want_s = _sqp_call(ps, SX, True, lo=lo, up=up, max_iter=3, multipliers=True)
    want_e = _eq_call(pe, EX, True, lo=b, up=b, max_iter=20)
    Cs, lod, upd, Ce, bd = _cuda(SX), _cuda(lo), _cuda(up), _cuda(EX), _cuda(b)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        rs = ps.solve_sqp(Cs, max_iter=3, multipliers=True, lowerb=lod, upperb=upd, sync=False)
    with torch.cuda.stream(s2):
        re_ = pe.solve_eq(Ce, max_iter=20, lowerb=bd, upperb=bd, sync=False)
    torch.cuda.synchronize()
    _assert_same_bits(_host([Cs, *rs]), want_s)
    _assert_same_bits(_host([Ce, *re_]), want_e)
    ps.close()
    pe.close()
