"""GPU tests of the solvers' per-call device scratch, which a Problem keeps and grows between calls: a solver
called on one Problem at P = 3, then 300, then 3 again returns exactly what the same call returns on a fresh
Problem, and so do solve_eq, solve_sqp and solve_nlp called one after the other on one Problem, which share its
reduced form."""
import numpy as np
import pytest

from ntg_b200 import configs

pytestmark = pytest.mark.gpu


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _eq_spec():
    return configs.kincar(64, constraints=False, name="scratch_eq")


def _active_spec():
    from test_gpu_next import _kincar_active_constraints
    return _kincar_active_constraints()


def _eq(pb, P, seed):
    C = _cuda(configs.coefficients("cfg4", P, pb.spec, seed=seed))
    return (C,) + tuple(pb.solve_eq(C))


def _eq_bounds(pb, P, seed):
    from test_gpu_mpc import _lane_changes
    b = _lane_changes(P, seed)
    lo, up = b.copy(), b.copy()
    lo[P // 2, 1] = up[P // 2, 1] + 1.0            # lower > upper: this problem's bounds are rejected
    C = _cuda(configs.coefficients("cfg4", P, pb.spec, seed=seed))
    return (C,) + tuple(pb.solve_eq(C, lowerb=_cuda(lo), upperb=_cuda(up)))


def _nlp(pb, P, seed):
    C = _cuda(configs.coefficients("cfg3", P, pb.spec, seed=seed))
    return (C,) + tuple(pb.solve_nlp(C))


def _sqp(pb, P, seed):
    C = _cuda(configs.coefficients("cfg3", P, pb.spec, seed=seed))
    return (C,) + tuple(pb.solve_sqp(C, multipliers=True))


def _sqp_bounds(pb, P, seed):
    from test_gpu_mpc import _active_specs
    _, lo, up = _active_specs(P, seed)
    lo[P // 2, 12] = up[P // 2, 12] + 1.0          # lower > upper on the speed row: rejected
    C = _cuda(configs.coefficients("cfg3", P, pb.spec, seed=seed))
    return (C,) + tuple(pb.solve_sqp(C, multipliers=True, lowerb=_cuda(lo), upperb=_cuda(up)))


def _sqp_warm(pb, P, seed):
    """a cold call that fills the warm rows, then a warm call from them"""
    X = configs.coefficients("cfg3", P, pb.spec, seed=seed)
    W = pb.sqp_warm_state(P)
    C1, C2 = _cuda(X), _cuda(X)
    out1 = pb.solve_sqp(C1, warm=W)
    W1 = W.clone()
    out2 = pb.solve_sqp(C2, warm=W)
    return (C1, W1) + tuple(out1) + (C2, W) + tuple(out2)


def _linesearch(pb, P, seed):
    import torch
    rng = np.random.default_rng(seed)
    C = _cuda(configs.coefficients("cfg3", P, pb.spec, seed=seed))
    dC = _cuda(rng.uniform(-0.1, 0.1, (P, pb.spec.nC)))
    alphas = _cuda(np.ldexp(1.0, -np.arange(8)))
    phi0 = torch.full((P,), 1e300, dtype=torch.float64, device="cuda")
    return tuple(pb.linesearch(C, dC, alphas, 10.0, phi0=phi0))


CALLS = {
    "solve_eq": (_eq_spec, _eq),
    "solve_eq_bounds": (_eq_spec, _eq_bounds),
    "solve_nlp": (_active_spec, _nlp),
    "solve_sqp": (_active_spec, _sqp),
    "solve_sqp_bounds": (_active_spec, _sqp_bounds),
    "solve_sqp_warm": (_active_spec, _sqp_warm),
    "linesearch": (_active_spec, _linesearch),
}


def _same_bytes(got, ref, what):
    assert len(got) == len(ref)
    for i, (a, b) in enumerate(zip(got, ref)):
        a, b = a.cpu().numpy(), b.cpu().numpy()
        assert a.dtype == b.dtype and a.shape == b.shape, f"{what}: output {i}"
        assert a.tobytes() == b.tobytes(), f"{what}: output {i} differs from the call on a fresh Problem"


@pytest.mark.parametrize("call", list(CALLS))
def test_scratch_growth_and_reuse(call):
    """P = 3, 300, 3 on one Problem: the scratch is sized, grown, then reused at its larger size"""
    from ntg_b200 import Problem
    make_spec, run = CALLS[call]
    spec = make_spec()
    pb = Problem(spec, 0)
    for k, P in enumerate((3, 300, 3)):
        got = run(pb, P, seed=40 + k)
        fresh = Problem(spec, 0)
        ref = run(fresh, P, seed=40 + k)
        fresh.close()
        _same_bytes(got, ref, f"{call} at P = {P} (call {k + 1})")
    pb.close()


def test_solvers_sharing_the_reduced_form():
    """solve_eq, solve_sqp and solve_nlp on one Problem use the same reduced form"""
    from ntg_b200 import Problem
    spec = _eq_spec()
    pb = Problem(spec, 0)
    for k, run in enumerate((_eq, _sqp, _nlp)):
        got = run(pb, 64, seed=50 + k)
        fresh = Problem(spec, 0)
        ref = run(fresh, 64, seed=50 + k)
        fresh.close()
        _same_bytes(got, ref, run.__name__)
    pb.close()
