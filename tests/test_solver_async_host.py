"""CPU checks of the stream-ordered solver entry points: bad arguments are NTGB_EINVAL, refused before any
CUDA call, so they need no device."""
import ctypes as C


def test_async_arguments_are_refused_before_cuda(built_libs):
    from ntg_b200 import problem
    lib = problem.core()
    C_ = (C.c_double * 4)()
    for fn in (lib.ntgb_solve_eq_reserve, lib.ntgb_solve_sqp_reserve):
        assert fn(None, 4) == -1
        assert "null argument" in lib.ntgb_last_error().decode()
    for fn, extra in ((lib.ntgb_solve_eq_async, 5), (lib.ntgb_solve_sqp_async, 9)):
        assert fn(None, 4, C_, None, None, *([None] * extra)) == -1
        assert "null argument" in lib.ntgb_last_error().decode()
