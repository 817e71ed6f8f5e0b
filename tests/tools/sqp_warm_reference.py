"""tests/tools/sqp_warm_reference.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The SQP warm start of ntgb_solve_sqp_warm on the host: sqp_reference.sqp_via_core (the g++-compiled core
of ntg_sqp.cuh's sqp_step, driven with oracle evaluations) started the way k_sqp_init starts a problem
from a matching row of warm-start state -- B and nu from the row, flags "no previous step" (flag[0] = 0,
as sqp_via_core starts) and "B is not the identity" (flag[3] = 0).  The loop itself is sqp_via_core's,
unchanged: the core library is wrapped so that its FIRST sqp_host_step call sees that state, and every
call's resulting B and nu are kept -- what k_sqp_warm_store writes back after the last pass.
"""
from __future__ import annotations

import numpy as np

from sqp_reference import sqp_via_core


class _WarmCore:
    """the core library with sqp_host_step wrapped (arguments as in tests/tools/sqp_host.cpp:
    n, m, f, gr, h, hl, hu, A, B, lam, sprev, grLold, grold, d, scal, flag, istate, gtol, ctol, rho_pen)"""

    def __init__(self, lib, B0, nu0):
        self._lib = lib
        self._first = B0 is not None
        self.B, self.nu = None, None

        def step(*a):
            n, B, scal, flag = a[0], a[8], a[14], a[15]
            if self._first:
                self._first = False
                for e, v in enumerate(np.asarray(B0, dtype=np.float64).ravel()):
                    B[e] = float(v)
                scal[0] = float(nu0)
                flag[3] = 0
            lib.sqp_host_step.argtypes = step.argtypes  # set by sqp_via_core on this wrapper
            lib.sqp_host_step(*a)
            self.B = np.array([B[e] for e in range(n * n)]).reshape(n, n)
            self.nu = float(scal[0])

        self.sqp_host_step = step

    def __getattr__(self, name):
        return getattr(self._lib, name)


def sqp_via_core_warm(lib, nlp, y0, B0=None, nu0=0.0, **kw):
    """sqp_via_core warm-started from B0 [nr][nr] and nu0 (B0 None: the cold start B = I, nu = 0); the result
    also carries the final B and nu, what the solve writes into its row"""
    core = _WarmCore(lib, B0, nu0)
    r = sqp_via_core(core, nlp, y0, **kw)
    r.update(B=core.B, nu=core.nu)
    return r
