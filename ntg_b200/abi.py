"""ctypes mirror of include/ntg_b200.h.

The structures here are byte-for-byte the C structs of the public header; the
same `ntgb_setup` is accepted by the product library (ntg_b200/lib) and by the
CPU oracle drivers under oracle/ (test infrastructure), so parity tests hand
both sides literally the same problem description -- the argument list of the
reference's ntg() (reference src/ntg.h:72-99).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class AV(C.Structure):
    """reference src/av.h:18-26"""
    _fields_ = [("output", C.c_int), ("deriv", C.c_int)]


class NtgbSetup(C.Structure):
    _fields_ = [
        ("nout", C.c_int),
        ("bps", c_double_p),
        ("nbps", C.c_int),
        ("kninterv", c_int_p),
        ("knots", C.POINTER(c_double_p)),
        ("order", c_int_p),
        ("mult", c_int_p),
        ("maxderiv", c_int_p),
        ("nlic", C.c_int), ("lic", C.POINTER(c_double_p)),
        ("nltc", C.c_int), ("ltc", C.POINTER(c_double_p)),
        ("nlfc", C.c_int), ("lfc", C.POINTER(c_double_p)),
        ("nnlic", C.c_int), ("nlicf", C.c_void_p),
        ("nnltc", C.c_int), ("nltcf", C.c_void_p),
        ("nnlfc", C.c_int), ("nlfcf", C.c_void_p),
        ("ninitialconstrav", C.c_int), ("initialconstrav", C.POINTER(AV)),
        ("ntrajectoryconstrav", C.c_int), ("trajectoryconstrav", C.POINTER(AV)),
        ("nfinalconstrav", C.c_int), ("finalconstrav", C.POINTER(AV)),
        ("lowerb", c_double_p),
        ("upperb", c_double_p),
        ("nicf", C.c_int), ("icf", C.c_void_p),
        ("nucf", C.c_int), ("ucf", C.c_void_p),
        ("nfcf", C.c_int), ("fcf", C.c_void_p),
        ("ninitialcostav", C.c_int), ("initialcostav", C.POINTER(AV)),
        ("ntrajectorycostav", C.c_int), ("trajectorycostav", C.POINTER(AV)),
        ("nfinalcostav", C.c_int), ("finalcostav", C.POINTER(AV)),
    ]


class NtgbDims(C.Structure):
    _fields_ = [(n, C.c_int) for n in
                ("nout", "nbps", "nC", "nz", "nZ", "nclin", "ncnln", "sorder", "device", "band_tile")]


class NtgbEvalArgs(C.Structure):
    _fields_ = [
        ("P", C.c_int),
        ("C", C.c_void_p),
        ("mode_obj", C.c_int),
        ("mode_con", C.c_int),
        ("nstate", C.c_int),
        ("f", C.c_void_p),
        ("g", C.c_void_p),
        ("c", C.c_void_p),
        ("J", C.c_void_p),
        ("jac_layout", C.c_int),
        ("Z", C.c_void_p),
        ("result", C.c_void_p),
        ("stream", C.c_void_p),
        ("abort_flag", C.c_void_p),
        ("npeers", C.c_int),
        ("peer_row0", C.c_int),
        ("peer_result", C.c_void_p),
    ]


class SolveOpts(C.Structure):
    """ntgb_solve_opts (include/ntg_b200.h)"""
    _fields_ = [("max_iter", C.c_int), ("gtol", C.c_double), ("c1", C.c_double), ("check_every", C.c_int)]


class LbfgsOpts(C.Structure):
    """ntgb_lbfgs_opts (include/ntg_b200.h)"""
    _fields_ = [("max_iter", C.c_int), ("gtol", C.c_double), ("c1", C.c_double), ("memory", C.c_int),
                ("check_every", C.c_int)]


class NewtonOpts(C.Structure):
    """ntgb_newton_opts (include/ntg_b200.h)"""
    _fields_ = [("max_iter", C.c_int), ("gtol", C.c_double), ("c1", C.c_double), ("check_every", C.c_int)]


class NlpOpts(C.Structure):
    """ntgb_nlp_opts (include/ntg_b200.h)"""
    _fields_ = [("max_outer", C.c_int), ("max_inner", C.c_int), ("gtol", C.c_double), ("ctol", C.c_double),
                ("rho0", C.c_double), ("rho_mul", C.c_double), ("rho_max", C.c_double), ("c1", C.c_double),
                ("check_every", C.c_int)]


class SqpOpts(C.Structure):
    """ntgb_sqp_opts (include/ntg_b200.h)"""
    _fields_ = [("max_iter", C.c_int), ("gtol", C.c_double), ("ctol", C.c_double), ("rho_pen", C.c_double),
                ("c1", C.c_double), ("check_every", C.c_int)]


class NtgbPack(C.Structure):
    _fields_ = [
        ("name", C.c_char_p),
        ("icf", C.c_void_p), ("ucf", C.c_void_p), ("fcf", C.c_void_p),
        ("nlicf", C.c_void_p), ("nltcf", C.c_void_p), ("nlfcf", C.c_void_p),
        ("max_nout", C.c_int), ("max_maxderiv", C.c_int), ("max_order", C.c_int),
        ("max_nnlic", C.c_int), ("max_nnltc", C.c_int), ("max_nnlfc", C.c_int),
        ("maxderiv", C.c_int * 8),
        ("exact", C.c_int),
        ("launch", C.c_void_p),
        ("abi", C.c_int),
    ]


JAC_NONE, JAC_DENSE, JAC_BAND = 0, 1, 2
STATUS_BAD_BOUNDS = 5  # NTGB_STATUS_BAD_BOUNDS: the per-problem bounds of that problem were rejected
ROLES = ("icf", "ucf", "fcf", "nlicf", "nltcf", "nlfcf")


def linspace(d0: float, d1: float, n: int) -> np.ndarray:
    """The reference's linspace (src/ntg.c:374-389): an ACCUMULATING recurrence
    v[i] = v[i-1] + step, not numpy's.  linspace(0,5,20)[-1] is 5.000000000000001
    (past the last knot), which decides the knot interval of the final
    breakpoint (SURVEY.md section 8, quirk Q1), so inputs must be generated this way.
    """
    v = np.empty(n, dtype=np.float64)
    if d0 == d1:
        v[:] = d0
        return v
    step = np.float64(d1 - d0) / np.float64(n - 1)
    v[0] = d0
    for i in range(1, n):
        v[i] = v[i - 1] + step
    return v


@dataclass
class ProblemSpec:
    """Host-side description of one NTG problem family (the arguments of ntg()
    minus the NPSOL workspaces), with callbacks named by (pack, symbol)."""
    name: str
    pack: str                       # callback pack name
    order: List[int]
    mult: List[int]
    maxderiv: List[int]
    ninterv: List[int]
    nbps: int
    t0: float = 0.0
    t1: float = 5.0
    bps: Optional[np.ndarray] = None          # default linspace(t0,t1,nbps)
    knots: Optional[List[np.ndarray]] = None  # default linspace(t0,t1,ninterv+1)
    # callbacks: role -> symbol name in the pack ('' = unused); counts
    callbacks: Dict[str, str] = field(default_factory=dict)
    nicf: int = 0
    nucf: int = 0
    nfcf: int = 0
    nnlic: int = 0
    nnltc: int = 0
    nnlfc: int = 0
    initialcostav: Sequence[Tuple[int, int]] = ()
    trajectorycostav: Sequence[Tuple[int, int]] = ()
    finalcostav: Sequence[Tuple[int, int]] = ()
    initialconstrav: Sequence[Tuple[int, int]] = ()
    trajectoryconstrav: Sequence[Tuple[int, int]] = ()
    finalconstrav: Sequence[Tuple[int, int]] = ()
    lic: Optional[np.ndarray] = None  # [nlic][nz]
    ltc: Optional[np.ndarray] = None
    lfc: Optional[np.ndarray] = None
    lowerb: Optional[np.ndarray] = None
    upperb: Optional[np.ndarray] = None

    def __post_init__(self):
        if self.bps is None:
            self.bps = linspace(self.t0, self.t1, self.nbps)
        self.bps = np.ascontiguousarray(self.bps, dtype=np.float64)
        self.nbps = int(self.bps.shape[0])
        if self.knots is None:
            self.knots = [linspace(self.t0, self.t1, ni + 1) for ni in self.ninterv]
        self.knots = [np.ascontiguousarray(k, dtype=np.float64) for k in self.knots]

    # derived sizes (reference src/colloc.c:47-50,67; src/ntg.c:155-157)
    @property
    def nout(self) -> int:
        return len(self.order)

    @property
    def ncoef(self) -> List[int]:
        return [l * (k - m) + m for l, k, m in zip(self.ninterv, self.order, self.mult)]

    @property
    def nC(self) -> int:
        return sum(self.ncoef)

    @property
    def nz(self) -> int:
        return sum(self.maxderiv)

    @property
    def nZ(self) -> int:
        return self.nz * self.nbps

    @property
    def nlic(self) -> int:
        return 0 if self.lic is None else int(self.lic.shape[0])

    @property
    def nltc(self) -> int:
        return 0 if self.ltc is None else int(self.ltc.shape[0])

    @property
    def nlfc(self) -> int:
        return 0 if self.lfc is None else int(self.lfc.shape[0])

    @property
    def nclin(self) -> int:
        return self.nlic + self.nltc * self.nbps + self.nlfc

    @property
    def ncnln(self) -> int:
        return self.nnlic + self.nnltc * self.nbps + self.nnlfc

    @property
    def sorder(self) -> int:
        return sum(self.order)

    @property
    def nbounds(self) -> int:
        return self.nlic + self.nltc + self.nlfc + self.nnlic + self.nnltc + self.nnlfc

    def bytes_per_eval(self, dense: bool = False) -> int:
        """Algorithmic bytes of one evaluation (SURVEY.md section 8(d)):
        read C; write f, g, c and the Jacobian band (or the dense matrix)."""
        nnz = self.ncnln * (self.nC if dense else self.sorder)
        return 8 * (self.nC + 1 + self.nC + self.ncnln + nnz)


class BuiltSetup:
    """An NtgbSetup plus every numpy/ctypes object it points into."""

    def __init__(self, spec: ProblemSpec, resolve):
        """resolve(role, symbol) -> integer address of the host callback"""
        self.spec = spec
        self._keep = []
        s = NtgbSetup()
        nout = spec.nout

        def ints(v):
            a = (C.c_int * len(v))(*[int(x) for x in v])
            self._keep.append(a)
            return C.cast(a, c_int_p)

        def dbl(a):
            a = np.ascontiguousarray(a, dtype=np.float64)
            self._keep.append(a)
            return a.ctypes.data_as(c_double_p)

        def rows(m):
            if m is None or m.shape[0] == 0:
                return C.cast(None, C.POINTER(c_double_p))
            m = np.ascontiguousarray(m, dtype=np.float64)
            self._keep.append(m)
            arr = (c_double_p * m.shape[0])(*[m[i].ctypes.data_as(c_double_p)
                                              for i in range(m.shape[0])])
            self._keep.append(arr)
            return C.cast(arr, C.POINTER(c_double_p))

        def avs(lst):
            lst = list(lst)
            if not lst:
                return 0, C.cast(None, C.POINTER(AV))
            arr = (AV * len(lst))(*[AV(int(o), int(d)) for o, d in lst])
            self._keep.append(arr)
            return len(lst), C.cast(arr, C.POINTER(AV))

        s.nout = nout
        s.bps = dbl(spec.bps)
        s.nbps = spec.nbps
        s.kninterv = ints(spec.ninterv)
        karr = (c_double_p * nout)(*[dbl(k) for k in spec.knots])
        self._keep.append(karr)
        s.knots = C.cast(karr, C.POINTER(c_double_p))
        s.order = ints(spec.order)
        s.mult = ints(spec.mult)
        s.maxderiv = ints(spec.maxderiv)
        s.nlic, s.lic = spec.nlic, rows(spec.lic)
        s.nltc, s.ltc = spec.nltc, rows(spec.ltc)
        s.nlfc, s.lfc = spec.nlfc, rows(spec.lfc)

        def cb(role, count):
            sym = spec.callbacks.get(role, "")
            if count == 0 or not sym:
                return None
            return resolve(role, sym)

        s.nnlic, s.nlicf = spec.nnlic, cb("nlicf", spec.nnlic)
        s.nnltc, s.nltcf = spec.nnltc, cb("nltcf", spec.nnltc)
        s.nnlfc, s.nlfcf = spec.nnlfc, cb("nlfcf", spec.nnlfc)
        s.ninitialconstrav, s.initialconstrav = avs(spec.initialconstrav)
        s.ntrajectoryconstrav, s.trajectoryconstrav = avs(spec.trajectoryconstrav)
        s.nfinalconstrav, s.finalconstrav = avs(spec.finalconstrav)
        nb = spec.nbounds
        lo = np.zeros(max(nb, 1)) if spec.lowerb is None else np.asarray(spec.lowerb, dtype=np.float64)
        hi = np.zeros(max(nb, 1)) if spec.upperb is None else np.asarray(spec.upperb, dtype=np.float64)
        assert lo.shape[0] >= nb and hi.shape[0] >= nb, "bounds shorter than constraint count"
        s.lowerb, s.upperb = dbl(lo), dbl(hi)
        s.nicf, s.icf = spec.nicf, cb("icf", spec.nicf)
        s.nucf, s.ucf = spec.nucf, cb("ucf", spec.nucf)
        s.nfcf, s.fcf = spec.nfcf, cb("fcf", spec.nfcf)
        s.ninitialcostav, s.initialcostav = avs(spec.initialcostav)
        s.ntrajectorycostav, s.trajectorycostav = avs(spec.trajectorycostav)
        s.nfinalcostav, s.finalcostav = avs(spec.finalcostav)
        self.struct = s

    def ref(self):
        return C.byref(self.struct)
