"""Python host mirror of the C ABI (include/ntg_b200.h) for tests and bench.

PyTorch is plumbing here: device memory, streams, torch.distributed.  All
compute goes through libntg_b200.so + a callback pack; if either shared object
is missing this module raises -- there is no Python/CPU evaluation path.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import numpy as np

from . import abi
from .abi import (JAC_BAND, JAC_DENSE, JAC_NONE, BuiltSetup, NtgbDims, NtgbEvalArgs, NtgbPack, SolveOpts, LbfgsOpts, NewtonOpts, NlpOpts, SqpOpts,
                  ProblemSpec, c_double_p, c_int_p)

_LIBDIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
_core = None
_packs: Dict[str, C.CDLL] = {}


class NtgError(RuntimeError):
    pass


def core() -> C.CDLL:
    global _core
    if _core is None:
        path = os.path.join(_LIBDIR, "libntg_b200.so")
        if not os.path.exists(path):
            raise NtgError(f"{path} is missing: build it with `python -m ntg_b200.build` "
                           "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = C.CDLL(path)  # RTLD_LOCAL: it exports ntg(), linspace(), ... like the reference does
        lib.ntgb_last_error.restype = C.c_char_p
        lib.ntgb_version.restype = C.c_char_p
        lib.ntgb_find_pack.restype = C.POINTER(NtgbPack)
        lib.ntgb_find_pack.argtypes = [C.c_char_p]
        lib.ntgb_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(abi.NtgbSetup), C.c_int]
        lib.ntgb_destroy.argtypes = [C.c_void_p]
        lib.ntgb_get_dims.argtypes = [C.c_void_p, C.POINTER(NtgbDims)]
        lib.ntgb_eval.argtypes = [C.c_void_p, C.POINTER(NtgbEvalArgs)]
        lib.ntgb_eval_host.argtypes = [C.c_void_p, C.POINTER(NtgbEvalArgs)]
        lib.ntgb_get_tables.argtypes = [C.c_void_p, c_double_p, c_int_p, c_int_p]
        lib.ntgb_get_augknots.argtypes = [C.c_void_p, C.c_int, c_double_p, c_int_p]
        lib.ntgb_get_pattern.argtypes = [C.c_void_p, c_int_p, c_int_p]
        lib.ntgb_get_linear.argtypes = [C.c_void_p, c_double_p]
        lib.ntgb_get_bounds.argtypes = [C.c_void_p, c_double_p, c_double_p]
        lib.ntgb_eval_linear.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ntgb_solve_eq.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
        lib.ntgb_solve_eq.restype = C.c_int
        lib.ntgb_solve_eq_lbfgs.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
        lib.ntgb_solve_eq_lbfgs.restype = C.c_int
        lib.ntgb_solve_eq_newton.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
        lib.ntgb_solve_eq_newton.restype = C.c_int
        lib.ntgb_newton_structure.argtypes = [C.c_void_p] * 4
        lib.ntgb_newton_structure.restype = C.c_int
        lib.ntgb_solve_nlp.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ntgb_solve_nlp.restype = C.c_int
        lib.ntgb_solve_sqp.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 9
        lib.ntgb_solve_sqp.restype = C.c_int
        lib.ntgb_solve_eq_bounds.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
        lib.ntgb_solve_eq_bounds.restype = C.c_int
        lib.ntgb_solve_sqp_bounds.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 11
        lib.ntgb_solve_sqp_bounds.restype = C.c_int
        lib.ntgb_sqp_warm_doubles.argtypes = [C.c_void_p, C.POINTER(C.c_size_t)]
        lib.ntgb_sqp_warm_doubles.restype = C.c_int
        lib.ntgb_solve_sqp_warm.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 12
        lib.ntgb_solve_sqp_warm.restype = C.c_int
        for name in ("ntgb_solve_eq_reserve", "ntgb_solve_sqp_reserve"):
            getattr(lib, name).argtypes = [C.c_void_p, C.c_int]
            getattr(lib, name).restype = C.c_int
        lib.ntgb_solve_eq_async.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
        lib.ntgb_solve_eq_async.restype = C.c_int
        lib.ntgb_solve_sqp_async.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 12
        lib.ntgb_solve_sqp_async.restype = C.c_int
        lib.ntgb_peer_table_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p]
        lib.ntgb_peer_table_open.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]
        lib.ntgb_peer_table_close.argtypes = [C.c_void_p, C.c_void_p]
        lib.ntgb_peer_table_free.argtypes = [C.c_void_p, C.c_void_p]
        lib.ntgb_linesearch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ntgb_spline_interp.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p]
        _core = lib
    return _core


def load_pack(name: str) -> C.CDLL:
    """dlopen a callback pack; its static initialiser registers it with the core."""
    core()
    if name not in _packs:
        path = os.path.join(os.environ.get("NTG_B200_PACK_DIR", _LIBDIR), f"libntgpack_{name}.so")
        if not os.path.exists(path):
            raise NtgError(f"callback pack {path} is missing: build it with `python -m ntg_b200.build`")
        _packs[name] = C.CDLL(path)  # RTLD_LOCAL: exact/fast variants define the same symbols
        if not core().ntgb_find_pack(name.encode()):
            raise NtgError(f"pack '{name}' loaded but did not register")
    return _packs[name]


def _check(rc: int):
    if rc != 0:
        raise NtgError(f"ntg_b200 error {rc}: {core().ntgb_last_error().decode()}")


def _ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Problem:
    """One NTG problem family on one GPU: tables built once on the device (K0),
    then batched evaluations (K1)."""

    def __init__(self, spec: ProblemSpec, device: int = 0, fast: bool = False):
        self.spec = spec
        self.fast = fast
        self.packname = spec.pack + ("_fast" if fast else "")
        lib = load_pack(self.packname)
        self._built = BuiltSetup(spec, lambda role, sym: C.cast(getattr(lib, sym), C.c_void_p).value)
        self._h = C.c_void_p()
        _check(core().ntgb_create(C.byref(self._h), self._built.ref(), device))
        self.dims = NtgbDims()
        _check(core().ntgb_get_dims(self._h, C.byref(self.dims)))
        self.device = device

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            core().ntgb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- one-time tables (K0) ----
    def tables(self):
        s = self.spec
        tot = sum(s.nbps * k * m for k, m in zip(s.order, s.maxderiv))
        B = np.zeros(tot)
        off = np.zeros((s.nout, s.nbps), dtype=np.int32)
        left = np.zeros((s.nout, s.nbps), dtype=np.int32)
        _check(core().ntgb_get_tables(self._h, B.ctypes.data_as(c_double_p), off.ctypes.data_as(c_int_p),
                                      left.ctypes.data_as(c_int_p)))
        out, pos = [], 0
        for k, m in zip(s.order, s.maxderiv):
            n = s.nbps * k * m
            out.append(B[pos:pos + n].reshape(s.nbps, k, m).copy())
            pos += n
        return out, off, left

    def augknots(self, j: int) -> np.ndarray:
        n = C.c_int(0)
        _check(core().ntgb_get_augknots(self._h, j, None, C.byref(n)))
        t = np.zeros(n.value)
        _check(core().ntgb_get_augknots(self._h, j, t.ctypes.data_as(c_double_p), C.byref(n)))
        return t

    def pattern(self):
        col0 = np.zeros((max(self.dims.ncnln, 1), self.dims.nout), dtype=np.int32)
        jk0 = np.zeros(self.dims.nout, dtype=np.int32)
        _check(core().ntgb_get_pattern(self._h, col0.ctypes.data_as(c_int_p), jk0.ctypes.data_as(c_int_p)))
        return col0[:self.dims.ncnln], jk0

    def linear(self) -> np.ndarray:
        """A as [nclin][nC] (stored column-major nclin x nC for NPSOL)"""
        A = np.zeros((self.dims.nC, max(self.dims.nclin, 1)))
        _check(core().ntgb_get_linear(self._h, A.ctypes.data_as(c_double_p)))
        return A[:, :self.dims.nclin].T.copy()

    def bounds(self):
        n = self.dims.nC + self.dims.nclin + self.dims.ncnln
        bl, bu = np.zeros(n), np.zeros(n)
        _check(core().ntgb_get_bounds(self._h, bl.ctypes.data_as(c_double_p), bu.ctypes.data_as(c_double_p)))
        return bl, bu

    # ---- batched evaluation (K1), device tensors ----
    def alloc_outputs(self, P: int, jac: int = JAC_BAND, want_Z: bool = False, zero: bool = True):
        import torch
        d = self.dims
        dev = torch.device("cuda", self.device)
        mk = torch.zeros if zero else torch.empty
        out = {
            "f": mk(P, dtype=torch.float64, device=dev),
            "g": mk((P, d.nC), dtype=torch.float64, device=dev),
            "c": mk((P, max(d.ncnln, 1)), dtype=torch.float64, device=dev),
            "result": mk((P, 2), dtype=torch.float64, device=dev),
            "J": None, "Z": None,
        }
        if jac == JAC_BAND and d.ncnln:
            out["J"] = mk((P, d.ncnln * d.sorder), dtype=torch.float64, device=dev)
        elif jac == JAC_DENSE and d.ncnln:
            out["J"] = torch.zeros((P, d.nC, d.ncnln), dtype=torch.float64, device=dev)
        if want_Z:
            out["Z"] = mk((P, d.nZ), dtype=torch.float64, device=dev)
        return out

    def eval_args(self, Cdev, out, mode_obj=2, mode_con=2, jac=JAC_BAND, nstate=0, stream=None,
                  abort_flag=None, peers=None) -> NtgbEvalArgs:
        """peers: a shard.PeerGather -- the kernel then also stores every (objective, violation) pair
        into all ranks' gathered tables (fused multi-GPU gather)"""
        a = NtgbEvalArgs()
        a.P = int(Cdev.shape[0])
        a.C = Cdev.data_ptr()
        a.mode_obj, a.mode_con, a.nstate = mode_obj, mode_con, nstate
        a.f, a.g, a.c = _ptr(out["f"]), _ptr(out["g"]), _ptr(out["c"])
        a.J = _ptr(out["J"])
        a.jac_layout = jac if out["J"] is not None else JAC_NONE
        a.Z = _ptr(out.get("Z"))
        a.result = _ptr(out.get("result"))
        a.stream = stream
        a.abort_flag = _ptr(abort_flag)
        if peers is not None:
            a.npeers = len(peers.tables)
            a.peer_row0 = peers.row0
            a.peer_result = peers.device_pointers()
        return a

    def launch(self, args: NtgbEvalArgs):
        _check(core().ntgb_eval(self._h, C.byref(args)))

    def eval(self, Cdev, mode_obj=2, mode_con=2, jac=JAC_BAND, want_Z=False, nstate=0, out=None):
        """Cdev: cuda float64 tensor [P][nC].  Runs on torch's current stream."""
        import torch
        assert Cdev.is_cuda and Cdev.dtype == torch.float64 and Cdev.is_contiguous()
        assert Cdev.shape[1] == self.dims.nC
        if out is None:
            out = self.alloc_outputs(Cdev.shape[0], jac, want_Z)
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        self.launch(self.eval_args(Cdev, out, mode_obj, mode_con, jac, nstate, st))
        return out

    def eval_host(self, X: np.ndarray, mode_obj=2, mode_con=2, jac=JAC_BAND, want_Z=False, nstate=0):
        """Host buffers in and out through ntgb_eval_host (H2D + launch + D2H inside)."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        P, d = X.shape[0], self.dims
        out = {"f": np.zeros(P), "g": np.zeros((P, d.nC)), "c": np.zeros((P, max(d.ncnln, 1))),
               "result": np.zeros((P, 2)), "J": None, "Z": np.zeros((P, d.nZ)) if want_Z else None}
        if d.ncnln and jac == JAC_BAND:
            out["J"] = np.zeros((P, d.ncnln * d.sorder))
        elif d.ncnln and jac == JAC_DENSE:
            out["J"] = np.zeros((P, d.nC, d.ncnln))
        a = NtgbEvalArgs()
        a.P = P
        a.C = X.ctypes.data
        a.mode_obj, a.mode_con, a.nstate = mode_obj, mode_con, nstate
        a.f, a.g, a.c = out["f"].ctypes.data, out["g"].ctypes.data, out["c"].ctypes.data
        a.J = None if out["J"] is None else out["J"].ctypes.data
        a.jac_layout = jac if out["J"] is not None else JAC_NONE
        a.Z = None if out["Z"] is None else out["Z"].ctypes.data
        a.result = out["result"].ctypes.data
        _check(core().ntgb_eval_host(self._h, C.byref(a)))
        out["c"] = out["c"][:, :d.ncnln]
        return out

    def eval_host_tensors(self, Xh, out, mode_obj=2, mode_con=2, jac=JAC_BAND, nstate=0):
        """ntgb_eval_host on (ideally pinned) host torch tensors: Xh [P][nC]; out: dict with any of
        f [P], g [P][nC], c [P][ncnln], J [P][ncnln*S or nC*ncnln], result [P][2]."""
        a = NtgbEvalArgs()
        a.P = int(Xh.shape[0])
        a.C = Xh.data_ptr()
        a.mode_obj, a.mode_con, a.nstate = mode_obj, mode_con, nstate
        a.f, a.g, a.c = _ptr(out.get("f")), _ptr(out.get("g")), _ptr(out.get("c"))
        a.J = _ptr(out.get("J"))
        a.jac_layout = jac if out.get("J") is not None else JAC_NONE
        a.Z = _ptr(out.get("Z"))
        a.result = _ptr(out.get("result"))
        _check(core().ntgb_eval_host(self._h, C.byref(a)))

    # ---- band <-> (row, col, value) ----
    def band_to_rows(self, Jband: np.ndarray) -> np.ndarray:
        """device band layout [P][ncnln*S] (trajectory rows breakpoint-fastest, in tiles of
        dims.band_tile breakpoints: include/ntg_b200.h, NTGB_JAC_BAND) -> row-major [P][ncnln][S],
        the layout the CPU oracles report"""
        s, d = self.spec, self.dims
        P, S, nb, TB = Jband.shape[0], d.sorder, s.nbps, d.band_tile
        out = np.empty((P, d.ncnln, S))
        pos = 0
        n = s.nnlic * S
        out[:, :s.nnlic, :] = Jband[:, pos:pos + n].reshape(P, s.nnlic, S)
        pos += n
        traj = out[:, s.nnlic:s.nnlic + s.nnltc * nb, :].reshape(P, s.nnltc, nb, S)
        for b0 in range(0, nb, TB):          # tile = breakpoints [b0, b0 + nt): values [m][slot][bp - b0]
            nt = min(TB, nb - b0)
            n = s.nnltc * S * nt
            traj[:, :, b0:b0 + nt, :] = Jband[:, pos:pos + n].reshape(P, s.nnltc, S, nt).transpose(0, 1, 3, 2)
            pos += n
        n = s.nnlfc * S
        out[:, s.nnlic + s.nnltc * nb:, :] = Jband[:, pos:pos + n].reshape(P, s.nnlfc, S)
        return out

    def eval_linear(self, Cdev):
        import torch
        P, d = Cdev.shape[0], self.dims
        lin = torch.zeros((P, max(d.nclin, 1)), dtype=torch.float64, device=Cdev.device)
        viol = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        _check(core().ntgb_eval_linear(self._h, P, Cdev.data_ptr(), lin.data_ptr(), viol.data_ptr(), st))
        return lin[:, :d.nclin], viol

    def linesearch(self, Cdev, dCdev, alphas, mu, c1=1e-4, phi0=None, dphi0=None):
        """batched merit line search (ntgb_linesearch); returns alpha_best [P], phi_best [P], C_new"""
        import torch
        P = Cdev.shape[0]
        ab = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        pbest = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        Cn = torch.zeros_like(Cdev)
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        _check(core().ntgb_linesearch(self._h, P, Cdev.data_ptr(), dCdev.data_ptr(), int(alphas.shape[0]),
                                      alphas.data_ptr(), float(mu), float(c1), _ptr(phi0), _ptr(dphi0),
                                      ab.data_ptr(), pbest.data_ptr(), Cn.data_ptr(), st))
        return ab, pbest, Cn

    def _check_bounds(self, Cdev, lowerb, upperb):
        """per-problem bounds: both or neither, float64 CUDA tensors [P][spec.nbounds] next to Cdev"""
        import torch
        if lowerb is None and upperb is None:
            return False
        shape = (Cdev.shape[0], self.spec.nbounds)
        for name, b in (("lowerb", lowerb), ("upperb", upperb)):
            if b is None:
                raise ValueError(f"{name} is missing: per-problem bounds need both lowerb and upperb")
            if not (b.is_cuda and b.dtype == torch.float64 and b.is_contiguous() and tuple(b.shape) == shape
                    and b.device == Cdev.device):
                raise ValueError(f"{name} must be a contiguous float64 tensor of shape {shape} on {Cdev.device}")
        return True

    def solver_reserve(self, solver: str, P_max: int):
        """one-time work and the work space of the stream-ordered solver ("eq" or "sqp") for up to P_max
        problems (ntgb_solve_eq_reserve / ntgb_solve_sqp_reserve); needed before solve_eq / solve_sqp with
        sync=False.  Synchronizes the device.  Reserving more replaces the work space: capture graphs again."""
        fn = {"eq": core().ntgb_solve_eq_reserve, "sqp": core().ntgb_solve_sqp_reserve}.get(solver)
        if fn is None:
            raise ValueError(f"solver must be 'eq' or 'sqp', not {solver!r}")
        _check(fn(self._h, int(P_max)))

    def solve_eq(self, Cdev, max_iter=0, gtol=0.0, c1=0.0, check_every=0, lowerb=None, upperb=None, sync=True):
        """batched reduced-space BFGS (ntgb_solve_eq); Cdev [P][nC] is overwritten with the solutions.
        Returns f [P], iters [P], status [P] (1 converged, 2 no further decrease, 0 iteration limit).
        lowerb / upperb [P][spec.nbounds] (device): each problem's own bounds, in the layout of
        spec.lowerb / upperb (ntgb_solve_eq_bounds; status 5 = that problem's bounds were rejected).
        sync=False: ntgb_solve_eq_async on torch's current stream (after solver_reserve("eq", P)): exactly
        max_iter iterations, the same outputs bit for bit, returned without waiting; capturable in a
        torch.cuda.graph."""
        import torch
        P = Cdev.shape[0]
        per_problem = self._check_bounds(Cdev, lowerb, upperb)
        f = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        it = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        stt = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        opts = SolveOpts(int(max_iter), float(gtol), float(c1), int(check_every))
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        if not sync:
            lo_p, up_p = (lowerb.data_ptr(), upperb.data_ptr()) if per_problem else (None, None)
            _check(core().ntgb_solve_eq_async(self._h, P, Cdev.data_ptr(), lo_p, up_p, f.data_ptr(), it.data_ptr(),
                                              stt.data_ptr(), C.addressof(opts), st))
        elif per_problem:
            _check(core().ntgb_solve_eq_bounds(self._h, P, Cdev.data_ptr(), lowerb.data_ptr(), upperb.data_ptr(),
                                               f.data_ptr(), it.data_ptr(), stt.data_ptr(), C.addressof(opts), st))
        else:
            _check(core().ntgb_solve_eq(self._h, P, Cdev.data_ptr(), f.data_ptr(), it.data_ptr(), stt.data_ptr(),
                                        C.addressof(opts), st))
        return f, it, stt

    def solve_eq_lbfgs(self, Cdev, max_iter=0, gtol=0.0, c1=0.0, memory=0, check_every=0, lowerb=None, upperb=None):
        """batched projected L-BFGS (ntgb_solve_eq_lbfgs): the problems of solve_eq with any number of free
        directions.  Cdev [P][nC] is overwritten with the solutions.  Returns f [P], iters [P], status [P]
        (1 converged, 2 no further decrease, 0 iteration limit, 5 rejected per-problem bounds).  memory: the
        curvature pairs kept per problem, 1..32 (0: 8); the other options take their defaults at 0.
        lowerb / upperb [P][spec.nbounds] (device): each problem's own bounds, as in solve_eq."""
        import torch
        P = Cdev.shape[0]
        per_problem = self._check_bounds(Cdev, lowerb, upperb)
        f = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        it = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        stt = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        opts = LbfgsOpts(int(max_iter), float(gtol), float(c1), int(memory) if memory else 8, int(check_every))
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        lo_p, up_p = (lowerb.data_ptr(), upperb.data_ptr()) if per_problem else (None, None)
        _check(core().ntgb_solve_eq_lbfgs(self._h, P, Cdev.data_ptr(), lo_p, up_p, f.data_ptr(), it.data_ptr(),
                                          stt.data_ptr(), C.addressof(opts), st))
        return f, it, stt

    def solve_eq_newton(self, Cdev, max_iter=0, gtol=0.0, c1=0.0, check_every=0, lowerb=None, upperb=None):
        """batched banded Newton (ntgb_solve_eq_newton): the problems of solve_eq_lbfgs, with the Hessian from
        coloured gradient differences.  Cdev [P][nC] is overwritten with the solutions.  Returns f [P], iters [P],
        status [P] (1 converged, 2 no further decrease, 0 iteration limit, 5 rejected per-problem bounds); the
        options take their defaults at 0.  lowerb / upperb [P][spec.nbounds] (device): each problem's own bounds."""
        import torch
        P = Cdev.shape[0]
        per_problem = self._check_bounds(Cdev, lowerb, upperb)
        f = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        it = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        stt = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        opts = NewtonOpts(int(max_iter), float(gtol), float(c1), int(check_every))
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        lo_p, up_p = (lowerb.data_ptr(), upperb.data_ptr()) if per_problem else (None, None)
        _check(core().ntgb_solve_eq_newton(self._h, P, Cdev.data_ptr(), lo_p, up_p, f.data_ptr(), it.data_ptr(),
                                           stt.data_ptr(), C.addressof(opts), st))
        return f, it, stt

    def newton_structure(self):
        """-> (K colours, half-bandwidth w, perm [nC]) of solve_eq_newton for this setup"""
        K, w = C.c_int(), C.c_int()
        perm = np.zeros(self.spec.nC, dtype=np.int32)
        _check(core().ntgb_newton_structure(self._h, C.byref(K), C.byref(w), perm.ctypes.data))
        return K.value, w.value, perm

    def solve_nlp(self, Cdev, max_outer=0, max_inner=0, gtol=0.0, ctol=0.0, rho0=0.0, rho_mul=0.0, rho_max=0.0,
                  c1=0.0, check_every=0):
        """batched augmented-Lagrangian solve (ntgb_solve_nlp); Cdev [P][nC] is overwritten.
        Returns f [P], violation [P], iters [P], status [P]."""
        import torch
        P = Cdev.shape[0]
        f = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        v = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        it = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        stt = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        opts = NlpOpts(int(max_outer), int(max_inner), float(gtol), float(ctol), float(rho0), float(rho_mul),
                       float(rho_max), float(c1), int(check_every))
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        _check(core().ntgb_solve_nlp(self._h, P, Cdev.data_ptr(), f.data_ptr(), v.data_ptr(), it.data_ptr(),
                                     stt.data_ptr(), C.addressof(opts), st))
        return f, v, it, stt

    def sqp_warm_doubles(self) -> int:
        """doubles in one problem's row of SQP warm-start state (ntgb_sqp_warm_doubles)"""
        n = C.c_size_t(0)
        _check(core().ntgb_sqp_warm_doubles(self._h, C.byref(n)))
        return n.value

    def sqp_warm_state(self, P: int):
        """zeroed warm-start state for P problems, float64 [P][sqp_warm_doubles()] on this Problem's device:
        every row starts cold; solve_sqp(..., warm=) fills it"""
        import torch
        return torch.zeros((P, self.sqp_warm_doubles()), dtype=torch.float64, device=torch.device("cuda", self.device))

    def solve_sqp(self, Cdev, max_iter=0, gtol=0.0, ctol=0.0, rho_pen=0.0, c1=0.0, check_every=0, multipliers=False,
                  lowerb=None, upperb=None, warm=None, sync=True):
        """batched SQP solve (ntgb_solve_sqp); Cdev [P][nC] is overwritten.  Returns f [P], violation [P],
        iters [P], status [P] and, with multipliers=True, lambda and istate [P][nclin + ncnln] (NPSOL's order).
        lowerb / upperb [P][spec.nbounds] (device): each problem's own bounds (ntgb_solve_sqp_bounds).
        warm [P][sqp_warm_doubles()] (device, from sqp_warm_state): solver state carried from the previous
        call and updated in place (ntgb_solve_sqp_warm).
        sync=False: ntgb_solve_sqp_async on torch's current stream (after solver_reserve("sqp", P)): exactly
        max_iter iterations, the same outputs bit for bit, returned without waiting; capturable in a
        torch.cuda.graph."""
        import torch
        P, d = Cdev.shape[0], self.dims
        per_problem = self._check_bounds(Cdev, lowerb, upperb)
        if warm is not None:
            shape = (P, self.sqp_warm_doubles())
            if not (isinstance(warm, torch.Tensor) and warm.is_cuda and warm.dtype == torch.float64
                    and warm.is_contiguous() and tuple(warm.shape) == shape and warm.device == Cdev.device):
                raise ValueError(f"warm must be a contiguous float64 tensor of shape {shape} on {Cdev.device}")
        f = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        v = torch.zeros(P, dtype=torch.float64, device=Cdev.device)
        it = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        stt = torch.zeros(P, dtype=torch.int32, device=Cdev.device)
        lam = ist = None
        if multipliers:
            lam = torch.zeros((P, d.nclin + d.ncnln), dtype=torch.float64, device=Cdev.device)
            ist = torch.zeros((P, d.nclin + d.ncnln), dtype=torch.int32, device=Cdev.device)
        opts = SqpOpts(int(max_iter), float(gtol), float(ctol), float(rho_pen), float(c1), int(check_every))
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        lam_p, ist_p = (lam.data_ptr(), ist.data_ptr()) if multipliers else (None, None)
        if not sync:
            lo_p, up_p = (lowerb.data_ptr(), upperb.data_ptr()) if per_problem else (None, None)
            _check(core().ntgb_solve_sqp_async(self._h, P, Cdev.data_ptr(), lo_p, up_p, _ptr(warm), f.data_ptr(),
                                               v.data_ptr(), it.data_ptr(), stt.data_ptr(), lam_p, ist_p,
                                               C.addressof(opts), st))
        elif warm is not None:
            lo_p, up_p = (lowerb.data_ptr(), upperb.data_ptr()) if per_problem else (None, None)
            _check(core().ntgb_solve_sqp_warm(self._h, P, Cdev.data_ptr(), lo_p, up_p, warm.data_ptr(), f.data_ptr(),
                                              v.data_ptr(), it.data_ptr(), stt.data_ptr(), lam_p, ist_p,
                                              C.addressof(opts), st))
        elif per_problem:
            _check(core().ntgb_solve_sqp_bounds(self._h, P, Cdev.data_ptr(), lowerb.data_ptr(), upperb.data_ptr(),
                                                f.data_ptr(), v.data_ptr(), it.data_ptr(), stt.data_ptr(), lam_p, ist_p,
                                                C.addressof(opts), st))
        else:
            _check(core().ntgb_solve_sqp(self._h, P, Cdev.data_ptr(), f.data_ptr(), v.data_ptr(), it.data_ptr(),
                                         stt.data_ptr(), lam_p, ist_p, C.addressof(opts), st))
        return (f, v, it, stt, lam, ist) if multipliers else (f, v, it, stt)

    def spline_interp(self, Cdev, tdev):
        import torch
        P, nt, d = Cdev.shape[0], tdev.shape[0], self.dims
        out = torch.zeros((P, nt, d.nz), dtype=torch.float64, device=Cdev.device)
        st = torch.cuda.current_stream(Cdev.device).cuda_stream
        _check(core().ntgb_spline_interp(self._h, P, Cdev.data_ptr(), nt, tdev.data_ptr(), out.data_ptr(), st))
        return out
