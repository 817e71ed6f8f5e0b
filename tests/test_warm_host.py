"""CPU checks of the SQP warm start (ntgb_solve_sqp_warm).  The row format and its match / clamp rules
(ntg_b200/csrc/ntg_warm.h, compiled with g++ through tests/tools/warm_host.cpp -- the same text
k_sqp_init and k_sqp_warm_store run), and whole solves of a moved MPC problem by the g++-compiled core
of ntg_sqp.cuh started the way k_sqp_init starts a matching row, every evaluation by the CPU oracle.
The device half is checked in tests/test_gpu_sqp_warm.py."""
import ctypes as C
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "tools"))
from sqp_reference import ReducedNLP, sqp_via_core  # noqa: E402
from sqp_warm_reference import sqp_via_core_warm  # noqa: E402

TAG = float(0x4E545731)
HEADER = 6


def _build(tmp_path_factory, src, name):
    so = str(tmp_path_factory.mktemp(name) / f"{name}.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "ntg_b200", "csrc"),
                           "-o", so, os.path.join(HERE, "tools", src)])
    return C.CDLL(so)


@pytest.fixture(scope="module")
def warm_lib(tmp_path_factory):
    lib = _build(tmp_path_factory, "warm_host.cpp", "warm_host")
    dp = C.POINTER(C.c_double)
    lib.warm_host_doubles.restype = C.c_size_t
    lib.warm_host_doubles.argtypes = [C.c_int]
    lib.warm_host_digest.restype = C.c_uint64
    lib.warm_host_digest.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_int), dp]
    lib.warm_host_encode.argtypes = [dp, C.c_int, C.c_int, C.c_uint64, C.c_double, dp, C.c_int, C.c_int]
    lib.warm_host_load.restype = C.c_int
    lib.warm_host_load.argtypes = [dp, C.c_int, C.c_int, C.c_uint64, dp, dp]
    return lib


@pytest.fixture(scope="module")
def core_lib(tmp_path_factory):
    return _build(tmp_path_factory, "sqp_host.cpp", "sqp_host")


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _encode(lib, nr, m, digest, nu, B, start=0, step=1, row=None):
    if row is None:
        row = np.zeros(lib.warm_host_doubles(nr))
    B = np.ascontiguousarray(B, dtype=np.float64)
    lib.warm_host_encode(_dp(row), nr, m, digest, nu, _dp(B), start, step)
    return row


def _load(lib, row, nr, m, digest):
    """-> (matched, B, nu) as k_sqp_init starts a problem from this row"""
    row = np.ascontiguousarray(row, dtype=np.float64)
    B, nu = np.full((nr, nr), np.nan), np.full(1, np.nan)
    hot = lib.warm_host_load(_dp(row), nr, m, digest, _dp(B), _dp(nu))
    return bool(hot), B, float(nu[0])


def _spd(rng, n):
    M = rng.normal(size=(n, n))
    return M @ M.T + n * np.eye(n)


def _fnv1a(data: bytes) -> int:
    h = 14695981039346656037
    for b in data:
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


# ---- the row format ---------------------------------------------------------------------------------

def test_encode_load_round_trip(warm_lib):
    rng = np.random.default_rng(0)
    for nr, m in ((1, 0), (10, 83), (31, 7), (40, 200)):
        digest = int(rng.integers(0, 2**63, dtype=np.int64)) * 2 + 1
        B, nu = _spd(rng, nr), float(rng.uniform(0, 5))
        assert warm_lib.warm_host_doubles(nr) == HEADER + nr * nr
        row = _encode(warm_lib, nr, m, digest, nu, B)
        assert row[0] == TAG and row[1] == nr and row[2] == m and row[5] == nu
        assert int(row[3]) + (int(row[4]) << 32) == digest
        assert np.array_equal(row[HEADER:].reshape(nr, nr), B)
        # k_sqp_warm_store's split: one warp per row, lane k writes entries k, k + 32, ...
        split = np.full_like(row, np.nan)
        for lane in range(32):
            _encode(warm_lib, nr, m, digest, nu, B, lane, 32, row=split)
        assert np.array_equal(split.view(np.int64), row.view(np.int64))
        hot, B2, nu2 = _load(warm_lib, row, nr, m, digest)
        assert hot and nu2 == nu
        assert np.array_equal(B2.view(np.int64), B.view(np.int64))


def test_rows_that_do_not_match_start_cold(warm_lib):
    rng = np.random.default_rng(1)
    nr, m = 10, 83
    digest = 0x9E3779B97F4A7C15
    good = _encode(warm_lib, nr, m, digest, 2.5, _spd(rng, nr))
    assert _load(warm_lib, good, nr, m, digest)[0]
    bad = {"zeros": np.zeros_like(good), "garbage": rng.normal(size=good.shape)}
    for k, v in ((0, TAG + 1), (1, nr + 1), (2, m - 1), (3, good[3] + 1), (4, good[4] - 1), (0, np.nan), (3, np.nan)):
        r = good.copy()
        r[k] = v
        bad[f"row[{k}] = {v}"] = r
    for name, r in bad.items():
        hot, B, nu = _load(warm_lib, r, nr, m, digest)
        assert not hot, name
        assert np.array_equal(B, np.eye(nr)) and nu == 0.0, name
    # the same row for another setup (another digest, nr or m) is cold too
    assert not _load(warm_lib, good, nr, m, digest ^ 1)[0]
    assert not _load(warm_lib, good, nr, m + 1, digest)[0]
    # no row at all (a rejected problem, or no warm array): cold
    B, nu = np.full((nr, nr), np.nan), np.full(1, np.nan)
    assert warm_lib.warm_host_load(None, nr, m, digest, _dp(B), _dp(nu)) == 0
    assert np.array_equal(B, np.eye(nr)) and nu[0] == 0.0


def test_nu_is_clamped_and_b_read_from_its_lower_triangle(warm_lib):
    rng = np.random.default_rng(2)
    nr, m, digest = 6, 20, 12345678901234567
    B = _spd(rng, nr)
    for nu, want in ((np.nan, 0.0), (np.inf, 0.0), (-np.inf, 0.0), (-1e-300, 0.0), (-3.0, 0.0), (0.0, 0.0),
                     (7.25, 7.25), (1e300, 1e300)):
        hot, _, got = _load(warm_lib, _encode(warm_lib, nr, m, digest, nu, B), nr, m, digest)
        assert hot and got == want, nu
    # a non-symmetric B: its lower triangle, mirrored
    G = rng.normal(size=(nr, nr))
    hot, B2, _ = _load(warm_lib, _encode(warm_lib, nr, m, digest, 1.0, G), nr, m, digest)
    L = np.tril(G)
    assert hot and np.array_equal(B2, L + np.tril(G, -1).T)


def test_digest_is_fnv1a_of_the_reduced_form(warm_lib):
    rng = np.random.default_rng(3)
    nC, nr, m = 22, 10, 83
    li = np.array([1, 4, 9], dtype=np.int32)
    N = rng.normal(size=(nr, nC))

    def dig(nC_, nr_, m_, li_, N_):
        N_ = np.ascontiguousarray(N_, dtype=np.float64)
        li_ = np.ascontiguousarray(li_, dtype=np.int32)
        return warm_lib.warm_host_digest(nC_, nr_, m_, len(li_), li_.ctypes.data_as(C.POINTER(C.c_int)), _dp(N_))

    d = dig(nC, nr, m, li, N)
    data = np.array([nC, nr, m, len(li)], dtype="<i4").tobytes() + li.astype("<i4").tobytes() + N.astype("<f8").tobytes()
    assert d == _fnv1a(data)
    assert dig(nC, nr, m, li, N.copy()) == d
    N2 = N.copy()
    N2.flat[37] = np.nextafter(N2.flat[37], np.inf)
    others = {dig(nC, nr, m, li, N2), dig(nC, nr, m + 1, li, N), dig(nC, nr, m, li[:2], N), dig(nC, nr, m, li + 1, N)}
    assert d not in others and len(others) == 4


# ---- warm re-solve of a moved MPC problem -------------------------------------------------------------

def _with_bounds(spec, lo, up):
    kw = {f.name: getattr(spec, f.name) for f in dataclasses.fields(spec)}
    kw.update(lowerb=np.asarray(lo, dtype=np.float64).copy(), upperb=np.asarray(up, dtype=np.float64).copy())
    return type(spec)(**kw)


def test_warm_resolve_after_moving_x0_matches_cold_in_fewer_iterations(warm_lib, core_lib, port):
    """the active-bound lane change: solve cold, move the initial state along the solution by dt, re-solve
    cold and warm (B and nu of the first solve, through a row of the warm format).  Both reach the same
    KKT point of the moved problem; the warm solves take fewer iterations in total."""
    from ntg_b200 import configs
    from test_gpu_next import _kincar_active_constraints
    spec = _kincar_active_constraints()
    X = configs.coefficients("cfg3", 512, spec, seed=5)
    nlp = ReducedNLP(port, spec)
    nr, m, dt = nlp.nr, nlp.m, 0.1
    digest = 0x0123456789ABCDEF
    ncoef = spec.nC // 2
    cold_its = warm_its = 0
    for p in range(8):
        a = sqp_via_core_warm(core_lib, nlp, nlp.N.T @ (X[p] - nlp.Cpart), max_iter=100)
        assert a["status"] == 1, p
        x0 = np.concatenate([port.spline_interp(dt, spec.knots[j], a["C"][j * ncoef:(j + 1) * ncoef], spec.order[j],
                                                spec.mult[j], spec.maxderiv[j]) for j in range(2)])
        lo, up = spec.lowerb.copy(), spec.upperb.copy()
        lo[:6] = up[:6] = x0
        moved = ReducedNLP(port, _with_bounds(spec, lo, up))
        assert np.array_equal(moved.N, nlp.N)      # the reduced space does not depend on the bounds
        y0 = moved.N.T @ (a["C"] - moved.Cpart)
        hot, B, nu = _load(warm_lib, _encode(warm_lib, nr, m, digest, a["nu"], a["B"]), nr, m, digest)
        assert hot and a["nu"] > 0
        c = sqp_via_core(core_lib, moved, y0, max_iter=100)
        w = sqp_via_core_warm(core_lib, moved, y0, B0=B, nu0=nu, max_iter=100)
        assert c["status"] == 1 and w["status"] == 1, p
        assert abs(w["f"] - c["f"]) <= 1e-7 * max(1.0, abs(c["f"])), p
        assert np.array_equal(w["istate"], c["istate"]), p
        assert w["viol"] <= 1e-7
        cold_its += c["iters"]
        warm_its += w["iters"]
    print(f"iterations after moving x0 by {dt}: cold {cold_its}, warm {warm_its}")
    assert warm_its < cold_its
