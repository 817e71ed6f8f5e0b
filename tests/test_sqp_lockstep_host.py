"""CPU checks of the lock-step SQP driver (tests/tools/sqp_lockstep.py) that tests/test_gpu_sqp_lockstep.py
compares the GPU solver with: its restatement of reduce_linear gives an orthonormal basis of the null space
and a right operator for Cpart, the driver adds only the GPU's bookkeeping to the iteration of sqp_via_core,
and it converges on every shape the GPU test runs."""
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
from sqp_lockstep import Core, Reduced, fnv1a, lockstep, reduce_linear, sqp_smem_bytes  # noqa: E402
from sqp_reference import ReducedNLP, sqp_via_core  # noqa: E402
from ntg_b200 import configs  # noqa: E402


def _build(tmp_path_factory, src):
    so = str(tmp_path_factory.mktemp("lockstep") / (src + ".so"))
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "ntg_b200", "csrc"),
                           "-o", so, os.path.join(HERE, "tools", src)])
    return C.CDLL(so)


@pytest.fixture(scope="module")
def core_lib(tmp_path_factory):
    return _build(tmp_path_factory, "sqp_host.cpp")


def _kincar(nbps=40, ninterv=4):
    from test_gpu_next import _kincar_active_constraints
    return _kincar_active_constraints(nbps=nbps, ninterv=ninterv)


# the shapes of tests/test_gpu_sqp_lockstep.py: (spec, starts); high-order starts are small, because from
# +-0.5 with these fine knots the core itself stops at its first iteration
SHAPES = {
    "kincar_tiled301": (lambda: _kincar(301, 4), "cfg3"),
    "kincar_nr30": (lambda: _kincar(40, 9), "cfg3"),
    "kincar_nr34": (lambda: _kincar(40, 10), "cfg3"),
    "hi_nr31": (lambda: configs.high_order(5, 3, 14, 33, name="lock_hi31"), 0.01),
    "hi_nr32": (lambda: configs.high_order(4, 2, 15, 33, name="lock_hi32"), 0.05),
    "hi_nr63": (lambda: configs.high_order(6, 3, 20, 65, name="lock_hi63"), 0.01),
    "hi_nr64": (lambda: configs.high_order(4, 2, 31, 65, name="lock_hi64"), 0.05),
    "hi_nr66": (lambda: configs.high_order(4, 2, 32, 81, name="lock_hi66"), 0.01),
    "hi_nr70": (lambda: configs.high_order(4, 2, 34, 81, name="lock_hi70"), 0.05),
    "hi_nr72": (lambda: configs.high_order(4, 2, 35, 81, name="lock_hi72"), 0.01),
    "endpoint": (lambda: configs.endpoint(), 0.5),
}


def starts(spec, kind, P, seed):
    if kind == "cfg3":
        return configs.coefficients("cfg3", P, spec, seed=seed)
    return np.random.default_rng(seed).uniform(-kind, kind, (P, spec.nC))


def test_restated_basis(port, tmp_path_factory):
    """N N' = I and A_eq N' = 0; A_eq Mop b = b on consistent rows, and a dependent row gets a zero column
    of Mop; N spans the same space as the SVD basis of sqp_reference; the digest is the library's FNV-1a"""
    for spec in (_kincar(40, 4), _kincar(301, 4), _kincar(40, 10), configs.kincar(64, constraints=False, name="lock_k64")):
        red = Reduced(port, spec)
        nr, Ae = red.nr, red.Ae
        assert nr == spec.nC - len(red.eq) and red.N.shape == (nr, spec.nC)
        assert np.abs(red.N @ red.N.T - np.eye(nr)).max() <= 1e-14
        assert np.abs(Ae @ red.N.T).max() <= 1e-14 * max(1.0, np.abs(Ae).max())
        b = np.random.default_rng(0).uniform(-5, 5, len(red.eq))
        assert np.abs(Ae @ (red.Mop @ b) - b).max() <= 1e-13 * (1 + np.abs(b).max())
        svd = ReducedNLP(port, spec).N
        assert np.abs(svd @ svd.T - red.N.T @ red.N).max() <= 1e-13
    # a duplicated initial row: rank 12 of 13 rows; one of the two copies gets a zero column
    base = configs.kincar(64, constraints=False, name="lock_dup")
    kw = {f.name: getattr(base, f.name) for f in dataclasses.fields(base)}
    b0 = np.concatenate([base.lowerb[:6], base.lowerb[3:4], base.lowerb[6:]])
    kw.update(lic=np.vstack([base.lic, base.lic[3:4]]), lowerb=b0.copy(), upperb=b0.copy())
    red = Reduced(port, type(base)(**kw))
    assert len(red.eq) == 13 and red.nr == base.nC - 12
    zero = [j for j in range(13) if not red.Mop[:, j].any()]
    assert len(zero) == 1 and zero[0] in (3, 6)
    b = np.random.default_rng(1).uniform(-5, 5, 13)
    b[6] = b[3]
    assert np.abs(red.Ae @ (red.Mop @ b) - b).max() <= 1e-13 * (1 + np.abs(b).max())
    assert np.array_equal(red.Mop @ b, red.Mop @ np.where(np.arange(13) == zero[0], 99.0, b))
    # the digest, against the header's own FNV-1a compiled with g++ (tests/tools/warm_host.cpp)
    lib = _build(tmp_path_factory, "warm_host.cpp")
    lib.warm_host_digest.restype = C.c_uint64
    lib.warm_host_digest.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_int), C.POINTER(C.c_double)]
    red = Reduced(port, configs.endpoint())
    li = np.ascontiguousarray(red.li, dtype=np.int32)
    N = np.ascontiguousarray(red.N)
    d = lib.warm_host_digest(red.nC, red.nr, red.m, red.n_li, li.ctypes.data_as(C.POINTER(C.c_int)),
                             N.ctypes.data_as(C.POINTER(C.c_double)))
    assert d == red.digest() and red.n_li == configs.endpoint().nclin and red.nr == red.nC
    assert fnv1a(b"") == 14695981039346656037


def test_reduce_linear_is_deterministic_on_random_rows():
    """random rows, some of them dependent: the restatement gives an orthonormal null-space basis and an
    Mop whose dependent columns are zero, and it is a pure function of its input"""
    rng = np.random.default_rng(4)
    for trial in range(20):
        m = int(rng.integers(1, 10))
        n = m + int(rng.integers(1, 10))
        A = rng.normal(size=(m, n))
        if m > 2:
            A[-1] = A[0] - 2.0 * A[1]
        N, Cp, Mop, r = reduce_linear(A, np.zeros(m))
        assert r == np.linalg.matrix_rank(A) and N.shape == (n - r, n)
        assert np.abs(N @ N.T - np.eye(n - r)).max() <= 1e-14 and np.abs(A @ N.T).max() <= 1e-13
        assert (np.abs(Mop).sum(axis=0) == 0).sum() == m - r
        b = A @ rng.normal(size=n)
        assert np.abs(A @ (Mop @ b) - b).max() <= 1e-12 * (1 + np.abs(b).max())
        N2, _, Mop2, _ = reduce_linear(A.copy(), np.zeros(m))
        assert np.array_equal(N, N2) and np.array_equal(Mop, Mop2)


@pytest.mark.parametrize("name", ["kincar40", "kincar_tiled301", "kincar_nr34"])
def test_lockstep_without_stage2_is_sqp_via_core(core_lib, port, name):
    """with no stage-2 step taken, the lock-step driver and sqp_via_core (same basis, same core) end at the
    same point after the same iterations and with the same active set: the driver adds nothing but the GPU's
    bookkeeping"""
    spec = {"kincar40": lambda: _kincar(40, 4), "kincar_tiled301": lambda: _kincar(301, 4),
            "kincar_nr34": lambda: _kincar(40, 10)}[name]()
    red = Reduced(port, spec)
    nlp = ReducedNLP(port, spec)
    nlp.N, nlp.Cpart = red.N.T.copy(), red.Cpart.copy()
    X = configs.coefficients("cfg3", 3, spec, seed=5)
    core = Core(core_lib)
    for p in range(3):
        r = lockstep(core, red, X[p], 150)
        last = r["snaps"][-1]
        assert last["status"] == 1 and all(s["a"] < 4 for s in r["steps"]), (name, p)
        b = sqp_via_core(core_lib, nlp, red.N @ (X[p] - red.Cpart), max_iter=150)
        assert b["status"] == 1 and b["iters"] == last["iters"] + 1, (name, p, b["iters"], last["iters"])
        # the two form C = Cpart + N y with differently laid out N: the last bits may differ
        assert np.abs(b["C"] - last["C"]).max() <= 1e-13 * max(1.0, np.abs(last["C"]).max()), (name, p)
        np.testing.assert_array_equal(b["istate"], last["istate"][spec.nclin:])


@pytest.mark.parametrize("name", list(SHAPES))
def test_lockstep_converges_on_gpu_shapes(core_lib, port, name):
    """the driver converges from the starts the GPU test uses; the cases are the CTA shapes of k_sqp_step
    (32 / 64 threads, nr below / above the thread count) and all fit in 227 KB of shared memory"""
    make, kind = SHAPES[name]
    spec = make()
    red = Reduced(port, spec)
    assert sqp_smem_bytes(red.nr, red.m) <= 227 * 1024
    X = starts(spec, kind, 4, seed=5 if kind == "cfg3" else 1)
    core = Core(core_lib)
    for p in range(2):
        last = lockstep(core, red, X[p], 250)["snaps"][-1]
        assert last["status"] == 1, (name, p, last["status"], last["iters"])
        assert last["viol"] <= 1e-8


def test_endpoint_300_is_over_the_shared_memory_limit(port):
    red = Reduced(port, configs.endpoint(300, name="lock_ep300"))
    assert (red.nr, red.m) == (18, 1207) and sqp_smem_bytes(red.nr, red.m) > 227 * 1024
