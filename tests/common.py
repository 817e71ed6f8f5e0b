"""Shared helpers for the parity tests."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# BASELINE.json north_star: "within 1e-12 relative (1e-14 absolute near zero)".
# The absolute clause is scaled by the infinity norm of the vector compared
# (SURVEY.md section 7, hard part 2 / section 8(c)).
RTOL = 1e-12
ATOL_SCALE = 1e-14


def assert_close(a, ref, what=""):
    a = np.asarray(a, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert a.shape == ref.shape, f"{what}: shape {a.shape} vs {ref.shape}"
    if ref.size == 0:
        return
    assert np.array_equal(np.isnan(a), np.isnan(ref)), f"{what}: NaN pattern differs"
    scale = np.nanmax(np.abs(ref))
    tol = RTOL * np.abs(ref) + ATOL_SCALE * scale
    err = np.abs(a - ref)
    bad = np.nan_to_num(err - tol, nan=0.0) > 0
    if bad.any():
        i = np.unravel_index(np.nanargmax(err - tol), err.shape)
        raise AssertionError(f"{what}: {bad.sum()} entries outside 1e-12*|ref| + 1e-14*|ref|_inf; "
                             f"worst at {i}: got {a[i]!r} ref {ref[i]!r}")


def assert_bitexact(a, ref, what=""):
    a = np.asarray(a)
    ref = np.asarray(ref)
    assert a.shape == ref.shape, f"{what}: shape {a.shape} vs {ref.shape}"
    if not np.array_equal(a, ref, equal_nan=True):
        d = np.nanmax(np.abs(a.astype(np.float64) - ref.astype(np.float64)))
        raise AssertionError(f"{what}: not bit-identical (max |diff| = {d:.3e}, "
                             f"{(a != ref).sum()} of {a.size} entries differ)")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    d = {k: z[k] for k in z.files}
    d["B"] = [d[f"B{j}"] for j in range(sum(k.startswith("B") and k[1:].isdigit() for k in d))]
    return d


def golden_module():
    """tests/golden/make_golden.py: the seeded inputs of every fixture"""
    import importlib.util
    p = os.path.join(GOLDEN, "make_golden.py")
    spec = importlib.util.spec_from_file_location("make_golden", p)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def golden_spec(name):
    return golden_module().case_inputs(name)


GOLDEN_CASES = ["cfg2_vanderpol", "cfg3_kincar", "cfg4_kincar64", "cfg5_syn6", "syn6_small", "endpoint"]


def violation(spec, c):
    """max over nonlinear rows of max(lb-c, c-ub, 0), bounds expanded like bounds()
    (reference src/constraints.c:24-30)."""
    nlin = spec.nlic + spec.nltc + spec.nlfc
    lo, hi = np.asarray(spec.lowerb)[nlin:], np.asarray(spec.upperb)[nlin:]
    rep = [1] * spec.nnlic + [spec.nbps] * spec.nnltc + [1] * spec.nnlfc
    lb, ub = np.repeat(lo, rep), np.repeat(hi, rep)
    if c.shape[1] == 0:
        return np.zeros(c.shape[0])
    return np.maximum(np.maximum(lb - c, c - ub), 0.0).max(axis=1)
