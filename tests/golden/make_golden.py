"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED
reference (oracle/_ref, built by `make -C oracle ref` from /root/reference).

Run in the build container only (needs /root/reference):
    python tests/golden/make_golden.py

Each .npz holds the seeded inputs and the reference's own outputs for them:
tables, offsets, Jacobian pattern, f, g, c, band Jacobian, A, bl, bu.  The
reference-example fixtures come from running examples/vanderpol.c and
examples/kincar.c unmodified (their own callbacks, their own setup code).

rows_<case>.npz (more rows, dense Jacobian), endpoint_modes.npz (funobj /
funcon modes 0 and 1) and integrate.npz (IntegrateVector, all three rules) are
what the tests compared against the reference itself while it was built
alongside: main() writes them from the reference.  The committed copies were
recorded from the oracle port and from ntgb_integrate on a B200 at a commit
where both matched the reference bit for bit on exactly these inputs
(write_rows / write_modes / write_integrate take the evaluator to record).
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from ntg_b200 import configs  # noqa: E402
from oracle import oracle  # noqa: E402

CASES = {
    # name: (spec factory, P, coefficient sampler key)
    "cfg2_vanderpol": (lambda: configs.get("cfg2")[0], 8, "cfg2"),
    "cfg3_kincar": (lambda: configs.get("cfg3")[0], 8, "cfg3"),
    "cfg4_kincar64": (lambda: configs.get("cfg4")[0], 4, "cfg4"),
    "cfg5_syn6": (lambda: configs.get("cfg5")[0], 1, "cfg5"),
    "syn6_small": (lambda: configs.syn6(12, name="syn6_small"), 4, "cfg5"),
    "endpoint": (lambda: configs.endpoint(), 8, "endpoint"),
}


def case_inputs(name):
    fac, P, key = CASES[name]
    spec = fac()
    X = configs.coefficients(key, P, spec)
    if name == "cfg2_vanderpol":  # the two known-answer vectors of SURVEY.md section 8(c)
        X[0] = 1.0
        X[1] = [1, .5, -.25, .75, 2, -1, .125]
    return spec, X


ROW_CASES = ["cfg2_vanderpol", "cfg4_kincar64", "syn6_small", "endpoint"]


def row_inputs(name):
    """the golden rows of `name` and five more, seeded"""
    spec, X = case_inputs(name)
    rng = np.random.default_rng(11)
    return spec, np.vstack([X, rng.uniform(-3, 3, (5, spec.nC))])


def digest(a):
    """sha256 of the float64 bytes: a bit-for-bit comparison, NaN payloads included, that keeps large
    Jacobians out of the repository"""
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def write_rows(o):
    for name in ROW_CASES:
        spec, X = row_inputs(name)
        r = o.eval(spec, X, linear=True)
        assert r["pattern_bad"] == 0
        np.savez_compressed(os.path.join(HERE, f"rows_{name}.npz"), X_sha256=digest(X), f=r["f"], g=r["g"],
                            c=r["c"], Jband_sha256=digest(r["Jband"]), Jdense_sha256=digest(r["Jdense"]))


def write_modes(o):
    """modes 0 and 1 on the endpoint case (mode 2 is endpoint.npz).  Mode 1 with trajectory
    constraints is taken for the objective only (funcon mode 1 writes through C == NULL in the
    reference, src/constraints.c:152-153)"""
    spec, X = case_inputs("endpoint")
    m0 = o.eval(spec, X, mode_obj=0, mode_con=0)
    m1 = o.eval(spec, X, mode_obj=1, mode_con=-1)
    np.savez_compressed(os.path.join(HERE, "endpoint_modes.npz"), X_sha256=digest(X), mode0_f=m0["f"],
                        mode0_c=m0["c"], mode1_g=m1["g"])


INTEGRATE_N = (1, 2, 17, 401)
INTEGRATE_ROWS = 37


def integrate_inputs():
    """-> [(t [n] sorted, f [INTEGRATE_ROWS][n])] for n in INTEGRATE_N, seeded"""
    rng = np.random.default_rng(11)
    out = []
    for n in INTEGRATE_N:
        t = np.sort(rng.uniform(0, 3, n))
        out.append((t, rng.normal(size=(INTEGRATE_ROWS, n))))
    return out


def write_integrate(integrate, path=None):
    """integrate(rule, f [rows][n], t [n]) -> [rows]: the FEULER (0), BEULER (1) and TRAPEZOID (2) sums"""
    d = {}
    for t, f in integrate_inputs():
        n = t.size
        d[f"t{n}"] = t
        for rule in (0, 1, 2):
            d[f"I{n}_rule{rule}"] = integrate(rule, f, t)
    np.savez_compressed(path or os.path.join(HERE, "integrate.npz"), **d)


def reference_integrate(ref):
    import ctypes as C

    def integrate(rule, f, t):
        out = np.zeros(f.shape[0])
        for q in range(f.shape[0]):
            I = C.c_double(0.0)
            row = np.ascontiguousarray(f[q])
            ref.lib.IntegrateVector(C.byref(I), row.ctypes.data_as(C.POINTER(C.c_double)),
                                    t.ctypes.data_as(C.POINTER(C.c_double)), t.size, rule)
            out[q] = I.value
        return out
    return integrate


def main():
    os.chdir(HERE)
    ref = oracle.Oracle("ref")
    for name in CASES:
        spec, X = case_inputs(name)
        r = ref.eval(spec, X, dense=False, band=True, linear=True)
        B, off, col0 = ref.tables(spec)
        assert r["pattern_bad"] == 0
        np.savez_compressed(os.path.join(HERE, name + ".npz"), X=X, f=r["f"], g=r["g"], c=r["c"],
                            Jband=r["Jband"], A=r["A"], bl=r["bl"], bu=r["bu"], off=off, col0=col0,
                            **{f"B{j}": b for j, b in enumerate(B)})
        print(name, X.shape, "->", os.path.getsize(os.path.join(HERE, name + ".npz")), "bytes")
    # the reference's own example programs, unmodified
    rng = np.random.default_rng(2024)
    for ex, n in (("vanderpol", 7), ("kincar", 14)):
        X = rng.uniform(-2, 2, (6, n))
        X[0] = 1.0  # the shipped initial guess
        if ex == "vanderpol":
            X[1] = [1, .5, -.25, .75, 2, -1, .125]
        r = oracle.run_reference_example(ex, X)
        assert r["calls"] == 1
        np.savez_compressed(os.path.join(HERE, f"example_{ex}.npz"), X=X, f=r["f"], g=r["g"], A=r["A"],
                            bl=r["bl"], bu=r["bu"], dims=np.array([r["n"], r["nclin"], r["ncnln"]]))
        print("example", ex, r["f"][:2])
    write_rows(ref)
    write_modes(ref)
    write_integrate(reference_integrate(ref))
    if os.path.exists("coef1"):
        os.remove("coef1")


if __name__ == "__main__":
    main()
