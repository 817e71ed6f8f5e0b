"""The oracle port (oracle/ntg_oracle.c) against the committed golden vectors
generated from the UNMODIFIED reference (tests/golden/make_golden.py), bit for bit."""
import os

import numpy as np
import pytest

from common import GOLDEN, GOLDEN_CASES, assert_bitexact, golden_module, golden_spec, load_golden
from ntg_b200 import configs


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_port_matches_golden_bit_exact(port, name):
    spec, X = golden_spec(name)
    g = load_golden(name)
    assert_bitexact(X, g["X"], "seeded inputs reproduce")
    r = port.eval(spec, X, dense=False, band=True, linear=True)
    for k in ("f", "g", "c", "Jband", "A", "bl", "bu"):
        assert_bitexact(r[k], g[k], f"{name}.{k}")
    B, off, col0 = port.tables(spec)
    for j, b in enumerate(B):
        assert_bitexact(b, g["B"][j], f"{name}.B{j}")
    assert_bitexact(off, g["off"], f"{name}.offset (knot-interval indices)")
    assert_bitexact(col0, g["col0"], f"{name}.col0 (Jacobian pattern)")


@pytest.mark.parametrize("name", ["cfg2_vanderpol", "cfg4_kincar64", "syn6_small", "endpoint"])
def test_port_matches_reference_bit_exact(port, name):
    """The golden rows and five more against the reference's outputs for them (rows_<name>.npz: f, g, c;
    band and dense Jacobians, NaN where the reference never writes, by the sha256 of their bytes); the
    linear rows, bounds and tables against <name>.npz."""
    gm = golden_module()
    spec, X = gm.row_inputs(name)
    want = np.load(os.path.join(GOLDEN, f"rows_{name}.npz"))
    assert gm.digest(X) == str(want["X_sha256"]), "seeded inputs reproduce"
    b = port.eval(spec, X, linear=True)
    assert b["pattern_bad"] == 0, "wrote outside / skipped inside the expected band"
    for k in ("f", "g", "c"):
        assert_bitexact(b[k], want[k], f"{name}.{k}")
    g = load_golden(name)
    assert_bitexact(b["Jband"][:g["X"].shape[0]], g["Jband"], f"{name}.Jband (golden rows)")
    for k in ("Jband", "Jdense"):
        assert gm.digest(b[k]) == str(want[k + "_sha256"]), f"{name}.{k}: not bit-identical to the reference"
    for k in ("A", "bl", "bu"):
        assert_bitexact(b[k], g[k], f"{name}.{k}")
    Bb, offb, colb = port.tables(spec)
    for j, x in enumerate(Bb):
        assert_bitexact(x, g["B"][j], "tables")
    assert_bitexact(offb, g["off"], "offsets")
    assert_bitexact(colb, g["col0"], "pattern")


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_port_modes_match_reference(port, mode):
    """mode 0 values only, 1 derivatives only, 2 both (reference src/ntg.c:294-334, :354-370), against
    the reference's outputs in each mode (endpoint_modes.npz; mode 2 is endpoint.npz).
    The reference crashes in funcon mode 1 with trajectory constraints (writes through
    C == NULL, src/constraints.c:152-153), so mode 1 is compared on the objective only."""
    gm = golden_module()
    spec, X = golden_spec("endpoint")
    m = np.load(os.path.join(GOLDEN, "endpoint_modes.npz"))
    assert gm.digest(X) == str(m["X_sha256"]), "seeded inputs reproduce"
    e = load_golden("endpoint")
    want = {0: {"f": m["mode0_f"], "c": m["mode0_c"]}, 1: {"g": m["mode1_g"]},
            2: {k: e[k] for k in ("f", "c", "g", "Jband")}}[mode]
    mc = mode if mode != 1 else -1
    b = port.eval(spec, X, mode_obj=mode, mode_con=mc)
    for k, v in want.items():
        assert_bitexact(b[k], v, k)
    full = port.eval(spec, X)
    if mode == 1:
        b1 = port.eval(spec, X, mode_obj=1, mode_con=1)
        assert_bitexact(b1["g"], full["g"], "mode-1 gradient equals mode-2 gradient")
        assert_bitexact(b1["Jband"], full["Jband"], "mode-1 Jacobian equals mode-2 Jacobian")


def test_reference_examples_known_answers(port):
    """SURVEY.md section 8(c)(4): examples/vanderpol.c at its shipped initial guess has
    objective bps[19]-bps[0] and a gradient summing to 10; kincar at ones(14) has zero cost.
    The fixtures hold what the reference's own build of the two example programs returned; the
    port evaluates the problems they pose (20 breakpoints, no nonlinear constraints) and must
    reproduce them bit for bit."""
    def run(spec, ex):
        r = port.eval(spec, ex["X"], mode_con=-1, dense=False, band=False, linear=True)
        assert [spec.nC, spec.nclin, spec.ncnln] == list(ex["dims"])
        for k in ("f", "g", "A", "bl", "bu"):
            assert_bitexact(r[k], ex[k], f"example fixture reproduces: {k}")
        return r
    r = run(configs.vanderpol(20, constraints=False), load_golden("example_vanderpol"))
    # the survey's independent derivation (5.0000000000000036) is good to ~1e-14; the reference itself
    # returns the trapezoid sum of a constant 1 over the accumulated breakpoints
    assert abs(r["f"][0] - 5.0000000000000036) < 1e-14 and r["f"][0] == 5.000000000000001
    np.testing.assert_allclose(r["g"][0], [2.62731102431688, -0.64058440312766, 2.01328105217118,
                                           1.99998465327921, 2.01328105217118, -0.64058440312767,
                                           2.62731102431689], rtol=0, atol=2e-14)
    np.testing.assert_allclose(r["f"][1], 12.92863341437716, rtol=1e-14)
    rk = run(configs.kincar(20, constraints=False), load_golden("example_kincar"))
    assert abs(rk["f"][0]) < 1e-25 and np.abs(rk["g"][0]).max() < 1e-14


def test_bytes_per_eval_match_baseline_md():
    """BASELINE.md table: 1080 / 3752 / 11496 / 705960 B per eval."""
    want = {"cfg2": 1080, "cfg3": 3752, "cfg4": 11496, "cfg5": 705960}
    for cfg, b in want.items():
        assert configs.get(cfg)[0].bytes_per_eval() == b
