"""CPU tests of the checker itself: the restatement must reproduce the unmodified reference headers run over minieigen, bit
for bit, on the inputs whose results were frozen from that build (golden/lbfgs_ref.json, golden/pins_ref.json)."""
import numpy as np
import pytest

import pyoracle as po
from util import LS, fingerprint, golden_cases, golden_pins, pin_cases, unhex


def run_golden_lbfgs(orc, c):
    dtype = np.float64 if c["dtype"] == "f64" else np.float32
    p = orc.default_param(**c["param"])
    d0, d1 = (unhex(c["data"][0]), unhex(c["data"][1])) if c["data"] else (None, None)
    return orc.lbfgs(c["objective"], unhex(c["x0"]), LS[c["ls"]], p, data0=d0, data1=d1, dtype=dtype)


@pytest.mark.parametrize("case", golden_cases("lbfgs"), ids=lambda c: c["name"])
def test_restatement_matches_golden_lbfgs(orc, case):
    r = run_golden_lbfgs(orc, case)
    assert r["status"] == case["status"] and r["msg"] == case["msg"]
    assert (r["niter"], r["nfev"]) == (case["niter"], case["nfev"])
    assert np.array_equal(r["trace"], unhex(case["trace"]))
    assert np.array_equal(r["x"].astype(np.float64), unhex(case["x"]))
    assert np.array_equal(r["grad"].astype(np.float64), unhex(case["grad"]))
    if case["status"] == "ok":
        assert float(r["fx"]).hex() == case["fx"] and float(r["gnorm"]).hex() == case["gnorm"]


@pytest.mark.parametrize("case", golden_cases("apply_Hv"), ids=lambda c: c["name"])
def test_restatement_matches_golden_apply_Hv(orc, case):
    n, npairs = case["n"], case["npairs"]
    S = unhex(case["S"]).reshape(npairs, n)
    Y = unhex(case["Y"]).reshape(npairs, n)
    res, _, theta = orc.apply_Hv(S, Y, unhex(case["v"]), case["a"], case["m"])
    assert np.array_equal(res, unhex(case["res"]))
    assert float(theta).hex() == case["theta"]


@pytest.mark.parametrize("case", golden_cases("lbfgsb"), ids=lambda c: c["name"])
def test_restatement_matches_golden_lbfgsb(orc, case):
    p = orc.default_param(lbfgsb=True, **case["param"])
    r = orc.lbfgsb(case["objective"], unhex(case["x0"]), unhex(case["lb"]), unhex(case["ub"]), p)
    assert r["status"] == case["status"] and r["msg"] == case["msg"]
    assert (r["niter"], r["nfev"]) == (case["niter"], case["nfev"])
    assert np.array_equal(r["trace"], unhex(case["trace"]))
    assert np.array_equal(r["x"], unhex(case["x"])) and np.array_equal(r["grad"], unhex(case["grad"]))
    assert float(r["fx"]).hex() == case["fx"] and float(r["gnorm"]).hex() == case["gnorm"]


def test_survey_probe_values(orc):
    """BASELINE.md section 4 (independent numpy transliteration): iteration / evaluation counts must agree."""
    expect = {"NocedalWright": (22, 36), "MoreThuente": (21, 28), "Bracketing": (22, 31), "Backtracking": (22, 31)}
    for ls, (it, fev) in expect.items():
        r = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(10), LS[ls], orc.default_param())
        assert (r["niter"], r["nfev"]) == (it, fev)
    r = orc.lbfgs(po.OBJ_QUAD_SHIFT, np.zeros(10), LS["NocedalWright"], orc.default_param())
    assert r["niter"] == 2 and np.allclose(r["x"], np.arange(10.0))
    r = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(1000), LS["MoreThuente"], orc.default_param(m=10))
    assert (r["niter"], r["nfev"]) == (23, 31)


def test_self_checking_examples_property(orc):
    """example-rosenbrock-comparison.cpp:44-51,83-86: |x - 1|_inf <= 1e-4 from random starts, all line searches."""
    rng = np.random.default_rng(7)
    for n in (2, 8, 24):
        for _ in range(16):
            x0 = rng.uniform(-1, 1, n)
            for ls in range(4):
                r = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, x0, ls, orc.default_param(max_linesearch=256))
                assert r["status"] == "ok" and np.max(np.abs(r["x"] - 1.0)) <= 1e-4


def test_lanes_and_omp_modes_agree_with_sequential(orc):
    """Summation-order variants used for the CPU baseline stay within rounding of the faithful one."""
    x0 = np.zeros(2000)
    base = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, x0, 3, orc.default_param(m=10))
    for mode in (po.SUM_LANES8, po.SUM_LANES8_OMP):
        r = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, x0, 3, orc.default_param(m=10), sum_mode=mode)
        assert (r["niter"], r["nfev"]) == (base["niter"], base["nfev"])
        assert abs(r["fx"] - base["fx"]) <= 1e-10 * max(1.0, abs(base["fx"]))
        assert np.max(np.abs(r["x"] - base["x"])) <= 1e-8


def test_gram_form_matches_two_loop_on_cpu(orc):
    """The vector-free (Gram) two-loop is the same recursion up to rounding: same counts, same fx."""
    for n in (10, 1000, 20000):
        a = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(n), 3, orc.default_param(m=10))
        b = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(n), 3, orc.default_param(m=10), gram=True)
        assert (a["niter"], a["nfev"]) == (b["niter"], b["nfev"])
        assert abs(a["fx"] - b["fx"]) <= 1e-10 * max(1.0, abs(a["fx"]))


# ---- against the unmodified reference headers: their results on these inputs, frozen in golden/pins_ref.json ------------------
def check_pins(orc, group):
    frozen = golden_pins(group)
    cases = pin_cases(group)
    assert sorted(name for name, _ in cases) == sorted(frozen)
    for name, run in cases:
        assert fingerprint(run(orc)) == frozen[name], name


def test_pin_against_reference_headers(orc):
    check_pins(orc, "lbfgs")


def test_pin_float32_against_reference_headers(orc):
    check_pins(orc, "lbfgs_f32")


def test_pin_apply_Hv_against_reference_headers(orc):
    check_pins(orc, "apply_Hv")


def test_pin_lbfgsb_against_reference_headers(orc):
    """Cauchy point, subspace minimisation, Bunch-Kaufman LDL' and the L-BFGS-B driver, bit for bit: mixed finite /
    infinite / degenerate (l == u) bounds, history sizes 1..10, 0..10 BOXCQP sweeps, delta-based stopping."""
    check_pins(orc, "lbfgsb")


def test_pin_lbfgsb_larger_against_reference_headers(orc):
    check_pins(orc, "lbfgsb_larger")
    assert all(c["status"] == "ok" for c in golden_pins("lbfgsb_larger").values())


def test_lbfgsb_parameter_and_bound_errors(orc):
    """LBFGSB.h:132-133 (size check) and Param.h:351-376 (check_param) surface as invalid_argument."""
    r = orc.lbfgsb(po.OBJ_QUAD_SHIFT, np.zeros(4), 0.0, 1.0, orc.default_param(lbfgsb=True, m=0))
    assert r["status"] == "invalid_argument" and "'m' must be positive" in r["msg"]
    r = orc.lbfgsb(po.OBJ_QUAD_SHIFT, np.zeros(4), 0.0, 1.0, orc.default_param(lbfgsb=True, max_submin=-1))
    assert r["status"] == "invalid_argument" and "max_submin" in r["msg"]


def test_restatement_is_sanitizer_clean():
    """`make -C oracle sanitize`: the restatement under ASan + UBSan over 552 small solves (all line searches, summation modes,
    L-BFGS-B with mixed bounds)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run(["make", "-C", os.path.join(root, "oracle"), "sanitize"], capture_output=True, text=True, timeout=600)
    if r.returncode != 0 and ("cannot find -lasan" in r.stderr or "cannot find -lubsan" in r.stderr):
        pytest.skip("sanitizer runtimes not installed")
    assert r.returncode == 0 and "selfcheck ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
