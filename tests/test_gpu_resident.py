"""The device-resident solve (whole minimize() = ONE persistent kernel launch; line search / convergence / curvature gate decided
on the device, pair update folded into the first apply_Hv pass, first trial of every search folded into the second) against the
CPU checker and the frozen outputs of the unmodified reference headers -- the same parity bar as the host-driven loop
(test_gpu_solver.py): same iteration and evaluation counts, |fx - fx_cpu| <= 1e-10 max(1, |fx_cpu|), x to 1e-8..1e-6, the trace of f
within a tolerance that starts at 1e-10, and the reference's exception (type + message) on the error paths."""
import numpy as np
import pytest

import lbfgspp_b200 as lb
import pyoracle as po
from test_gpu_solver import check_parity, cpu_param
from util import LS, golden_cases, unhex

pytestmark = pytest.mark.gpu
LS_NAMES = ["Backtracking", "Bracketing", "NocedalWright", "MoreThuente"]


def resident(prm, ls, dtype=np.float64):
    return lb.LBFGSSolver(prm, ls, dtype=dtype, resident=True)


@pytest.mark.parametrize("ls", LS_NAMES)
@pytest.mark.parametrize("n", [10, 4098, 100000])
def test_resident_matches_cpu_checker(orc, ls, n):
    prm = lb.LBFGSParam(m=10 if n > 10 else 6)
    g = resident(prm, ls).minimize(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(n))
    c = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(n), LS[ls], cpu_param(orc, prm), sum_mode=po.SUM_LANES8)
    check_parity(g, c, xtol=1e-7)
    assert g["launches"] == 1      # one kernel launch per minimize()


def test_resident_other_objectives(orc):
    n = 20000
    d, b, xs = po.quad_tridiag_data(n, kappa=1e3, seed=0)   # config 3's shape at a size where the reference's run ends normally
    prm = lb.LBFGSParam(m=20)
    g = resident(prm, "Bracketing").minimize(lb.OBJ_QUAD_TRIDIAG, np.zeros(n), data0=d, data1=b)
    c = orc.lbfgs(po.OBJ_QUAD_TRIDIAG, np.zeros(n), LS["Bracketing"], cpu_param(orc, prm), data0=d, data1=b)
    assert g["status"] == c["status"] == "ok"
    assert abs(g["fx"] - c["fx"]) <= 1e-9 * abs(c["fx"]) and abs(g["niter"] - c["niter"]) <= max(3, c["niter"] // 20)
    prm = lb.LBFGSParam()
    g = resident(prm, "NocedalWright").minimize(lb.OBJ_ROSENBROCK_CHAINED, np.full(300, 1.3))
    c = orc.lbfgs(po.OBJ_ROSENBROCK_CHAINED, np.full(300, 1.3), LS["NocedalWright"], cpu_param(orc, prm))
    check_parity(g, c, xtol=1e-6)
    g = resident(prm, "NocedalWright").minimize(lb.OBJ_QUAD_SHIFT, np.zeros(10))
    assert g["niter"] == 2 and np.allclose(g["x"], np.arange(10.0), atol=1e-12)


def test_resident_random_start(orc):
    x0 = np.random.default_rng(3).uniform(-1, 1, 2000)
    prm = lb.LBFGSParam(m=7, max_linesearch=64)
    g = resident(prm, "MoreThuente").minimize(lb.OBJ_ROSENBROCK_PAIRED, x0)
    c = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, x0, LS["MoreThuente"], cpu_param(orc, prm))
    assert g["status"] == c["status"] == "ok"
    if c["niter"] <= 60:
        check_parity(g, c, xtol=1e-6)
    else:   # chaotic regime (a ~200-iteration run: the checker's own count moves by 10+ % between summation orders): the stop rule of
        # LBFGS.h:137-140 must hold at the returned point, near x* = 1, after a comparable number of iterations
        assert g["gnorm"] <= max(prm.epsilon, prm.epsilon_rel * np.linalg.norm(g["x"])) * (1 + 1e-12)
        assert np.max(np.abs(g["x"] - 1.0)) <= 2e-3 and g["fx"] <= 1e-5
        assert 0.7 * c["niter"] <= g["niter"] <= 1.4 * c["niter"]


def test_resident_float32(orc):
    prm = lb.LBFGSParam()
    g = resident(prm, "NocedalWright", dtype=np.float32).minimize(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(64))
    c = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(64), LS["NocedalWright"], cpu_param(orc, prm), dtype=np.float32)
    assert g["status"] == "ok" and abs(g["niter"] - c["niter"]) <= 3 and np.max(np.abs(g["x"] - 1.0)) <= 1e-2


def test_resident_stopping_rules_and_error_paths(orc):
    for prm, ls in ((lb.LBFGSParam(max_iterations=5), "NocedalWright"), (lb.LBFGSParam(past=3, delta=1e-6), "MoreThuente"),
                    (lb.LBFGSParam(max_linesearch=1), "Backtracking"), (lb.LBFGSParam(max_linesearch=1), "Bracketing"),
                    (lb.LBFGSParam(max_linesearch=1, max_iterations=3), "MoreThuente"),
                    (lb.LBFGSParam(max_linesearch=1, max_iterations=3), "NocedalWright"),
                    (lb.LBFGSParam(linesearch=1), "NocedalWright"), (lb.LBFGSParam(linesearch=1, max_linesearch=64), "Backtracking"),
                    (lb.LBFGSParam(linesearch=2, max_linesearch=64), "Bracketing"), (lb.LBFGSParam(m=0), "MoreThuente"),
                    (lb.LBFGSParam(max_step=0.5), "MoreThuente"), (lb.LBFGSParam(min_step=10.0), "MoreThuente")):
        g = resident(prm, ls).minimize(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(12))
        c = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(12), LS[ls], cpu_param(orc, prm))
        check_parity(g, c, xtol=1e-6)
    # start point already optimal: minimize returns 1 without a line search
    g = resident(lb.LBFGSParam(), "MoreThuente").minimize(lb.OBJ_ROSENBROCK_PAIRED, np.ones(6))
    assert g["status"] == "ok" and g["niter"] == 1 and g["nfev"] == 1


@pytest.mark.parametrize("case", [c for c in golden_cases("lbfgs") if c["dtype"] == "f64"], ids=lambda c: c["name"])
def test_resident_on_golden_cases(case):
    """Frozen outputs of the unmodified reference headers (tests/golden/make_golden.py)."""
    prm = lb.LBFGSParam(**case["param"])
    d0, d1 = (unhex(case["data"][0]), unhex(case["data"][1])) if case["data"] else (None, None)
    g = resident(prm, case["ls"]).minimize(case["objective"], unhex(case["x0"]), data0=d0, data1=d1)
    c = dict(status=case["status"], msg=case["msg"], niter=case["niter"], nfev=case["nfev"], fx=float.fromhex(case["fx"]),
             x=unhex(case["x"]), trace=unhex(case["trace"]))
    if case["niter"] > 60:  # chaotic regime: compare the optimum, not the path
        assert g["status"] == c["status"] and abs(g["fx"] - c["fx"]) <= 1e-9 * max(1.0, abs(c["fx"]))
    else:
        check_parity(g, c, xtol=1e-6)


@pytest.mark.parametrize("ls", LS_NAMES)
def test_host_loop_agrees_with_resident_to_rounding(ls):
    """Two independent drivers of the same kernels' arithmetic (host-driven loop with separate launches per pass / persistent
    kernel): same counts, fx within the parity tolerance on a well-conditioned run."""
    n = 100000
    prm = lb.LBFGSParam(m=10)
    host = lb.LBFGSSolver(prm, ls, resident=False).minimize(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(n))
    res = lb.LBFGSSolver(prm, ls, resident=True).minimize(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(n))
    assert host["status"] == res["status"] == "ok"
    assert (host["niter"], host["nfev"]) == (res["niter"], res["nfev"])
    assert abs(host["fx"] - res["fx"]) <= 1e-10 * max(1.0, abs(res["fx"]))
    assert np.max(np.abs(host["x"] - res["x"])) <= 1e-8


def test_resident_solve_is_bitwise_repeatable():
    x0 = np.random.default_rng(5).uniform(-1, 1, 30000)
    a = resident(lb.LBFGSParam(m=10), "MoreThuente").minimize(lb.OBJ_ROSENBROCK_PAIRED, x0)
    b = resident(lb.LBFGSParam(m=10), "MoreThuente").minimize(lb.OBJ_ROSENBROCK_PAIRED, x0)
    assert (a["niter"], a["nfev"], a["fx"]) == (b["niter"], b["nfev"], b["fx"])
    assert np.array_equal(a["x"], b["x"]) and np.array_equal(a["trace"], b["trace"])


def test_final_approx_hessian_after_resident_solve():
    """final_approx_hessian() / final_approx_inverse_hessian() (reference LBFGS.h:192-197) must describe the solve that just ran, also
    when that solve was device-resident (its S/Y ring lives in the solver, tiled; the front fetches a column-major copy on demand)."""
    x0 = np.zeros(10)
    it_r, x_r, B_r, H_r = lb.solve_dense(lb.OBJ_ROSENBROCK_PAIRED, x0, lb.LBFGSParam(), "NocedalWright", resident=True)
    it_h, x_h, B_h, H_h = lb.solve_dense(lb.OBJ_ROSENBROCK_PAIRED, x0, lb.LBFGSParam(), "NocedalWright", resident=False)
    assert it_r == it_h and np.max(np.abs(x_r - x_h)) <= 1e-8
    scale = np.max(np.abs(B_h))
    assert np.max(np.abs(B_r - B_h)) <= 1e-6 * scale and np.max(np.abs(H_r - H_h)) <= 1e-6 * np.max(np.abs(H_h))
    assert np.max(np.abs(B_r - B_r.T)) <= 1e-9 * scale                      # symmetric
    assert np.max(np.abs(B_r @ H_r - np.eye(10))) <= 1e-6                   # H = inv(B)
    # a second solve on the same solver type from another start must refresh the matrices
    it2, _, B2, _ = lb.solve_dense(lb.OBJ_ROSENBROCK_PAIRED, np.full(10, 0.5), lb.LBFGSParam(), "NocedalWright", resident=True)
    assert it2 > 1 and np.max(np.abs(B2 - B_r)) > 0


@pytest.mark.parametrize("m,iters", [(30, 45), (64, 80)])
def test_resident_large_history(orc, m, iters):
    """History sizes beyond one column pair per warp (m > 24: the dots pass works in rounds; the tiled history uses short blocks):
    the first `iters` iterations of the tridiagonal quadratic, evaluation by evaluation against the CPU checker."""
    n = 30000
    d, b, _ = po.quad_tridiag_data(n, kappa=1e3, seed=3)
    prm = lb.LBFGSParam(m=m, max_iterations=iters)
    g = resident(prm, "Bracketing").minimize(lb.OBJ_QUAD_TRIDIAG, np.zeros(n), data0=d, data1=b)
    c = orc.lbfgs(po.OBJ_QUAD_TRIDIAG, np.zeros(n), LS["Bracketing"], cpu_param(orc, prm), data0=d, data1=b)
    assert g["status"] == c["status"] == "ok"
    assert (g["niter"], g["nfev"]) == (c["niter"], c["nfev"]) == (iters, c["nfev"])
    k = min(len(g["trace"]), len(c["trace"]))
    rel = np.abs(g["trace"][1:k] - c["trace"][1:k]) / np.abs(c["trace"][1:k])
    assert np.max(rel) <= 1e-9, np.max(rel)
    h = lb.LBFGSSolver(prm, "Bracketing", resident=False).minimize(lb.OBJ_QUAD_TRIDIAG, np.zeros(n), data0=d, data1=b)
    assert (h["niter"], h["nfev"]) == (g["niter"], g["nfev"]) and abs(h["fx"] - g["fx"]) <= 1e-9 * abs(g["fx"])


@pytest.mark.parametrize("resident_loop", [True, False])
def test_session_download_returns_the_last_solve(resident_loop):
    """Session.download() after a solve that left x on the device gives the x that the same solve copies back with to_host=True."""
    n = 4098
    prm = lb.LBFGSParam(m=10)
    sess = lb.Session(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(n), prm, "MoreThuente", resident=resident_loop)
    r = sess.solve()
    x = sess.download()
    r2 = sess.solve(to_host=True)
    x2 = sess.result()
    sess.close()
    lone = lb.LBFGSSolver(prm, "MoreThuente", resident=resident_loop).minimize(lb.OBJ_ROSENBROCK_PAIRED, np.zeros(n))
    assert (r["niter"], r["nfev"], r["fx"]) == (r2["niter"], r2["nfev"], r2["fx"])
    assert np.array_equal(x, x2)
    assert (r["niter"], r["nfev"]) == (lone["niter"], lone["nfev"]) and np.max(np.abs(x - lone["x"])) <= 1e-8
