import hashlib
import json
import os

import numpy as np

import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
LS = {"Backtracking": 0, "Bracketing": 1, "NocedalWright": 2, "MoreThuente": 3}


def unhex(xs):
    return np.array([float.fromhex(v) for v in xs], dtype=np.float64)


def golden_cases(kind=None):
    with open(os.path.join(HERE, "golden", "lbfgs_ref.json")) as fh:
        cases = json.load(fh)["cases"]
    return [c for c in cases if kind is None or c["kind"] == kind]


# ---- pins of the restatement to the unmodified reference headers ---------------------------------------------------------------
# The reference's results for these inputs are frozen in golden/pins_ref.json (generator golden/make_pins.py); a run's arrays are
# stored as SHA-256 digests of their bytes, so the comparison stays bit for bit while the file stays small.  Whoever changes an
# input here regenerates the file from the reference build.
def fingerprint(r):
    """A result dict as stored in golden/pins_ref.json: arrays as the SHA-256 of their bytes, everything else as it is."""
    return {k: hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest() if isinstance(v, np.ndarray) else v
            for k, v in r.items()}


def golden_pins(group):
    with open(os.path.join(HERE, "golden", "pins_ref.json")) as fh:
        return json.load(fh)["groups"][group]


def _run(r):
    return {k: r[k] for k in ("status", "msg", "niter", "nfev", "trace", "x", "grad")}


def pin_cases(group):
    """[(name, run)] of one group of pins, run(oracle) -> the fields compared (for a solve: status, message, counts, trace, x,
    grad).  The inputs come from fixed seeds."""
    cases = []
    if group == "lbfgs":
        rng = np.random.default_rng(1)
        for n in (2, 6, 24, 100, 2002):
            for t in range(6):
                x0 = rng.uniform(-1, 1, n)
                for ls in range(4):
                    cases.append(("rosenbrock_n%d_t%d_ls%d" % (n, t, ls), lambda o, x0=x0, ls=ls, m=3 + t % 8: _run(
                        o.lbfgs(po.OBJ_ROSENBROCK_PAIRED, x0, ls, o.default_param(max_linesearch=256, m=m)))))
        d, b, _ = po.quad_tridiag_data(3000)
        for ls in range(4):
            cases.append(("quad_tridiag_n3000_ls%d" % ls, lambda o, ls=ls: _run(
                o.lbfgs(po.OBJ_QUAD_TRIDIAG, np.zeros(3000), ls, o.default_param(m=20), data0=d, data1=b))))
    elif group == "lbfgs_f32":
        for ls in range(4):
            cases.append(("rosenbrock_n10_f32_ls%d" % ls, lambda o, ls=ls: _run(
                o.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(10), ls, o.default_param(), dtype=np.float32))))
    elif group == "apply_Hv":
        rng = np.random.default_rng(3)
        n, m = 1000, 5
        for npairs in (0, 1, 4, 5, 6, 13):
            S = rng.standard_normal((npairs, n))
            Y = S + 0.1 * rng.standard_normal((npairs, n))
            v = rng.standard_normal(n)

            def run(o, S=S, Y=Y, v=v):
                res, _, theta = o.apply_Hv(S, Y, v, -1.0, m)
                return {"res": res, "theta": float(theta).hex()}
            cases.append(("hv_n%d_m%d_p%d" % (n, m, npairs), run))
    elif group == "lbfgsb":
        # mixed finite / infinite / degenerate (l == u) bounds, history sizes 1..10, 0..10 BOXCQP sweeps, delta-based stopping
        rng = np.random.default_rng(3)
        for obj in (po.OBJ_ROSENBROCK_CHAINED, po.OBJ_ROSENBROCK_PAIRED, po.OBJ_QUAD_SHIFT, po.OBJ_QUAD_TRIDIAG):
            for n in (2, 4, 10, 25, 26, 100):
                if obj == po.OBJ_ROSENBROCK_PAIRED and n % 2:
                    continue
                for trial in range(6):
                    lo = rng.uniform(-2, 1, n)
                    hi = lo + rng.uniform(0, 3, n)
                    if trial == 0:
                        lo[:], hi[:] = 2.0, 4.0
                    elif trial == 1:
                        lo[:], hi[:] = -np.inf, np.inf
                    elif trial == 2:
                        hi[::3] = lo[::3]
                    elif trial == 3:
                        lo[::2], hi[1::3] = -np.inf, np.inf
                    x0 = rng.uniform(-3, 5, n)
                    d0, d1 = po.quad_tridiag_data(n, seed=trial)[:2] if obj == po.OBJ_QUAD_TRIDIAG else (None, None)
                    kw = dict(m=int(rng.choice([1, 2, 3, 6, 10])), max_iterations=int(rng.choice([0, 5, 50])),
                              max_submin=int(rng.choice([0, 1, 10])), past=int(rng.choice([0, 0, 2])))
                    if kw["past"]:
                        kw["delta"] = 1e-8
                    cases.append(("obj%d_n%d_t%d" % (obj, n, trial), lambda o, a=(obj, x0, lo, hi), kw=kw, d=(d0, d1): _run(
                        o.lbfgsb(*a, o.default_param(lbfgsb=True, **kw), data0=d[0], data1=d[1]))))
    elif group == "lbfgsb_larger":
        for n, obj in ((2000, po.OBJ_ROSENBROCK_CHAINED), (5000, po.OBJ_ROSENBROCK_PAIRED)):
            cases.append(("obj%d_n%d" % (obj, n), lambda o, n=n, obj=obj: _run(
                o.lbfgsb(obj, np.full(n, 3.0), 2.0, 4.0, o.default_param(lbfgsb=True)))))
    else:
        raise KeyError(group)
    return cases


PIN_GROUPS = ("lbfgs", "lbfgs_f32", "apply_Hv", "lbfgsb", "lbfgsb_larger")
