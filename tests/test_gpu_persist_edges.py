"""The device-resident solve (k_persist, lbfgspp_b200/csrc/persist.cuh) at the edges of its tiling: ragged tails (odd n, n not a
multiple of 4 in fp32), the ends of history blocks, trial tiles and per-CTA chunks, neighbour-coupled objectives across tiles and
CTAs, the single-stage staged pass, history sizes where the block length or the dots-pass rounds change, and batches with data.

Four families of checks, every case generated from a mirror of the solver's geometry (persist_geometry.h) rather than hand-listed:
  (a) local invariants: the returned gradient is the objective's gradient at the returned x, fx and gnorm are its value and norm;
  (b) the S/Y ring, bit for bit, against iterates of shorter runs of the same (bitwise repeatable) solve;
  (c) the first iterations against the CPU checker and the host-driven loop (fp64);
  (d) batches through the C ABI: every member bit-identical to the same problem solved alone.
A halo slip at a chunk or tile boundary or an unmasked tail lane gives an O(1) error at one index, which (a) and (b) see directly."""
import ctypes as C

import numpy as np
import pytest

import lbfgspp_b200 as lb
import pyoracle as po
from test_gpu_solver import check_parity, cpu_param
from util import LS

pytestmark = pytest.mark.gpu

PAIRED, SHIFT, CHAINED, TRIDIAG = lb.OBJ_ROSENBROCK_PAIRED, lb.OBJ_QUAD_SHIFT, lb.OBJ_ROSENBROCK_CHAINED, lb.OBJ_QUAD_TRIDIAG
OBJ_NAMES = {PAIRED: "paired", SHIFT: "shift", CHAINED: "chained", TRIDIAG: "tridiag"}
LS_NAMES = ["Backtracking", "Bracketing", "NocedalWright", "MoreThuente"]
MS = [1, 4, 5, 10, 22, 24, 25, 46, 49, 64]

# ---- mirror of lbfgspp_b200/csrc/persist_geometry.h (checked against the header by test_persist_geometry_cpu.py) ----------------
STAGE_BYTES, MAX_STAGES, TRIAL_TE = 196608, 4, 2016   # kPStageBytes, kPMaxStages, kTrialTE


def block_len(m, elem, want_stages=2):
    """persist_block_len: the largest power of two in [32, 1024] for which `want_stages` stages of 2m+4 rows fit the staging ring
    (the host calls it with want_stages = 2 unless LBFGS_B200_STAGES is set, persist_host.cuh lbfgs_b200_solver_create_batch)."""
    bt = 1024
    while bt > 32 and want_stages * (2 * m + 4) * bt * elem > STAGE_BYTES:
        bt //= 2
    return bt


def _stages(stage_elems, elem):
    return min(STAGE_BYTES // (stage_elems * elem), MAX_STAGES)   # persist_stages


def stage_counts(m, elem, obj):
    """Stages of each staged pass with a full ring (c = m): dots_stages, combine_stages, trial_halo_stages and their minimum
    (persist_min_stages)."""
    bt = block_len(m, elem)
    halo = obj in (CHAINED, TRIDIAG)
    dv = 2 if obj == TRIDIAG else 0
    pad = 16 // elem
    dots = min(_stages((4 + 2 * (m - 1)) * bt, elem), _stages((1 + 2 * m) * bt, elem))
    fused_full = _stages((2 + (dv if halo else 0) + 2 * m) * bt + (2 * pad if halo else 0), elem)
    combine = min(fused_full, _stages((1 + 2 * m) * bt, elem))
    trial = min(_stages((nin + dv) * (TRIAL_TE + 2 * pad), elem) for nin in (1, 2)) if halo else MAX_STAGES
    return dict(bt=bt, dots=dots, fused_full=fused_full, trial=trial, least=min(dots, combine, trial))


def _sm_count():
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.get_device_properties(0).multi_processor_count
    except Exception:
        pass
    return 148   # a B200's SM count: only names the cases where no device is visible (they are deselected there)


SM = _sm_count()


def sizes(m, elem):
    """The lengths at which the tiling of one (dtype, m) changes: tiny vectors, one history block +-1, one trial tile +-1, one block
    per CTA then one CTA with two, and one vector above 2^20 with a ragged last 16-byte unit (n = 1 mod 32 fp64, 3 mod 32 fp32)."""
    bt = block_len(m, elem)
    big = (1 << 20) + (1 if elem == 8 else 3)
    return [("n1", 1), ("n2", 2), ("n3", 3), ("bt-1", bt - 1), ("bt", bt), ("bt+1", bt + 1), ("te-1", TRIAL_TE - 1),
            ("te+1", TRIAL_TE + 1), ("sm*bt-1", SM * bt - 1), ("sm*bt", SM * bt), ("sm*bt+1", SM * bt + 1), ("big", big)]


def allowed(obj, n):
    if obj == PAIRED:
        return n % 2 == 0          # pairs of coordinates
    if obj == CHAINED:
        return n >= 2              # the reference's functor reads x[1]
    return True


def make_cases():
    """Every (dtype, objective, size kind) once; m walks through MS so that the product m x sizes is sampled, not enumerated."""
    out = []
    i = 0
    for dt in (np.float64, np.float32):
        elem = np.dtype(dt).itemsize
        for obj in (PAIRED, SHIFT, CHAINED, TRIDIAG):
            for j in range(12):
                m = MS[(3 * j + obj + (5 if elem == 4 else 0)) % len(MS)]
                kind, n = sizes(m, elem)[j]
                if not allowed(obj, n):
                    n, kind = n + 1, kind + "+1"
                out.append(dict(dt=dt, obj=obj, n=n, m=m, kind=kind, ls=LS_NAMES[i % 4], seed=i))
                i += 1
    # the single-stage fused pass (a full ring of the tridiagonal quadratic at m where two stages fill the ring exactly) at a length
    # that spans several CTAs and tiles
    for dt in (np.float64, np.float32):
        elem = np.dtype(dt).itemsize
        for m in MS:
            if stage_counts(m, elem, TRIDIAG)["fused_full"] == 1:
                n = 3 * block_len(m, elem) * SM + 5
                out.append(dict(dt=dt, obj=TRIDIAG, n=n, m=m, kind="1stage", ls=LS_NAMES[i % 4], seed=i))
                i += 1
    return out


CASES = make_cases()
RING_CASES = [c for c in CASES if c["obj"] != SHIFT and c["n"] >= 4]   # the shifted quadratic converges in 2 iterations
# (the shifted quadratic's value near its optimum at large n is a sum of squares of x_i - i with x_i ~ i ~ 1e6: a last-bit change of
# the step moves it by more than the parity bar on fx, so its long vectors are left to the invariants above)
PREFIX_CASES = [c for c in CASES if c["dt"] == np.float64 and not (c["obj"] == SHIFT and c["n"] > 4096)]


def case_id(c):
    return "%s-%s-m%d-%s-n%d" % ("f64" if c["dt"] == np.float64 else "f32", OBJ_NAMES[c["obj"]], c["m"], c["kind"], c["n"])


def iters_for(c):
    return c["m"] + 3     # > m + 1: the ring fills and wraps, and the full-ring passes (single-stage included) run


# ---- problems and a float64 evaluation of the objectives with the magnitude of their terms -----------------------------------------
def problem(obj, n, dt, seed, kappa=1e3):
    rng = np.random.default_rng(seed)
    if obj == TRIDIAG:
        d, b, _ = po.quad_tridiag_data(n, kappa=kappa, seed=seed)
        return rng.uniform(-1, 1, n).astype(dt), d.astype(dt), b.astype(dt)
    if obj == SHIFT:
        return rng.uniform(-1, 1, n).astype(dt), None, None
    return rng.uniform(-1.2, 1.2, n).astype(dt), None, None


def optimum(obj, n, dt, d, b):
    if obj in (PAIRED, CHAINED):
        return np.ones(n, dt)
    if obj == SHIFT:
        return np.arange(n, dtype=dt)
    from scipy.linalg import solve_banded
    d64, b64 = d.astype(np.float64), b.astype(np.float64)
    ab = np.zeros((3, n))
    ab[0, 1:] = -0.5
    ab[1] = d64 + 1.0
    ab[2, :-1] = -0.5
    return solve_banded((1, 1), ab, b64).astype(dt)


def evaluate(obj, x, d=None, b=None):
    """f, grad and, per element, bounds on the magnitude of the terms that make up f and grad (float64).  A kernel that evaluates the
    same expressions in precision eps makes an error of a few eps times these magnitudes in each element."""
    x = x.astype(np.float64)
    n = x.size
    xl = np.concatenate(([0.0], x[:-1]))      # x_{i-1}, 0 outside the vector (the device's convention)
    xr = np.concatenate((x[1:], [0.0]))       # x_{i+1}
    if obj == PAIRED:
        x0, x1 = x[0::2], x[1::2]
        t1, t2 = 1.0 - x0, 10.0 * (x1 - x0 * x0)
        g = np.empty(n)
        g[1::2] = 20.0 * t2
        g[0::2] = -2.0 * (x0 * g[1::2] + t1)
        m2 = 200.0 * (np.abs(x1) + x0 * x0)
        gm = np.empty(n)
        gm[1::2] = m2
        gm[0::2] = 2.0 * (np.abs(x0) * m2 + 1.0 + np.abs(x0))
        fterms = t1 * t1 + t2 * t2
        fmag = fterms + 2 * np.abs(t1) * (1 + np.abs(x0)) + 2 * np.abs(t2) * 10.0 * (np.abs(x1) + x0 * x0)
    elif obj == SHIFT:
        i = np.arange(n, dtype=np.float64)
        r = x - i
        g = 2.0 * r
        gm = 2.0 * (np.abs(x) + i)
        fterms = r * r
        fmag = fterms + 2 * np.abs(r) * (np.abs(x) + i)
    elif obj == CHAINED:
        u = x - xl * xl
        v = 16.0 * (x * x - xr) * x
        vm = 16.0 * (x * x + np.abs(xr)) * np.abs(x)
        g = 8.0 * u + v
        gm = 8.0 * (np.abs(x) + xl * xl) + vm
        g[-1], gm[-1] = 8.0 * u[-1], 8.0 * (abs(x[-1]) + xl[-1] ** 2)
        g[0] = 2.0 * (x[0] - 1.0) + v[0]
        gm[0] = 2.0 * (abs(x[0]) + 1.0) + vm[0]
        fterms = 4.0 * u * u
        fmag = fterms + 8.0 * np.abs(u) * (np.abs(x) + xl * xl)
        fterms[0] = (x[0] - 1.0) ** 2
        fmag[0] = fterms[0] + 2 * abs(x[0] - 1.0) * (abs(x[0]) + 1.0)
    else:
        d64, b64 = d.astype(np.float64), b.astype(np.float64)
        ax = (d64 + 1.0) * x - 0.5 * (xl + xr)
        axm = (d64 + 1.0) * np.abs(x) + 0.5 * (np.abs(xl) + np.abs(xr))
        g = ax - b64
        gm = axm + np.abs(b64)
        fterms = x * (0.5 * ax - b64)
        fmag = np.abs(x) * (0.5 * axm + np.abs(b64))
    return float(np.sum(fterms)), g, gm, float(np.sum(fmag))


# ---- C ABI of the device-resident solver (include/lbfgs_b200.h) -------------------------------------------------------------------
class Param(C.Structure):       # lbfgs_b200_param
    _fields_ = [("m", C.c_int), ("epsilon", C.c_double), ("epsilon_rel", C.c_double), ("past", C.c_int), ("delta", C.c_double),
                ("max_iterations", C.c_int), ("linesearch", C.c_int), ("max_linesearch", C.c_int), ("min_step", C.c_double),
                ("max_step", C.c_double), ("ftol", C.c_double), ("wolfe", C.c_double)]


class Outcome(C.Structure):     # lbfgs_b200_outcome
    _fields_ = [("status", C.c_int), ("niter", C.c_int), ("nfev", C.c_longlong), ("fx", C.c_double), ("gnorm", C.c_double),
                ("rounds", C.c_longlong)]


def abi_param(m, max_iterations=0):
    p = lb.LBFGSParam(m=m, max_iterations=max_iterations)
    return Param(p.m, p.epsilon, p.epsilon_rel, p.past, p.delta, p.max_iterations, p.linesearch, p.max_linesearch, p.min_step,
                 p.max_step, p.ftol, p.wolfe)


def _suffix(dt):
    return "f64" if np.dtype(dt) == np.float64 else "f32"


def padded(rows, n, ld, dt):
    """Rows laid out `ld` apart (ld = 0: one shared row) in a buffer that keeps the padded-tail contract of lbfgs_b200.h: room for
    (B - 1) * ld + n rounded up to a whole 256-byte line."""
    unit = 256 // np.dtype(dt).itemsize
    B = len(rows)
    buf = np.zeros((B - 1) * ld + -(-n // unit) * unit, dt)
    for b, r in enumerate(rows if ld else rows[:1]):
        buf[b * ld:b * ld + n] = r
    return buf


class Solver:
    """lbfgs_b200_solver_create_batch / _minimize{,_batch}_{f64,f32} / _history / _final_grad through ctypes."""

    def __init__(self, ctx, n, m, dt, B=1):
        self.ctx, self.lib, self.n, self.m, self.dt, self.B = ctx, ctx.lib, n, m, np.dtype(dt), B
        self.h = C.c_void_p()
        ctx.check(self.lib.lbfgs_b200_solver_create_batch(ctx.h, n, m, self.dt.itemsize, B, C.byref(self.h)))

    def close(self):
        if self.h:
            self.lib.lbfgs_b200_solver_destroy(self.h)
            self.h = C.c_void_p()

    def minimize(self, obj, X, p0, p1, ldd, prm, ls, lone=False):
        """X: (B, n) start points (host).  p0, p1: device addresses of the data vectors or None.  Returns (status, [Outcome], X out)."""
        B, n = X.shape
        xd = lb.DeviceArray(self.ctx, X.reshape(-1).astype(self.dt))
        outs = (Outcome * B)()
        if lone:
            fn = getattr(self.lib, "lbfgs_b200_solver_minimize_" + _suffix(self.dt))
            st = fn(self.h, obj, p0, p1, C.addressof(prm), ls, xd.ptr, None, 0, C.addressof(outs))
        else:
            fn = getattr(self.lib, "lbfgs_b200_solver_minimize_batch_" + _suffix(self.dt))
            st = fn(self.h, obj, p0, p1, ldd, C.addressof(prm), ls, xd.ptr, n, C.addressof(outs))
        return st, list(outs), xd.get().reshape(B, n)

    def _d2h(self, dptr, n):
        out = np.empty(n, self.dt)
        self.ctx.check(self.lib.lbfgs_b200_memcpy_d2h(self.ctx.h, out.ctypes.data_as(C.c_void_p), dptr, out.nbytes))
        return out

    def final_grad(self):
        self.lib.lbfgs_b200_solver_final_grad.restype = C.c_void_p
        return self._d2h(C.c_void_p(self.lib.lbfgs_b200_solver_final_grad(self.h)), self.n)

    def history(self):
        """The ring of the last solve by age (newest first): ncorr, S, Y, theta, ys."""
        h = C.c_void_p(self.lib.lbfgs_b200_solver_history(self.h))
        assert h.value, self.lib.lbfgs_b200_last_error(self.ctx.h).decode()
        ncorr = self.lib.lbfgs_b200_hist_ncorr(h)
        S = [self._d2h(C.c_void_p(self.lib.lbfgs_b200_hist_s_col(h, a)), self.n) for a in range(ncorr)]
        Y = [self._d2h(C.c_void_p(self.lib.lbfgs_b200_hist_y_col(h, a)), self.n) for a in range(ncorr)]
        ct = C.c_double if self.dt == np.float64 else C.c_float
        theta, ys, al = (ct * 1)(), (ct * (self.m + 1))(), (ct * (self.m + 1))()
        self.ctx.check(getattr(self.lib, "lbfgs_b200_hist_scalars_" + _suffix(self.dt))(h, theta, ys, al))
        return ncorr, S, Y, float(theta[0]), np.array(ys[:ncorr], dtype=np.float64)


@pytest.fixture(scope="module")
def ctx():
    c = lb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", autouse=True)
def report_case_counts(request):
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    if tr is not None:
        tr.write_line("persist edges: %d invariant cases, %d ring cases, %d prefix-parity cases, %d batch cases (SM count %d)"
                      % (len(CASES), len(RING_CASES), len(PREFIX_CASES), len(BATCH_CASES), SM))
    yield


# ---- (a) local invariants -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_gradient_value_and_norm_at_the_returned_point(ctx, orc, case):
    dt, obj, n, m = case["dt"], case["obj"], case["n"], case["m"]
    eps = float(np.finfo(dt).eps)
    x0, d, b = problem(obj, n, dt, case["seed"])
    d0 = lb.DeviceArray(ctx, padded([d], n, 0, dt)) if d is not None else None
    d1 = lb.DeviceArray(ctx, padded([b], n, 0, dt)) if b is not None else None
    s = Solver(ctx, n, m, dt)
    try:
        before = ctx.launches()
        st, outs, X = s.minimize(obj, x0[None, :], d0.ptr if d0 else None, d1.ptr if d1 else None, 0, abi_param(m, iters_for(case)),
                                 LS[case["ls"]], lone=True)
        ctx.check(st)
        assert ctx.launches() - before == 1
        r = dict(status=outs[0].status, fx=outs[0].fx, gnorm=outs[0].gnorm, x=X[0], grad=s.final_grad())
    finally:
        s.close()
    f, g, gm, fmag = evaluate(obj, r["x"], d, b)
    if dt == np.float64:
        if n >= 2 or obj != CHAINED:
            fo, go = orc.objective(obj, r["x"], d, b)   # the float64 mirror above against the CPU checker's functors
            assert np.max(np.abs(go - g)) <= 1e-12 * (np.max(np.abs(g)) + 1) and abs(fo - f) <= 64 * eps * fmag
        tol = 1e-12 * (np.max(np.abs(g)) + 1)
    else:
        # fp32: each gradient element is a handful (<= 6) of fp32 roundings of terms bounded by gm (the same expressions as the
        # kernel's, see evaluate), so it lies within 6 eps gm of the exact value; 8 eps gm leaves room and still sits ~1e-6 relative
        # to the element's own terms, far below the O(1) error of a wrong neighbour or an unmasked lane
        tol = 8 * eps * gm
    err = np.abs(r["grad"].astype(np.float64) - g)
    assert np.all(err <= tol), (int(np.argmax(err - tol)), float(np.max(err - tol)))
    if r["status"] != 0:
        # a line search can exhaust fp32 resolution (e.g. the tridiagonal quadratic's gradient cannot reach 1e-5 |x| when its
        # rounding is eps * kappa |x|); the pair (x, g) it leaves must still agree, fx and gnorm belong to the last accepted point
        assert dt == np.float32, r["status"]
        return
    # fx and gnorm are reductions of what the kernel evaluated: 64 eps of the summed term magnitudes
    assert abs(r["fx"] - f) <= 64 * eps * fmag, (r["fx"], f, 64 * eps * fmag)
    gg = r["grad"].astype(np.float64)
    gnorm = float(np.sqrt(np.sum(gg * gg)))
    assert abs(r["gnorm"] - gnorm) <= 64 * eps * gnorm + 1e-300, (r["gnorm"], gnorm)


# ---- (b) the ring, exactly ------------------------------------------------------------------------------------------------------------
def ring_run(ctx, case, x0, p0, p1, K):
    s = Solver(ctx, case["n"], case["m"], case["dt"])
    try:
        st, outs, X = s.minimize(case["obj"], x0[None, :], p0, p1, 0, abi_param(case["m"], K), LS[case["ls"]], lone=True)
        ctx.check(st)
        return dict(out=outs[0], x=X[0], g=s.final_grad(), hist=s.history())
    finally:
        s.close()


@pytest.mark.parametrize("case", RING_CASES, ids=case_id)
def test_history_ring_holds_the_exact_pairs(ctx, case):
    """Run A stops after K iterations (N = its niter), runs B and C after N-1 and N-2.  The reference never adds the last iteration's
    pair (LBFGS.h returns before add_correction), so A's newest column is x_{N-1} - x_{N-2} = x_B - x_C and likewise for y, bit for
    bit (s = x - xp and y = g - gp are single roundings in the working precision).  Every older column of A is the column one age
    younger of B: the ring wrapped in the right place.  With Wolfe-condition line searches every pair passes the curvature gate, so
    add_correction (reference LBFGS.h:116-170, BFGSMat.h) leaves ncorr = min(N - 1, m)."""
    dt, obj, n, m = case["dt"], case["obj"], case["n"], case["m"]
    eps = float(np.finfo(dt).eps)
    x0, d, b = problem(obj, n, dt, case["seed"])
    d0 = lb.DeviceArray(ctx, padded([d], n, 0, dt)) if d is not None else None
    d1 = lb.DeviceArray(ctx, padded([b], n, 0, dt)) if b is not None else None
    p0, p1 = (d0.ptr, d1.ptr) if d is not None else (None, None)
    A = ring_run(ctx, case, x0, p0, p1, iters_for(case))
    N = A["out"].niter
    assert A["out"].status == 0 and N >= 3, (A["out"].status, N)
    Bq = ring_run(ctx, case, x0, p0, p1, N - 1)
    Cq = ring_run(ctx, case, x0, p0, p1, N - 2)
    assert (Bq["out"].niter, Cq["out"].niter) == (N - 1, N - 2)
    ncorr, S, Y, theta, ys = A["hist"]
    assert ncorr == min(N - 1, m)
    s_new, y_new = Bq["x"] - Cq["x"], Bq["g"] - Cq["g"]
    assert s_new.dtype == dt
    for got, want, what in ((S[0], s_new, "s"), (Y[0], y_new, "y")):
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, (what, int(bad[0]), float(got[bad[0]]), float(want[bad[0]]))
    ncB, SB, YB = Bq["hist"][:3]
    assert ncB == min(N - 2, m)
    for age in range(1, ncorr):
        assert np.array_equal(S[age], SB[age - 1]) and np.array_equal(Y[age], YB[age - 1]), age
    s64, y64 = s_new.astype(np.float64), y_new.astype(np.float64)
    sy, yy = float(s64 @ y64), float(y64 @ y64)
    assert sy > eps * yy
    tol_sy = 64 * eps * float(np.abs(s64) @ np.abs(y64))
    assert abs(ys[0] - sy) <= tol_sy, (ys[0], sy, tol_sy)
    assert abs(theta - yy / sy) <= (64 * eps + tol_sy / sy) * (yy / sy) * 1.01, (theta, yy / sy)


# ---- (c) prefix parity (fp64) ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", PREFIX_CASES, ids=case_id)
def test_first_iterations_match_cpu_checker_and_host_loop(orc, case):
    obj, n, m = case["obj"], case["n"], case["m"]
    x0, d, b = problem(obj, n, np.float64, case["seed"])
    prm = lb.LBFGSParam(m=m, max_iterations=min(iters_for(case), 15))
    g = lb.LBFGSSolver(prm, case["ls"], resident=True).minimize(obj, x0, data0=d, data1=b)
    c = orc.lbfgs(obj, x0, LS[case["ls"]], cpu_param(orc, prm), data0=d, data1=b, sum_mode=po.SUM_LANES8)
    check_parity(g, c, xtol=1e-6)
    h = lb.LBFGSSolver(prm, case["ls"], resident=False).minimize(obj, x0, data0=d, data1=b)
    assert h["status"] == g["status"] and (h["niter"], h["nfev"]) == (g["niter"], g["nfev"])
    assert abs(h["fx"] - g["fx"]) <= 1e-10 * max(1.0, abs(g["fx"]))


# ---- (d) batches ------------------------------------------------------------------------------------------------------------------------
def make_batch_cases():
    out = []
    i = 0
    for dt in (np.float64, np.float32):
        elem = np.dtype(dt).itemsize
        for obj in (PAIRED, SHIFT, CHAINED, TRIDIAG):
            for B in (1, 3, 7):
                m = MS[(2 * i + 1) % len(MS)]
                bt = block_len(m, elem)
                n = [bt + 1, TRIAL_TE + 1, 2 * bt * 3 + 7][i % 3]          # odd lengths ...
                if obj == PAIRED or i % 2:
                    n += 1                                                 # ... and even ones
                for ldd in ((0, "own") if obj == TRIDIAG else (0,)):
                    out.append(dict(dt=dt, obj=obj, B=B, n=n, m=m, ldd=ldd, ls=LS_NAMES[i % 4], seed=500 + i))
                i += 1
    return out


BATCH_CASES = make_batch_cases()


def batch_id(c):
    return "%s-%s-B%d-m%d-n%d%s" % ("f64" if c["dt"] == np.float64 else "f32", OBJ_NAMES[c["obj"]], c["B"], c["m"], c["n"],
                                    "" if c["obj"] != TRIDIAG else ("-shared" if c["ldd"] == 0 else "-ldd"))


@pytest.mark.parametrize("case", BATCH_CASES, ids=batch_id)
def test_batch_members_equal_lone_solves(ctx, case):
    dt, obj, B, n, m = case["dt"], case["obj"], case["B"], case["n"], case["m"]
    elem = np.dtype(dt).itemsize
    rows = [problem(obj, n, dt, case["seed"] + b, kappa=10.0) for b in range(B)]
    X0 = np.stack([r[0] for r in rows])
    if obj == TRIDIAG:
        ldd = 0 if case["ldd"] == 0 else -(-(n + 3) // (16 // elem)) * (16 // elem)    # >= n, a whole number of 16-byte units
        D, Bv = [r[1] for r in rows], [r[2] for r in rows]
        d0, d1 = lb.DeviceArray(ctx, padded(D, n, ldd, dt)), lb.DeviceArray(ctx, padded(Bv, n, ldd, dt))
        if ldd == 0:
            D, Bv = [D[0]] * B, [Bv[0]] * B
    else:
        ldd, d0, d1, D, Bv = 0, None, None, [None] * B, [None] * B
    if B > 1:
        X0[B // 2] = optimum(obj, n, dt, D[B // 2], Bv[B // 2])      # one member starts at its optimum
    prm = abi_param(m, m + 3)
    ls = LS[case["ls"]]
    s = Solver(ctx, n, m, dt, B)
    try:
        st, outs, X = s.minimize(obj, X0, d0.ptr if d0 else None, d1.ptr if d1 else None, ldd, prm, ls)
        ctx.check(st)
    finally:
        s.close()
    if B > 1:
        assert (outs[B // 2].niter, outs[B // 2].nfev) == (1, 1)
    for b in range(B):
        lone = Solver(ctx, n, m, dt)
        try:
            row = lambda a: None if a is None else C.c_void_p(a.ptr.value + b * ldd * elem)   # problem b's data inside the batch's
            st, o, Xl = lone.minimize(obj, X0[b:b + 1], row(d0), row(d1), 0, prm, ls, lone=True)
            ctx.check(st)
        finally:
            lone.close()
        got, want = outs[b], o[0]
        assert (got.status, got.niter, got.nfev, got.fx, got.gnorm) == (want.status, want.niter, want.nfev, want.fx, want.gnorm), b
        assert np.array_equal(X[b], Xl[0]), b


def test_batch_data_arguments_are_validated(ctx):
    """A misaligned data pointer or a batch stride that is not a whole number of 16-byte units (or shorter than n) is refused with
    LBFGS_B200_ERR_INVALID and a message before anything is launched."""
    for dt in (np.float64, np.float32):
        elem = np.dtype(dt).itemsize
        n, B, m = 1001, 3, 6
        unit = 16 // elem
        good = -(-n // unit) * unit
        _, d, b = problem(TRIDIAG, n, dt, 1)
        d0 = lb.DeviceArray(ctx, padded([d] * B, n, good, dt))
        d1 = lb.DeviceArray(ctx, padded([b] * B, n, good, dt))
        X0 = np.zeros((B, n), dt)
        s = Solver(ctx, n, m, dt, B)
        fn = getattr(ctx.lib, "lbfgs_b200_solver_minimize_batch_" + _suffix(dt))
        xd = lb.DeviceArray(ctx, X0.reshape(-1))
        outs = (Outcome * B)()
        prm = abi_param(m, 3)
        shifted = lambda a: C.c_void_p(a.ptr.value + elem)
        try:
            for p0, p1, ldd in ((shifted(d0), d1.ptr, good), (d0.ptr, shifted(d1), good), (d0.ptr, d1.ptr, good + 1),
                                (d0.ptr, d1.ptr, good - unit), (d0.ptr, d1.ptr, -unit)):
                before = ctx.launches()
                st = fn(s.h, TRIDIAG, p0, p1, ldd, C.addressof(prm), 3, xd.ptr, n, C.addressof(outs))
                assert st == 1, (dt, ldd, st)
                msg = ctx.lib.lbfgs_b200_last_error(ctx.h).decode()
                assert "data" in msg, msg
                assert ctx.launches() == before
        finally:
            s.close()
