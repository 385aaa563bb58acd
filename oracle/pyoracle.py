"""ctypes bindings for the two CPU checkers (TEST INFRASTRUCTURE ONLY).

  Oracle("orc")  -> oracle/liboracle.so            plain-C++ restatement (travels to the GPU box)
  Oracle("ref")  -> oracle/_ref/libref_lbfgspp.so  unmodified reference headers over minieigen
                                                    (built only in the container that has /root/reference)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module; nothing under lbfgspp_b200/ or include/ does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

OBJ_ROSENBROCK_PAIRED, OBJ_QUAD_SHIFT, OBJ_ROSENBROCK_CHAINED, OBJ_QUAD_TRIDIAG = 0, 1, 2, 3
LS_BACKTRACKING, LS_BRACKETING, LS_NOCEDAL_WRIGHT, LS_MORE_THUENTE = 0, 1, 2, 3
SUM_SEQUENTIAL, SUM_LANES8, SUM_LANES8_OMP = 0, 1, 2
STATUS_NAMES = {0: "ok", 1: "invalid_argument", 2: "logic_error", 3: "runtime_error", 4: "other"}


class Param(C.Structure):
    _fields_ = [("m", C.c_int), ("epsilon", C.c_double), ("epsilon_rel", C.c_double), ("past", C.c_int),
                ("delta", C.c_double), ("max_iterations", C.c_int), ("linesearch", C.c_int),
                ("max_submin", C.c_int), ("max_linesearch", C.c_int), ("min_step", C.c_double),
                ("max_step", C.c_double), ("ftol", C.c_double), ("wolfe", C.c_double)]


class Result(C.Structure):
    _fields_ = [("status", C.c_int), ("msg", C.c_char * 200), ("niter", C.c_int), ("nfev", C.c_long),
                ("fx", C.c_double), ("gnorm", C.c_double), ("trace_len", C.c_long), ("seconds", C.c_double)]


def build():
    """(Re)build the checkers with oracle/Makefile.  Building the checker is not using it."""
    subprocess.run(["make", "-s", "-C", HERE, "all"], check=True)


def build_native(outdir):
    """The timing build of the restatement (`make native`: -O3 -march=native for the host it runs on) into outdir, so that a
    read-only tree works; returns its path for Oracle("orc", path=...)."""
    path = os.path.join(outdir, "liboracle_native.so")
    subprocess.run(["make", "-s", "-C", HERE, "native", "NATIVE_LIB=" + path], check=True)
    return path


def _ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype)) if a is not None else None


class Oracle:
    def __init__(self, which="orc", path=None):
        assert which in ("orc", "ref")
        self.prefix = which + "_"
        if path is None:
            path = os.path.join(HERE, "_ref", "libref_lbfgspp.so") if which == "ref" else os.path.join(HERE, "liboracle.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.path = path
        self.lib = C.CDLL(path)
        dp, fp = C.POINTER(C.c_double), C.POINTER(C.c_float)
        f = self._fn
        f("default_param", None, [C.POINTER(Param), C.c_int])
        f("lbfgs_f64", C.c_int, [C.c_int, dp, dp, C.c_long, C.c_int, C.POINTER(Param), C.c_int, dp, dp, dp,
                                  C.c_long, C.POINTER(Result)])
        f("lbfgs_f32", C.c_int, [C.c_int, fp, fp, C.c_long, C.c_int, C.POINTER(Param), C.c_int, fp, fp, dp,
                                  C.c_long, C.POINTER(Result)])
        f("lbfgsb_f64", C.c_int, [C.c_int, dp, dp, C.c_long, C.POINTER(Param), C.c_int, dp, dp, dp, dp, dp,
                                   C.c_long, C.POINTER(Result)])
        f("bfgs_apply_Hv_f64", C.c_int, [C.c_long, C.c_int, C.c_int, dp, dp, dp, C.c_double, C.c_int, dp, dp, dp])
        f("objective_f64", C.c_double, [C.c_int, dp, dp, C.c_long, dp, dp])
        if which == "orc":
            self.lib.orc_lbfgs_gram_f64.restype = C.c_int
            self.lib.orc_lbfgs_gram_f64.argtypes = self.lib.orc_lbfgs_f64.argtypes
            self.lib.orc_bfgs_apply_Hv_bench_f64.restype = C.c_double
            self.lib.orc_bfgs_apply_Hv_bench_f64.argtypes = [C.c_long, C.c_int, C.c_int, C.c_int, C.c_int]
            self.lib.orc_hw_threads.restype = C.c_int

    def _fn(self, name, restype, argtypes):
        fn = getattr(self.lib, self.prefix + name)
        fn.restype, fn.argtypes = restype, argtypes
        setattr(self, "_" + name, fn)

    # ---- parameters -------------------------------------------------------------------------
    def default_param(self, lbfgsb=False, **overrides):
        p = Param()
        self._default_param(C.byref(p), int(lbfgsb))
        for k, v in overrides.items():
            setattr(p, k, v)
        return p

    # ---- solvers ----------------------------------------------------------------------------
    @staticmethod
    def _pack(res, x, grad, trace):
        n = int(res.trace_len)
        return dict(status=STATUS_NAMES[res.status], msg=res.msg.decode(), niter=res.niter, nfev=res.nfev,
                    fx=res.fx, gnorm=res.gnorm, x=x, grad=grad, trace=trace[:n].copy(), seconds=res.seconds)

    def lbfgs(self, objective, x0, ls, param, data0=None, data1=None, sum_mode=SUM_SEQUENTIAL, dtype=np.float64,
              trace_cap=100000, gram=False):
        x = np.array(x0, dtype=dtype, order="C").copy()
        n = x.size
        grad = np.zeros(n, dtype=dtype)
        trace = np.zeros(trace_cap, dtype=np.float64)
        res = Result()
        ct = C.c_double if dtype == np.float64 else C.c_float
        d0 = None if data0 is None else np.ascontiguousarray(data0, dtype=dtype)
        d1 = None if data1 is None else np.ascontiguousarray(data1, dtype=dtype)
        if gram:
            fn = self.lib.orc_lbfgs_gram_f64
        else:
            fn = self._lbfgs_f64 if dtype == np.float64 else self._lbfgs_f32
        fn(objective, _ptr(d0, ct), _ptr(d1, ct), n, ls, C.byref(param), sum_mode, _ptr(x, ct), _ptr(grad, ct),
           _ptr(trace, C.c_double), trace_cap, C.byref(res))
        return self._pack(res, x, grad, trace)

    def lbfgsb(self, objective, x0, lb, ub, param, data0=None, data1=None, sum_mode=SUM_SEQUENTIAL, trace_cap=100000):
        x = np.array(x0, dtype=np.float64).copy()
        n = x.size
        lb = np.ascontiguousarray(np.broadcast_to(lb, n), dtype=np.float64)
        ub = np.ascontiguousarray(np.broadcast_to(ub, n), dtype=np.float64)
        grad = np.zeros(n)
        trace = np.zeros(trace_cap)
        res = Result()
        d0 = None if data0 is None else np.ascontiguousarray(data0, dtype=np.float64)
        d1 = None if data1 is None else np.ascontiguousarray(data1, dtype=np.float64)
        ct = C.c_double
        self._lbfgsb_f64(objective, _ptr(d0, ct), _ptr(d1, ct), n, C.byref(param), sum_mode, _ptr(x, ct),
                         _ptr(lb, ct), _ptr(ub, ct), _ptr(grad, ct), _ptr(trace, ct), trace_cap, C.byref(res))
        return self._pack(res, x, grad, trace)

    # ---- BFGSMat::apply_Hv on an explicit history ----------------------------------------------
    def apply_Hv(self, S, Y, v, a, m, sum_mode=SUM_SEQUENTIAL):
        """S, Y: (npairs, n) arrays; pairs are appended in order with add_correction, ring size m."""
        S = np.ascontiguousarray(S, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        v = np.ascontiguousarray(v, dtype=np.float64)
        npairs = S.shape[0] if S.ndim == 2 else 0
        n = v.size
        res = np.zeros(n)
        ys = np.zeros(m)
        theta = C.c_double(0)
        ct = C.c_double
        self._bfgs_apply_Hv_f64(n, m, npairs, _ptr(S, ct), _ptr(Y, ct), _ptr(v, ct), a, sum_mode, _ptr(res, ct),
                                _ptr(ys, ct), C.byref(theta))
        return res, ys, theta.value

    def objective(self, objective, x, data0=None, data1=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        g = np.zeros_like(x)
        ct = C.c_double
        d0 = None if data0 is None else np.ascontiguousarray(data0, dtype=np.float64)
        d1 = None if data1 is None else np.ascontiguousarray(data1, dtype=np.float64)
        fx = self._objective_f64(objective, _ptr(d0, ct), _ptr(d1, ct), x.size, _ptr(x, ct), _ptr(g, ct))
        return fx, g

    def apply_Hv_bench(self, n, m, reps, sum_mode, threads=0):
        return self.lib.orc_bfgs_apply_Hv_bench_f64(n, m, reps, sum_mode, threads)

    def hw_threads(self):
        return self.lib.orc_hw_threads()


def quad_tridiag_data(n, kappa=1e3, seed=0):
    """SURVEY.md 8d config C3: d_i = exp(U[0, ln kappa]), x* ~ N(0,1), b = A x*."""
    rng = np.random.default_rng(seed)
    d = np.exp(rng.uniform(0.0, np.log(kappa), n))
    xs = rng.standard_normal(n)
    xl = np.concatenate(([0.0], xs[:-1]))
    xr = np.concatenate((xs[1:], [0.0]))
    b = (d + 1.0) * xs - 0.5 * (xl + xr)
    return d, b, xs
