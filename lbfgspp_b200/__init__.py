"""lbfgspp_b200 -- B200-native L-BFGS hot path behind LBFGSpp's solver interface.

Layers (top to bottom):
  LBFGSParam / LBFGSSolver (this module)   Python mirror of the reference's classes for tests and bench.py;
                                           calls the C++ front through liblbfgs_b200_driver.so
  include/LBFGS.h, include/LBFGSpp/*.h     header-only C++ front = the drop-in (same class names as the reference)
  include/lbfgs_b200.h                     C ABI
  csrc/*.cu                                hand-written sm_100a kernels (liblbfgs_b200.so)

There is no CPU fallback: importing works anywhere, but creating a Context / solving raises unless the CUDA
library is built (lbfgspp_b200.build.build_all()) and a B200 is present.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

PKG = os.path.dirname(os.path.abspath(__file__))

OBJ_ROSENBROCK_PAIRED, OBJ_QUAD_SHIFT, OBJ_ROSENBROCK_CHAINED, OBJ_QUAD_TRIDIAG = 0, 1, 2, 3
HV_AUTO, HV_TWO_LOOP, HV_GRAM, HV_GRAM_UNFUSED = 0, 1, 2, 3
LINE_SEARCHES = {"Backtracking": 0, "Bracketing": 1, "NocedalWright": 2, "MoreThuente": 3}
LBFGS_LINESEARCH_BACKTRACKING_ARMIJO = 1
LBFGS_LINESEARCH_BACKTRACKING = 2
LBFGS_LINESEARCH_BACKTRACKING_WOLFE = 2
LBFGS_LINESEARCH_BACKTRACKING_STRONG_WOLFE = 3


class NativeLibraryMissing(RuntimeError):
    pass


class LbfgsB200Error(RuntimeError):
    def __init__(self, status, message):
        super().__init__("lbfgs_b200 status %d: %s" % (status, message))
        self.status = status


_libs = {}


def _load(name):
    if name not in _libs:
        path = os.path.join(PKG, name)
        if not os.path.exists(path):
            raise NativeLibraryMissing(
                "%s is not built; run `python -m lbfgspp_b200.build` (there is no CPU fallback)" % path)
        _libs[name] = C.CDLL(path)   # RTLD_LOCAL: nothing here may interpose with other loaded libraries
    return _libs[name]


def abi():
    """The raw C ABI (include/lbfgs_b200.h) as a ctypes library with argument types declared."""
    lib = _load("liblbfgs_b200.so")
    if getattr(lib, "_typed", False):
        return lib
    vp, i64, ci, sz = C.c_void_p, C.c_int64, C.c_int, C.c_size_t
    lib.lbfgs_b200_version.restype = C.c_char_p
    lib.lbfgs_b200_last_error.restype = C.c_char_p
    lib.lbfgs_b200_last_error.argtypes = [vp]
    lib.lbfgs_b200_ctx_create.argtypes = [C.POINTER(vp), ci, vp]
    lib.lbfgs_b200_ctx_destroy.argtypes = [vp]
    lib.lbfgs_b200_ctx_destroy.restype = None
    lib.lbfgs_b200_stream.restype = vp
    lib.lbfgs_b200_stream.argtypes = [vp]
    lib.lbfgs_b200_sm_count.argtypes = [vp]
    lib.lbfgs_b200_launch_count.restype = C.c_uint64
    lib.lbfgs_b200_launch_count.argtypes = [vp]
    lib.lbfgs_b200_malloc.argtypes = [vp, C.POINTER(vp), sz]
    lib.lbfgs_b200_free.argtypes = [vp, vp]
    lib.lbfgs_b200_memcpy_h2d.argtypes = [vp, vp, vp, sz]
    lib.lbfgs_b200_memcpy_d2h.argtypes = [vp, vp, vp, sz]
    lib.lbfgs_b200_memcpy_d2d.argtypes = [vp, vp, vp, sz]
    lib.lbfgs_b200_memset_zero.argtypes = [vp, vp, sz]
    lib.lbfgs_b200_sync.argtypes = [vp]
    lib.lbfgs_b200_trim.argtypes = [vp]
    lib.lbfgs_b200_timer_start.argtypes = [vp]
    lib.lbfgs_b200_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    lib.lbfgs_b200_set_index_offset.argtypes = [vp, i64]
    lib.lbfgs_b200_profile_enable.argtypes = [vp, ci]
    lib.lbfgs_b200_profile_read.argtypes = [vp, ci, C.POINTER(C.c_double), C.POINTER(C.c_uint64), ci]
    lib.lbfgs_b200_profile_bytes.argtypes = [vp, ci, C.POINTER(C.c_double), ci]
    lib.lbfgs_b200_comm_unique_id.argtypes = [vp]
    lib.lbfgs_b200_comm_init.argtypes = [vp, vp, ci, ci]
    lib.lbfgs_b200_comm_size.argtypes = [vp]
    lib.lbfgs_b200_hist_create.argtypes = [vp, C.POINTER(vp), i64, ci, ci]
    lib.lbfgs_b200_hist_destroy.argtypes = [vp]
    lib.lbfgs_b200_hist_destroy.restype = None
    lib.lbfgs_b200_hist_reset.argtypes = [vp]
    lib.lbfgs_b200_hist_ncorr.argtypes = [vp]
    lib.lbfgs_b200_hist_m.argtypes = [vp]
    lib.lbfgs_b200_hist_s_col.restype = vp
    lib.lbfgs_b200_hist_s_col.argtypes = [vp, ci]
    lib.lbfgs_b200_hist_y_col.restype = vp
    lib.lbfgs_b200_hist_y_col.argtypes = [vp, ci]
    for suf, ct in (("f64", C.c_double), ("f32", C.c_float)):
        pt = C.POINTER(ct)
        getattr(lib, "lbfgs_b200_dot_" + suf).argtypes = [vp, i64, vp, vp, pt]
        getattr(lib, "lbfgs_b200_dot3_" + suf).argtypes = [vp, i64, vp, vp, vp, pt]
        getattr(lib, "lbfgs_b200_axpy_out_" + suf).argtypes = [vp, i64, vp, ct, vp, vp]
        getattr(lib, "lbfgs_b200_scale_out_" + suf).argtypes = [vp, i64, ct, vp, vp]
        getattr(lib, "lbfgs_b200_objective_" + suf).argtypes = [vp, ci, vp, vp, i64, vp, vp, pt]
        getattr(lib, "lbfgs_b200_trial_" + suf).argtypes = [vp, ci, vp, vp, i64, vp, vp, ct, vp, vp, pt]
        getattr(lib, "lbfgs_b200_hist_update_" + suf).argtypes = [vp, vp, vp, vp, vp, ct, C.POINTER(ci), pt]
        getattr(lib, "lbfgs_b200_hist_add_" + suf).argtypes = [vp, vp, vp]
        getattr(lib, "lbfgs_b200_hist_apply_Hv_" + suf).argtypes = [vp, vp, ct, vp, ci, pt]
        getattr(lib, "lbfgs_b200_hist_update_apply_Hv_" + suf).argtypes = [vp, vp, vp, vp, vp, ct, ct, vp, ci, C.POINTER(ci), pt]
        getattr(lib, "lbfgs_b200_hist_scalars_" + suf).argtypes = [vp, pt, pt, pt]
    # device-resident solve (persistent kernel; single problem or batch)
    lib.lbfgs_b200_solver_create.argtypes = [vp, i64, ci, ci, C.POINTER(vp)]
    lib.lbfgs_b200_solver_create_batch.argtypes = [vp, i64, ci, ci, ci, C.POINTER(vp)]
    lib.lbfgs_b200_solver_destroy.argtypes = [vp]
    lib.lbfgs_b200_solver_destroy.restype = None
    lib.lbfgs_b200_solver_batch.argtypes = [vp]
    lib.lbfgs_b200_solver_profile.argtypes = [vp, vp, vp, vp, vp, vp]
    for name in ("lbfgs_b200_solver_final_grad", "lbfgs_b200_solver_history"):
        getattr(lib, name).restype = vp
        getattr(lib, name).argtypes = [vp]
    for name in ("lbfgs_b200_solver_final_grad_of", "lbfgs_b200_solver_history_of"):
        getattr(lib, name).restype = vp
        getattr(lib, name).argtypes = [vp, ci]
    for suf in ("f64", "f32"):
        getattr(lib, "lbfgs_b200_solver_minimize_" + suf).argtypes = [vp, ci, vp, vp, vp, ci, vp, vp, C.c_longlong, vp]
        getattr(lib, "lbfgs_b200_solver_minimize_batch_" + suf).argtypes = [vp, ci, vp, vp, i64, vp, ci, vp, i64, vp]
    lib._typed = True
    return lib


class _DrvParam(C.Structure):
    _fields_ = [("m", C.c_int), ("epsilon", C.c_double), ("epsilon_rel", C.c_double), ("past", C.c_int),
                ("delta", C.c_double), ("max_iterations", C.c_int), ("linesearch", C.c_int),
                ("max_submin", C.c_int), ("max_linesearch", C.c_int), ("min_step", C.c_double),
                ("max_step", C.c_double), ("ftol", C.c_double), ("wolfe", C.c_double)]


class _BatchItem(C.Structure):
    _fields_ = [("status", C.c_int), ("niter", C.c_int), ("nfev", C.c_long), ("fx", C.c_double), ("gnorm", C.c_double)]


class _DrvResult(C.Structure):
    _fields_ = [("status", C.c_int), ("msg", C.c_char * 200), ("niter", C.c_int), ("nfev", C.c_long),
                ("fx", C.c_double), ("gnorm", C.c_double), ("trace_len", C.c_long), ("seconds", C.c_double),
                ("seconds_e2e", C.c_double), ("launches", C.c_ulonglong), ("h2d_bytes", C.c_long),
                ("d2h_bytes", C.c_long)]


def driver():
    abi()  # the driver links against the kernel library: load it first, globally
    lib = _load("liblbfgs_b200_driver.so")
    if getattr(lib, "_typed", False):
        return lib
    dp, fp = C.POINTER(C.c_double), C.POINTER(C.c_float)
    lib.lbfgsb200_drv_lbfgs_f64.argtypes = [C.c_int, C.c_int, dp, dp, C.c_long, C.c_int, C.POINTER(_DrvParam), C.c_int,
                                            C.c_int, dp, dp, dp, C.c_long, C.POINTER(_DrvResult)]
    lib.lbfgsb200_drv_lbfgs_f32.argtypes = [C.c_int, C.c_int, fp, fp, C.c_long, C.c_int, C.POINTER(_DrvParam), C.c_int,
                                            C.c_int, fp, fp, dp, C.c_long, C.POINTER(_DrvResult)]
    lib.lbfgsb200_drv_ctx.restype = C.c_void_p
    lib.lbfgsb200_drv_ctx.argtypes = [C.c_int]
    lib.lbfgsb200_drv_lbfgsb_f64.argtypes = [C.c_int, C.c_int, dp, dp, C.c_long, C.POINTER(_DrvParam), dp, dp, dp, dp, dp, C.c_long,
                                             C.POINTER(_DrvResult)]
    lib.lbfgsb200_drv_session_create.restype = C.c_void_p
    lib.lbfgsb200_drv_session_create.argtypes = [C.c_int, C.c_int, dp, dp, C.c_long, C.c_int, C.POINTER(_DrvParam), C.c_int, dp,
                                                 C.c_char_p, C.c_int, C.c_int]
    lib.lbfgsb200_drv_session_destroy.argtypes = [C.c_void_p]
    lib.lbfgsb200_drv_session_destroy.restype = None
    lib.lbfgsb200_drv_session_solve.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(_DrvResult)]
    lib.lbfgsb200_drv_session_result.restype = dp
    lib.lbfgsb200_drv_session_result.argtypes = [C.c_void_p]
    lib.lbfgsb200_drv_batch_session_create.restype = C.c_void_p
    lib.lbfgsb200_drv_batch_session_create.argtypes = [C.c_int, C.c_int, C.c_long, C.c_int, dp, C.c_int, C.POINTER(_DrvParam), C.c_char_p, C.c_int]
    lib.lbfgsb200_drv_batch_session_destroy.argtypes = [C.c_void_p]
    lib.lbfgsb200_drv_batch_session_destroy.restype = None
    lib.lbfgsb200_drv_batch_session_solve.argtypes = [C.c_void_p, C.POINTER(_BatchItem), C.POINTER(C.c_long), dp, dp, C.c_char_p, C.c_int]
    lib.lbfgsb200_drv_comm_init.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_char_p, C.c_int]
    lib.lbfgsb200_drv_p2p_export.argtypes = [C.c_int, C.c_void_p, C.c_char_p, C.c_int]
    lib.lbfgsb200_drv_p2p_attach.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_char_p, C.c_int]
    lib._typed = True
    return lib


# ------------------------------------------------------------------------------------------------------
# Python mirror of the reference's classes
# ------------------------------------------------------------------------------------------------------
class LBFGSParam:
    """Same fields and defaults as LBFGSpp::LBFGSParam<Scalar> (reference Param.h:171-182)."""

    def __init__(self, **kw):
        self.m = 6
        self.epsilon = 1e-5
        self.epsilon_rel = 1e-5
        self.past = 0
        self.delta = 0.0
        self.max_iterations = 0
        self.linesearch = LBFGS_LINESEARCH_BACKTRACKING_STRONG_WOLFE
        self.max_linesearch = 20
        self.min_step = 1e-20
        self.max_step = 1e20
        self.ftol = 1e-4
        self.wolfe = 0.9
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError("LBFGSParam has no field %r" % k)
            setattr(self, k, v)

    def _c(self):
        return _DrvParam(self.m, self.epsilon, self.epsilon_rel, self.past, self.delta, self.max_iterations,
                         self.linesearch, 10, self.max_linesearch, self.min_step, self.max_step, self.ftol, self.wolfe)


class LBFGSBParam:
    """Same fields and defaults as LBFGSpp::LBFGSBParam<Scalar> (reference Param.h:330-341)."""

    def __init__(self, **kw):
        self.m = 6
        self.epsilon = 1e-5
        self.epsilon_rel = 1e-5
        self.past = 1
        self.delta = 1e-10
        self.max_iterations = 0
        self.max_submin = 10
        self.max_linesearch = 20
        self.min_step = 1e-20
        self.max_step = 1e20
        self.ftol = 1e-4
        self.wolfe = 0.9
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError("LBFGSBParam has no field %r" % k)
            setattr(self, k, v)

    def _c(self):
        return _DrvParam(self.m, self.epsilon, self.epsilon_rel, self.past, self.delta, self.max_iterations, 3, self.max_submin,
                         self.max_linesearch, self.min_step, self.max_step, self.ftol, self.wolfe)


_EXC = {1: ValueError, 2: ArithmeticError, 3: RuntimeError, 4: RuntimeError}
STATUS_NAMES = {0: "ok", 1: "invalid_argument", 2: "logic_error", 3: "runtime_error", 4: "other"}


class LBFGSSolver:
    """LBFGSpp::LBFGSSolver<Scalar, LineSearch> on the GPU, host buffers in and out.

    minimize(objective, x0) returns a dict(niter, nfev, fx, gnorm, x, grad, trace, status, msg, seconds, ...);
    with raise_errors=True the reference's exceptions come back as ValueError (std::invalid_argument),
    ArithmeticError (std::logic_error) or RuntimeError (std::runtime_error).
    """

    def __init__(self, param=None, linesearch="NocedalWright", dtype=np.float64, device=0, hv_algo=HV_AUTO,
                 fused=True, resident=False):
        self.param = param if param is not None else LBFGSParam()
        self.ls = LINE_SEARCHES[linesearch] if isinstance(linesearch, str) else int(linesearch)
        self.dtype = np.dtype(dtype)
        self.device = device
        self.hv_algo = hv_algo
        self.fused = 2 if resident else fused   # 2: device-resident solve (one persistent kernel launch per minimize)

    def minimize(self, objective, x0, data0=None, data1=None, trace_cap=100000, raise_errors=False, want_grad=True):
        drv = driver()
        dt = self.dtype
        ct = C.c_double if dt == np.float64 else C.c_float
        x = np.array(x0, dtype=dt, order="C").copy()
        n = x.size
        grad = np.zeros(n, dtype=dt) if want_grad else None
        trace = np.zeros(trace_cap, dtype=np.float64)
        d0 = None if data0 is None else np.ascontiguousarray(data0, dtype=dt)
        d1 = None if data1 is None else np.ascontiguousarray(data1, dtype=dt)
        ptr = lambda a, t=ct: a.ctypes.data_as(C.POINTER(t)) if a is not None else None
        res = _DrvResult()
        p = self.param._c()
        fn = drv.lbfgsb200_drv_lbfgs_f64 if dt == np.float64 else drv.lbfgsb200_drv_lbfgs_f32
        fn(self.device, objective, ptr(d0), ptr(d1), n, self.ls, C.byref(p), self.hv_algo, int(self.fused), ptr(x),
           ptr(grad), ptr(trace, C.c_double), trace_cap, C.byref(res))
        if res.status and raise_errors:
            raise _EXC.get(res.status, RuntimeError)(res.msg.decode())
        return dict(status=STATUS_NAMES[res.status], msg=res.msg.decode(), niter=res.niter, nfev=res.nfev, fx=res.fx,
                    gnorm=res.gnorm, x=x, grad=grad, trace=trace[:res.trace_len].copy(), seconds=res.seconds,
                    seconds_e2e=res.seconds_e2e, launches=res.launches, h2d_bytes=res.h2d_bytes,
                    d2h_bytes=res.d2h_bytes)


class LBFGSBSolver:
    """LBFGSpp::LBFGSBSolver<double> (More-Thuente line search) on the GPU, host buffers in and out."""

    def __init__(self, param=None, device=0):
        self.param = param if param is not None else LBFGSBParam()
        self.device = device

    def minimize(self, objective, x0, lb, ub, data0=None, data1=None, trace_cap=100000, raise_errors=False):
        drv = driver()
        x = np.array(x0, dtype=np.float64, order="C").copy()
        n = x.size
        lbv = np.ascontiguousarray(np.broadcast_to(lb, n), dtype=np.float64)
        ubv = np.ascontiguousarray(np.broadcast_to(ub, n), dtype=np.float64)
        grad = np.zeros(n)
        trace = np.zeros(trace_cap)
        d0 = None if data0 is None else np.ascontiguousarray(data0, dtype=np.float64)
        d1 = None if data1 is None else np.ascontiguousarray(data1, dtype=np.float64)
        dp = C.POINTER(C.c_double)
        ptr = lambda a: a.ctypes.data_as(dp) if a is not None else None
        res = _DrvResult()
        p = self.param._c()
        drv.lbfgsb200_drv_lbfgsb_f64(self.device, objective, ptr(d0), ptr(d1), n, C.byref(p), ptr(x), ptr(lbv), ptr(ubv),
                                     ptr(grad), ptr(trace), trace_cap, C.byref(res))
        if res.status and raise_errors:
            raise _EXC.get(res.status, RuntimeError)(res.msg.decode())
        return dict(status=STATUS_NAMES[res.status], msg=res.msg.decode(), niter=res.niter, nfev=res.nfev, fx=res.fx,
                    gnorm=res.gnorm, x=x, grad=grad, trace=trace[:res.trace_len].copy(), seconds=res.seconds,
                    seconds_e2e=res.seconds_e2e, launches=res.launches)


# ------------------------------------------------------------------------------------------------------
# thin object wrappers over the raw C ABI (kernel-level tests, microbenchmarks)
# ------------------------------------------------------------------------------------------------------
class Context:
    def __init__(self, device=0, stream=None):
        self.lib = abi()
        self.h = C.c_void_p()
        st = self.lib.lbfgs_b200_ctx_create(C.byref(self.h), device, stream)
        if st:
            raise LbfgsB200Error(st, self.lib.lbfgs_b200_last_error(None).decode())

    @classmethod
    def borrow(cls, handle):
        """Non-owning wrapper around an existing lbfgs_b200_ctx* (e.g. driver_ctx(device), which may carry a communicator)."""
        self = cls.__new__(cls)
        self.lib = abi()
        self.h = handle if isinstance(handle, C.c_void_p) else C.c_void_p(handle)
        self.owned = False
        return self

    def check(self, st):
        if st:
            raise LbfgsB200Error(st, self.lib.lbfgs_b200_last_error(self.h).decode())

    def close(self):
        if self.h and getattr(self, "owned", True):
            self.lib.lbfgs_b200_ctx_destroy(self.h)
        self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def array(self, host, dtype=None):
        return DeviceArray(self, host, dtype)

    def empty(self, n, dtype=np.float64):
        return DeviceArray(self, None, dtype, n)

    def sync(self):
        self.check(self.lib.lbfgs_b200_sync(self.h))

    def trim(self):
        """Give the context's cached device blocks back to the driver (lbfgs_b200_trim)."""
        self.check(self.lib.lbfgs_b200_trim(self.h))

    def launches(self):
        return self.lib.lbfgs_b200_launch_count(self.h)

    def timer_start(self):
        self.check(self.lib.lbfgs_b200_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float(0)
        self.check(self.lib.lbfgs_b200_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def _fn(self, name, dtype):
        return getattr(self.lib, "lbfgs_b200_%s_%s" % (name, "f64" if np.dtype(dtype) == np.float64 else "f32"))

    def dot(self, a, b):
        out = (a.ct * 1)()
        self.check(self._fn("dot", a.dtype)(self.h, a.n, a.ptr, b.ptr, out))
        return out[0]

    def dot3(self, g, d, x):
        out = (g.ct * 3)()
        self.check(self._fn("dot3", g.dtype)(self.h, g.n, g.ptr, d.ptr, x.ptr, out))
        return list(out)

    def axpy_out(self, a, s, b, out):
        self.check(self._fn("axpy_out", a.dtype)(self.h, a.n, a.ptr, s, b.ptr, out.ptr))

    def scale_out(self, s, a, out):
        self.check(self._fn("scale_out", a.dtype)(self.h, a.n, s, a.ptr, out.ptr))

    def objective(self, kind, x, g, data0=None, data1=None):
        out = (x.ct * 4)()
        self.check(self._fn("objective", x.dtype)(self.h, kind, data0.ptr if data0 else None,
                                                  data1.ptr if data1 else None, x.n, x.ptr, g.ptr, out))
        return list(out)

    def trial(self, kind, xp, d, step, x, g, data0=None, data1=None):
        out = (x.ct * 4)()
        self.check(self._fn("trial", x.dtype)(self.h, kind, data0.ptr if data0 else None, data1.ptr if data1 else None,
                                              xp.n, xp.ptr, d.ptr, step, x.ptr, g.ptr, out))
        return list(out)


class DeviceArray:
    def __init__(self, ctx, host=None, dtype=None, n=None, offset_elems=0):
        self.ctx = ctx
        if host is not None:
            host = np.ascontiguousarray(host, dtype=dtype)
            n = host.size
            dtype = host.dtype
        self.dtype = np.dtype(dtype)
        self.ct = C.c_double if self.dtype == np.float64 else C.c_float
        self.n = int(n)
        self.base = C.c_void_p()
        self.offset = offset_elems * self.dtype.itemsize
        ctx.check(ctx.lib.lbfgs_b200_malloc(ctx.h, C.byref(self.base), self.n * self.dtype.itemsize + self.offset))
        self.ptr = C.c_void_p(self.base.value + self.offset)
        if host is not None:
            ctx.check(ctx.lib.lbfgs_b200_memcpy_h2d(ctx.h, self.ptr, host.ctypes.data_as(C.c_void_p), host.nbytes))
            ctx.sync()

    def get(self):
        out = np.empty(self.n, dtype=self.dtype)
        self.ctx.check(self.ctx.lib.lbfgs_b200_memcpy_d2h(self.ctx.h, out.ctypes.data_as(C.c_void_p), self.ptr, out.nbytes))
        return out

    def __del__(self):
        try:
            if self.base and self.ctx.h:
                self.ctx.lib.lbfgs_b200_free(self.ctx.h, self.base)
        except Exception:
            pass


class History:
    """The S/Y ring (BFGSMat) through the C ABI."""

    def __init__(self, ctx, n, m, dtype=np.float64):
        self.ctx, self.n, self.m, self.dtype = ctx, n, m, np.dtype(dtype)
        self.suf = "f64" if self.dtype == np.float64 else "f32"
        self.ct = C.c_double if self.dtype == np.float64 else C.c_float
        self.h = C.c_void_p()
        ctx.check(ctx.lib.lbfgs_b200_hist_create(ctx.h, C.byref(self.h), n, m, self.dtype.itemsize))

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.ctx.lib.lbfgs_b200_hist_destroy(self.h)
        except Exception:
            pass

    def reset(self):
        self.ctx.check(self.ctx.lib.lbfgs_b200_hist_reset(self.h))

    @property
    def ncorr(self):
        return self.ctx.lib.lbfgs_b200_hist_ncorr(self.h)

    def add(self, s, y):
        self.ctx.check(getattr(self.ctx.lib, "lbfgs_b200_hist_add_" + self.suf)(self.h, s.ptr, y.ptr))

    def update(self, x, xp, g, gp, eps=None):
        eps = np.finfo(self.dtype).eps if eps is None else eps
        acc = C.c_int(0)
        sy = (self.ct * 2)()
        self.ctx.check(getattr(self.ctx.lib, "lbfgs_b200_hist_update_" + self.suf)(self.h, x.ptr, xp.ptr, g.ptr, gp.ptr,
                                                                                  eps, C.byref(acc), sy))
        return bool(acc.value), sy[0], sy[1]

    def update_apply_Hv(self, x, xp, g, gp, a, res, algo=HV_AUTO, eps=None):
        """hist_update(x, xp, g, gp) + apply_Hv(g, a, res) as one call (pair formed inside the dots pass); -> (accepted, g.res)"""
        eps = np.finfo(self.dtype).eps if eps is None else eps
        acc = C.c_int(0)
        out = (self.ct * 1)()
        self.ctx.check(getattr(self.ctx.lib, "lbfgs_b200_hist_update_apply_Hv_" + self.suf)(
            self.h, x.ptr, xp.ptr, g.ptr, gp.ptr, eps, a, res.ptr, algo, C.byref(acc), out))
        return bool(acc.value), out[0]

    def apply_Hv(self, v, a, res, algo=HV_AUTO, want_dot=False):
        out = (self.ct * 1)()
        self.ctx.check(getattr(self.ctx.lib, "lbfgs_b200_hist_apply_Hv_" + self.suf)(
            self.h, v.ptr, a, res.ptr, algo, out if want_dot else None))
        return out[0] if want_dot else None

    def scalars(self):
        theta = (self.ct * 1)()
        ys = (self.ct * (self.m + 1))()
        al = (self.ct * (self.m + 1))()
        self.ctx.check(getattr(self.ctx.lib, "lbfgs_b200_hist_scalars_" + self.suf)(self.h, theta, ys, al))
        c = self.ncorr
        return theta[0], np.array(ys[:c]), np.array(al[:c])

    def column(self, which, age):
        fn = self.ctx.lib.lbfgs_b200_hist_s_col if which == "s" else self.ctx.lib.lbfgs_b200_hist_y_col
        p = fn(self.h, age)
        out = np.empty(self.n, dtype=self.dtype)
        self.ctx.check(self.ctx.lib.lbfgs_b200_memcpy_d2h(self.ctx.h, out.ctypes.data_as(C.c_void_p), p, out.nbytes))
        return out


class Session:
    """A solver and its vectors kept resident on one GPU (bench.py): solve() repeats the same problem."""

    def __init__(self, objective, x0, param, linesearch="MoreThuente", device=0, hv_algo=HV_AUTO, data0=None, data1=None,
                 resident=True):
        self.drv = driver()
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        self.n = x0.size
        dp = C.POINTER(C.c_double)
        ptr = lambda a: a.ctypes.data_as(dp) if a is not None else None
        d0 = None if data0 is None else np.ascontiguousarray(data0, dtype=np.float64)
        d1 = None if data1 is None else np.ascontiguousarray(data1, dtype=np.float64)
        err = C.create_string_buffer(256)
        p = param._c()
        ls = LINE_SEARCHES[linesearch] if isinstance(linesearch, str) else int(linesearch)
        self.h = self.drv.lbfgsb200_drv_session_create(device, objective, ptr(d0), ptr(d1), self.n, ls, C.byref(p), hv_algo,
                                                       ptr(x0), err, 256, int(resident))
        if not self.h:
            raise RuntimeError("session_create failed: " + err.value.decode())

    def solve(self, from_host=False, to_host=False):
        res = _DrvResult()
        self.drv.lbfgsb200_drv_session_solve(self.h, int(from_host), int(to_host), C.byref(res))
        if res.status:
            raise RuntimeError(res.msg.decode())
        return dict(niter=res.niter, nfev=res.nfev, fx=res.fx, gnorm=res.gnorm, launches=res.launches,
                    h2d_bytes=res.h2d_bytes, d2h_bytes=res.d2h_bytes)

    OPS = ("mixed", "first", "trial", "dots_form", "dots_plain", "combine", "combine_trial", "restore", "materialize", "-")

    def profile(self):
        """Accounting of the last device-resident solve: dict(kernel_ms, sync_ms, ops={name: dict(ms, rounds, alg_bytes)}); None for
        the host-driven loop."""
        ms, rounds, nbytes = (C.c_double * 10)(), (C.c_ulonglong * 10)(), (C.c_double * 10)()
        kms, sync = C.c_double(0), (C.c_double * 3)()
        self.drv.lbfgsb200_drv_session_profile.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        if self.drv.lbfgsb200_drv_session_profile(self.h, C.byref(kms), ms, rounds, nbytes, sync):
            return None
        return dict(kernel_ms=kms.value, sync_ms=sync[0], wait_last_cta_ms=sync[1], exchange_ms=sync[2],
                    ops={self.OPS[k]: dict(ms=ms[k], rounds=int(rounds[k]), alg_bytes=nbytes[k]) for k in range(10) if rounds[k]})

    def result(self):
        p = self.drv.lbfgsb200_drv_session_result(self.h)
        return np.ctypeslib.as_array(p, shape=(self.n,)).copy()

    def download(self):
        """x as the last solve() left it on the device (also when that solve did not copy it to the host)."""
        x = np.empty(self.n)
        err = C.create_string_buffer(256)
        self.drv.lbfgsb200_drv_session_download.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_char_p, C.c_int]
        if self.drv.lbfgsb200_drv_session_download(self.h, x.ctypes.data_as(C.POINTER(C.c_double)), err, 256):
            raise RuntimeError("session download failed: " + err.value.decode())
        return x

    def close(self):
        if self.h:
            self.drv.lbfgsb200_drv_session_destroy(self.h)
            self.h = None


def solve_batch(objective, X0, param=None, linesearch="MoreThuente", device=0, hv_algo=HV_AUTO, threads=4, sharded=False,
                return_x=True):
    """B independent problems (rows of X0) on one GPU: LBFGSSolver::minimize per problem, `threads` host threads each with
    its own context/stream.  sharded=True: run on the driver's communicator-attached context (n-sharded over ranks), one
    thread.  Returns (list of dicts, X, seconds)."""
    drv = driver()
    X0 = np.ascontiguousarray(X0, dtype=np.float64)
    B, n = X0.shape
    param = param if param is not None else LBFGSParam()
    items = (_BatchItem * B)()
    X = np.empty_like(X0) if return_x else None
    secs = C.c_double(0)
    dp = C.POINTER(C.c_double)
    drv.lbfgsb200_drv_batch_f64.argtypes = [C.c_int, C.c_int, C.c_long, C.c_int, dp, C.c_int, C.POINTER(_DrvParam), C.c_int, C.c_int,
                                            C.c_int, C.POINTER(_BatchItem), dp, dp]
    p = param._c()
    ls = LINE_SEARCHES[linesearch] if isinstance(linesearch, str) else int(linesearch)
    drv.lbfgsb200_drv_batch_f64(device, objective, n, B, X0.ctypes.data_as(dp), ls, C.byref(p), hv_algo, threads, int(sharded), items,
                                X.ctypes.data_as(dp) if return_x else None, C.byref(secs))
    res = [dict(status=STATUS_NAMES[it.status], niter=it.niter, nfev=it.nfev, fx=it.fx, gnorm=it.gnorm) for it in items]
    return res, X, secs.value


class BatchSession:
    """B independent problems (rows of X0) minimised by ONE persistent kernel launch per solve() (LBFGSpp::LBFGSBatchSolver,
    include/LBFGSBatch.h).  The start points stay resident; with a communicator attached to the device's driver context the rows
    are this rank's blocks of n-sharded problems."""

    def __init__(self, objective, X0, param=None, linesearch="MoreThuente", device=0):
        self.drv = driver()
        X0 = np.ascontiguousarray(X0, dtype=np.float64)
        self.B, self.n = X0.shape
        param = param if param is not None else LBFGSParam()
        p = param._c()
        ls = LINE_SEARCHES[linesearch] if isinstance(linesearch, str) else int(linesearch)
        err = C.create_string_buffer(256)
        self.h = self.drv.lbfgsb200_drv_batch_session_create(device, objective, self.n, self.B, X0.ctypes.data_as(C.POINTER(C.c_double)), ls,
                                                             C.byref(p), err, 256)
        if not self.h:
            raise RuntimeError("batch_session_create failed: " + err.value.decode())

    def solve(self, return_x=True):
        items = (_BatchItem * self.B)()
        rounds = (C.c_long * self.B)()
        X = np.empty((self.B, self.n)) if return_x else None
        secs = C.c_double(0)
        err = C.create_string_buffer(256)
        bad = self.drv.lbfgsb200_drv_batch_session_solve(self.h, items, rounds, X.ctypes.data_as(C.POINTER(C.c_double)) if return_x else None,
                                                         C.byref(secs), err, 256)
        if bad < 0:
            raise RuntimeError("batch solve failed: " + err.value.decode())
        res = [dict(status=STATUS_NAMES[it.status], niter=it.niter, nfev=it.nfev, fx=it.fx, gnorm=it.gnorm, rounds=int(r))
               for it, r in zip(items, rounds)]
        return res, X, secs.value

    def upload(self, X0):
        """New start points (host array, B x n) for the following solves: the host -> device leg of the end-to-end path."""
        X0 = np.ascontiguousarray(X0, dtype=np.float64)
        assert X0.shape == (self.B, self.n)
        err = C.create_string_buffer(256)
        self.drv.lbfgsb200_drv_batch_session_upload.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_char_p, C.c_int]
        if self.drv.lbfgsb200_drv_batch_session_upload(self.h, X0.ctypes.data_as(C.POINTER(C.c_double)), err, 256):
            raise RuntimeError("batch upload failed: " + err.value.decode())
        return X0.nbytes

    def profile(self):
        """Accounting of the last batched solve (one kernel launch for the whole batch): same dict as Session.profile()."""
        ms, rounds, nbytes = (C.c_double * 10)(), (C.c_ulonglong * 10)(), (C.c_double * 10)()
        kms, sync = C.c_double(0), (C.c_double * 3)()
        self.drv.lbfgsb200_drv_batch_session_profile.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        if self.drv.lbfgsb200_drv_batch_session_profile(self.h, C.byref(kms), ms, rounds, nbytes, sync):
            return None
        return dict(kernel_ms=kms.value, sync_ms=sync[0], wait_last_cta_ms=sync[1], exchange_ms=sync[2],
                    ops={Session.OPS[k]: dict(ms=ms[k], rounds=int(rounds[k]), alg_bytes=nbytes[k]) for k in range(10) if rounds[k]})

    def close(self):
        if self.h:
            self.drv.lbfgsb200_drv_batch_session_destroy(self.h)
            self.h = None


def solve_dense(objective, x0, param=None, linesearch="NocedalWright", resident=True, device=0):
    """minimize() then final_approx_hessian() / final_approx_inverse_hessian() (small n).  Returns (niter, x, B, H)."""
    drv = driver()
    x = np.array(x0, dtype=np.float64, order="C").copy()
    n = x.size
    param = param if param is not None else LBFGSParam()
    p = param._c()
    ls = LINE_SEARCHES[linesearch] if isinstance(linesearch, str) else int(linesearch)
    Bm, Hm = np.zeros((n, n)), np.zeros((n, n))
    niter = C.c_int(0)
    err = C.create_string_buffer(256)
    dp = C.POINTER(C.c_double)
    drv.lbfgsb200_drv_solve_dense_f64.argtypes = [C.c_int, C.c_int, C.c_long, C.c_int, C.POINTER(_DrvParam), C.c_int, dp, dp, dp,
                                                  C.POINTER(C.c_int), C.c_char_p, C.c_int]
    if drv.lbfgsb200_drv_solve_dense_f64(device, objective, n, ls, C.byref(p), int(resident), x.ctypes.data_as(dp), Bm.ctypes.data_as(dp),
                                         Hm.ctypes.data_as(dp), C.byref(niter), err, 256):
        raise RuntimeError("solve_dense failed: " + err.value.decode())
    return niter.value, x, Bm, Hm


def phase_clock(on=True):
    """Enable / disable (and clear) the wall-clock accounting of the host-driven L-BFGS-B loop's phases (LBFGSpp/PhaseClock.h)."""
    driver().lbfgsb200_drv_phase_enable(int(on))


def phase_report():
    import json
    buf = C.create_string_buffer(8192)
    driver().lbfgsb200_drv_phase_report(buf, 8192)
    return json.loads(buf.value.decode() or "{}")


def driver_ctx(device=0):
    """The lbfgs_b200_ctx* the driver uses for `device` (so that the raw ABI / profiling can address it)."""
    return C.c_void_p(driver().lbfgsb200_drv_ctx(device))


def comm_init(device, unique_id_bytes, rank, nranks, index_offset=0):
    """Attach an NCCL communicator to the driver's context of `device`: n is sharded over `nranks` GPUs."""
    err = C.create_string_buffer(256)
    buf = C.create_string_buffer(bytes(unique_id_bytes), 128)
    st = driver().lbfgsb200_drv_comm_init(device, buf, rank, nranks, index_offset, err, 256)
    if st:
        raise RuntimeError("comm_init failed: " + err.value.decode())


def p2p_export(device):
    """64-byte cudaIpc handle of this rank's inbox for the in-kernel NVLink all-reduce."""
    err = C.create_string_buffer(256)
    buf = C.create_string_buffer(64)
    if driver().lbfgsb200_drv_p2p_export(device, buf, err, 256):
        raise RuntimeError("p2p_export failed: " + err.value.decode())
    return buf.raw


def p2p_attach(device, all_handles, rank, nranks, index_offset=0):
    """all_handles: the nranks 64-byte handles concatenated in rank order."""
    err = C.create_string_buffer(256)
    buf = C.create_string_buffer(bytes(all_handles), 64 * nranks)
    if driver().lbfgsb200_drv_p2p_attach(device, buf, rank, nranks, index_offset, err, 256):
        raise RuntimeError("p2p_attach failed: " + err.value.decode())


def set_global_extent(device, index_offset, n_global):
    """Declare this rank's block of the global vector (needed by the chained-Rosenbrock / tridiagonal objectives when sharded:
    they exchange one boundary coordinate per side with the neighbouring ranks before every evaluation)."""
    err = C.create_string_buffer(256)
    if driver().lbfgsb200_drv_set_global_extent(device, C.c_longlong(index_offset), C.c_longlong(n_global), err, 256):
        raise RuntimeError("set_global_extent failed: " + err.value.decode())


def comm_unique_id():
    buf = C.create_string_buffer(128)
    st = abi().lbfgs_b200_comm_unique_id(buf)
    if st:
        raise RuntimeError("ncclGetUniqueId failed")
    return buf.raw


def build_all(force=False):
    return _build.build_all(force)
