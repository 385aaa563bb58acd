// driver.cpp -- host-buffer entry points over the header-only C++ front (include/LBFGS.h), built into
// lbfgspp_b200/liblbfgs_b200_driver.so.  This is the "reference-facing call with HOST buffers" that tests and
// bench.py drive through ctypes: the caller hands over x0 in host memory, the driver uploads it, runs
// LBFGSpp::LBFGSSolver<Scalar, LineSearch>::minimize() on the GPU and downloads x / grad.  The argument structs
// have the same layout as the CPU checker's (oracle/oracle_api.h) so that a parity test calls both sides with the
// very same objects -- but nothing here includes or links anything from oracle/.
#include <chrono>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>

#include "../../include/LBFGS.h"
#include "../../include/LBFGSB.h"
#include "../../include/LBFGSBatch.h"
#include "../../include/LBFGSpp/DeviceObjectives.h"

using namespace LBFGSpp;

#pragma GCC visibility push(default)
extern "C" {

typedef struct
{
    int m;
    double epsilon, epsilon_rel;
    int past;
    double delta;
    int max_iterations;
    int linesearch;
    int max_submin;
    int max_linesearch;
    double min_step, max_step, ftol, wolfe;
} drv_param;

typedef struct
{
    int status;             // 0 ok, 1 invalid_argument, 2 logic_error, 3 runtime_error, 4 other
    char msg[200];
    int niter;
    long nfev;
    double fx;
    double gnorm;
    long trace_len;
    double seconds;         // minimize() alone, operands already in HBM (host wall clock around a synchronised call)
    double seconds_e2e;     // upload of x0 (+data) + minimize() + download of x
    unsigned long long launches;  // kernels launched by minimize()
    long h2d_bytes, d2h_bytes;
} drv_result;

enum { DRV_LS_BACKTRACKING = 0, DRV_LS_BRACKETING = 1, DRV_LS_NOCEDAL_WRIGHT = 2, DRV_LS_MORE_THUENTE = 3 };

}  // extern "C"

namespace {

std::map<int, std::shared_ptr<Device> >& devices()
{
    static std::map<int, std::shared_ptr<Device> > m;
    return m;
}
Device& device(int ordinal)
{
    std::shared_ptr<Device>& d = devices()[ordinal];
    if (!d) d = std::make_shared<Device>(ordinal);
    return *d;
}

// Records f of every evaluation (the reference offers the functor as its only observation point,
// examples/example-rosenbrock-comparison.cpp:14-41) while forwarding the fused hooks when Base has them.
template <class Base, class Scalar, bool Fused>
struct Traced;

template <class Base, class Scalar>
struct Traced<Base, Scalar, true>
{
    typedef DeviceVector<Scalar> Vector;
    Base& base;
    double* trace;
    long cap, count;
    Traced(Base& b, double* t, long c) : base(b), trace(t), cap(c), count(0) {}
    void note(Scalar fx) { if (trace && count < cap) trace[count] = double(fx); count++; }
    Scalar operator()(const Vector& x, Vector& g) { const Scalar fx = base(x, g); note(fx); return fx; }
    void fused_value(const Vector& x, Vector& g, Scalar* o) { base.fused_value(x, g, o); note(o[0]); }
    void fused_trial(const Vector& xp, const Vector& d, Scalar s, Vector& x, Vector& g, Scalar* o) { base.fused_trial(xp, d, s, x, g, o); note(o[0]); }
};
template <class Base, class Scalar>
struct Traced<Base, Scalar, false>
{
    typedef DeviceVector<Scalar> Vector;
    Base& base;
    double* trace;
    long cap, count;
    Traced(Base& b, double* t, long c) : base(b), trace(t), cap(c), count(0) {}
    Scalar operator()(const Vector& x, Vector& g)
    {
        const Scalar fx = base(x, g);
        if (trace && count < cap) trace[count] = double(fx);
        count++;
        return fx;
    }
};

void set_error(drv_result* out, int code, const char* what)
{
    out->status = code;
    std::strncpy(out->msg, what, sizeof(out->msg) - 1);
    out->msg[sizeof(out->msg) - 1] = 0;
}

template <class Body>
int guarded(drv_result* out, Body body)
{
    std::memset(out, 0, sizeof(*out));
    try { body(); }
    catch (const std::invalid_argument& e) { set_error(out, 1, e.what()); }
    catch (const std::logic_error& e) { set_error(out, 2, e.what()); }
    catch (const std::runtime_error& e) { set_error(out, 3, e.what()); }
    catch (const std::exception& e) { set_error(out, 4, e.what()); }
    return out->status;
}

template <class Scalar>
LBFGSParam<Scalar> to_param(const drv_param* q)
{
    LBFGSParam<Scalar> p;
    p.m = q->m;
    p.epsilon = Scalar(q->epsilon);
    p.epsilon_rel = Scalar(q->epsilon_rel);
    p.past = q->past;
    p.delta = Scalar(q->delta);
    p.max_iterations = q->max_iterations;
    p.linesearch = q->linesearch;
    p.max_linesearch = q->max_linesearch;
    p.min_step = Scalar(q->min_step);
    p.max_step = Scalar(q->max_step);
    p.ftol = Scalar(q->ftol);
    p.wolfe = Scalar(q->wolfe);
    return p;
}

double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

template <class Scalar, template <class> class LS, class Objective, bool Fused>
void solve_with(Device& dev, Objective& obj, const drv_param* q, int hv_algo, long n, Scalar* x_host, Scalar* grad_host,
                double* trace, long cap, drv_result* out, double t_begin, long h2d_extra)
{
    typedef DeviceVector<Scalar> Vector;
    const LBFGSParam<Scalar> prm = to_param<Scalar>(q);
    LBFGSSolver<Scalar, LS> solver(prm);
    solver.set_hv_algorithm(hv_algo);
    Traced<Objective, Scalar, Fused> f(obj, trace, cap);
    Vector x(dev);
    x.copy_from_host(x_host, n);
    Scalar fx = Scalar(0);
    const unsigned long long launches0 = lbfgs_b200_launch_count(dev.ctx());
    const double t0 = now();
    int niter = 0;
    try { niter = solver.minimize(f, x, fx); }
    catch (...)
    {
        out->nfev = f.count;
        out->trace_len = f.count < cap ? f.count : cap;
        x.copy_to_host(x_host);
        throw;
    }
    dev.synchronize();
    const double t1 = now();
    x.copy_to_host(x_host);
    if (grad_host) solver.final_grad().copy_to_host(grad_host);
    const double t2 = now();
    out->niter = niter;
    out->fx = double(fx);
    out->gnorm = double(solver.final_grad_norm());
    out->nfev = f.count;
    out->trace_len = f.count < cap ? f.count : cap;
    out->seconds = t1 - t0;
    out->seconds_e2e = t2 - t_begin;
    out->launches = lbfgs_b200_launch_count(dev.ctx()) - launches0;
    out->h2d_bytes = long(sizeof(Scalar)) * n + h2d_extra;
    out->d2h_bytes = long(sizeof(Scalar)) * n * (grad_host ? 2 : 1);
}

template <class Scalar, class Objective, bool Fused>
void solve_ls(int ls, Device& dev, Objective& obj, const drv_param* q, int hv_algo, long n, Scalar* x_host, Scalar* grad_host,
              double* trace, long cap, drv_result* out, double t_begin, long h2d_extra)
{
    switch (ls)
    {
    case DRV_LS_BACKTRACKING: solve_with<Scalar, LineSearchBacktracking, Objective, Fused>(dev, obj, q, hv_algo, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    case DRV_LS_BRACKETING: solve_with<Scalar, LineSearchBracketing, Objective, Fused>(dev, obj, q, hv_algo, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    case DRV_LS_NOCEDAL_WRIGHT: solve_with<Scalar, LineSearchNocedalWright, Objective, Fused>(dev, obj, q, hv_algo, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    case DRV_LS_MORE_THUENTE: solve_with<Scalar, LineSearchMoreThuente, Objective, Fused>(dev, obj, q, hv_algo, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    default: throw std::invalid_argument("unknown line search id");
    }
}

template <class Scalar, template <class> class LS>
void solve_resident_with(Device& dev, BuiltinObjective<Scalar>& obj, const drv_param* q, long n, Scalar* x_host, Scalar* grad_host,
                         double* trace, long cap, drv_result* out, double t_begin, long h2d_extra)
{
    typedef DeviceVector<Scalar> Vector;
    const LBFGSParam<Scalar> prm = to_param<Scalar>(q);
    LBFGSSolver<Scalar, LS> solver(prm);
    solver.set_device_resident(true);
    solver.set_trace_buffer(trace, cap);
    Vector x(dev);
    x.copy_from_host(x_host, n);
    Scalar fx = Scalar(0);
    const unsigned long long launches0 = lbfgs_b200_launch_count(dev.ctx());
    const double t0 = now();
    int niter = 0;
    try { niter = solver.minimize(obj, x, fx); }
    catch (...)
    {
        out->nfev = solver.num_evaluations();
        out->trace_len = out->nfev < cap ? out->nfev : cap;
        x.copy_to_host(x_host);
        throw;
    }
    dev.synchronize();
    const double t1 = now();
    x.copy_to_host(x_host);
    if (grad_host) solver.final_grad().copy_to_host(grad_host);
    out->niter = niter;
    out->fx = double(fx);
    out->gnorm = double(solver.final_grad_norm());
    out->nfev = solver.num_evaluations();
    out->trace_len = out->nfev < cap ? out->nfev : cap;
    out->seconds = t1 - t0;
    out->seconds_e2e = now() - t_begin;
    out->launches = lbfgs_b200_launch_count(dev.ctx()) - launches0;
    out->h2d_bytes = long(sizeof(Scalar)) * n + h2d_extra;
    out->d2h_bytes = long(sizeof(Scalar)) * n * (grad_host ? 2 : 1);
}

template <class Scalar>
void solve_resident(int ls, Device& dev, BuiltinObjective<Scalar>& obj, const drv_param* q, long n, Scalar* x_host, Scalar* grad_host,
                    double* trace, long cap, drv_result* out, double t_begin, long h2d_extra)
{
    switch (ls)
    {
    case DRV_LS_BACKTRACKING: solve_resident_with<Scalar, LineSearchBacktracking>(dev, obj, q, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    case DRV_LS_BRACKETING: solve_resident_with<Scalar, LineSearchBracketing>(dev, obj, q, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    case DRV_LS_NOCEDAL_WRIGHT: solve_resident_with<Scalar, LineSearchNocedalWright>(dev, obj, q, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    case DRV_LS_MORE_THUENTE: solve_resident_with<Scalar, LineSearchMoreThuente>(dev, obj, q, n, x_host, grad_host, trace, cap, out, t_begin, h2d_extra); break;
    default: throw std::invalid_argument("unknown line search id");
    }
}

template <class Scalar>
int lbfgs_any(int dev_ordinal, int objective, const Scalar* data0_host, const Scalar* data1_host, long n, int ls,
              const drv_param* q, int hv_algo, int fused, Scalar* x_host, Scalar* grad_host, double* trace, long cap,
              drv_result* out)
{
    return guarded(out, [&]() {
        const double t_begin = now();
        Device& dev = device(dev_ordinal);
        DeviceVector<Scalar> d0(dev), d1(dev);
        long extra = 0;
        if (data0_host) { d0.copy_from_host(data0_host, n); extra += long(sizeof(Scalar)) * n; }
        if (data1_host) { d1.copy_from_host(data1_host, n); extra += long(sizeof(Scalar)) * n; }
        if (fused == 2)   // device-resident solve: the objective must stay visible as a built-in (no tracing wrapper)
        {
            BuiltinObjective<Scalar> obj(objective, d0.data(), d1.data());
            solve_resident<Scalar>(ls, dev, obj, q, n, x_host, grad_host, trace, cap, out, t_begin, extra);
        }
        else if (fused)
        {
            BuiltinObjective<Scalar> obj(objective, d0.data(), d1.data());
            solve_ls<Scalar, BuiltinObjective<Scalar>, true>(ls, dev, obj, q, hv_algo, n, x_host, grad_host, trace, cap, out, t_begin, extra);
        }
        else
        {
            PlainObjective<Scalar> obj(objective, d0.data(), d1.data());
            solve_ls<Scalar, PlainObjective<Scalar>, false>(ls, dev, obj, q, hv_algo, n, x_host, grad_host, trace, cap, out, t_begin, extra);
        }
    });
}

}  // namespace

extern "C" {

// LBFGSSolver<double, LS>::minimize with host buffers.  fused = 1: BuiltinObjective (single-kernel trials),
// fused = 0: PlainObjective (what a user-written device functor gets).
int lbfgsb200_drv_lbfgs_f64(int device_ordinal, int objective, const double* data0_host, const double* data1_host, long n,
                            int ls, const drv_param* prm, int hv_algo, int fused, double* x_host, double* grad_host,
                            double* fx_trace, long trace_cap, drv_result* out)
{
    return lbfgs_any<double>(device_ordinal, objective, data0_host, data1_host, n, ls, prm, hv_algo, fused, x_host, grad_host, fx_trace, trace_cap, out);
}
int lbfgsb200_drv_lbfgs_f32(int device_ordinal, int objective, const float* data0_host, const float* data1_host, long n,
                            int ls, const drv_param* prm, int hv_algo, int fused, float* x_host, float* grad_host,
                            double* fx_trace, long trace_cap, drv_result* out)
{
    return lbfgs_any<float>(device_ordinal, objective, data0_host, data1_host, n, ls, prm, hv_algo, fused, x_host, grad_host, fx_trace, trace_cap, out);
}

// The context the driver uses for a device (so that Python can call the raw C ABI on the same stream)
void* lbfgsb200_drv_ctx(int device_ordinal)
{
    try { return device(device_ordinal).ctx(); }
    catch (...) { return nullptr; }
}

void lbfgsb200_drv_shutdown(void) { devices().clear(); }

}  // extern "C"

// ----------------------------------------------------------------------------------------------------------
// Sessions: a solver + its vectors kept alive across solves (what a long-running user of the C++ front does;
// the reference re-allocates everything per minimize() call, LBFGS.h:40-50).  bench.py times these.
// ----------------------------------------------------------------------------------------------------------
namespace {

struct Session
{
    Device* dev;
    long n;
    int ls;
    LBFGSParam<double> prm;
    DeviceVector<double> x0, x, d0, d1;
    BuiltinObjective<double> obj;
    // one solver per line-search policy (only the selected one is used)
    LBFGSSolver<double, LineSearchBacktracking> s_bt;
    LBFGSSolver<double, LineSearchBracketing> s_br;
    LBFGSSolver<double, LineSearchNocedalWright> s_nw;
    LBFGSSolver<double, LineSearchMoreThuente> s_mt;
    double* pinned_in;   // host staging (pinned): x0 for the end-to-end path
    double* pinned_out;  // host staging (pinned): result x
    Session(Device& d, long n_, int ls_, const drv_param* q, int objective) :
        dev(&d), n(n_), ls(ls_), prm(to_param<double>(q)), x0(d), x(d), d0(d), d1(d), obj(objective),
        s_bt(prm), s_br(prm), s_nw(prm), s_mt(prm), pinned_in(nullptr), pinned_out(nullptr) {}
};

}  // namespace

extern "C" {

// x0_host (n) is uploaded once and kept on the device; data0/data1 (n each, optional) likewise.
void* lbfgsb200_drv_session_create(int device_ordinal, int objective, const double* data0_host, const double* data1_host,
                                   long n, int ls, const drv_param* prm, int hv_algo, const double* x0_host, char* err, int errlen,
                                   int resident)
{
    try
    {
        Device& dev = device(device_ordinal);
        std::unique_ptr<Session> s(new Session(dev, n, ls, prm, objective));
        s->x0.copy_from_host(x0_host, n);
        s->x.resize(n);
        if (data0_host) s->d0.copy_from_host(data0_host, n);
        if (data1_host) s->d1.copy_from_host(data1_host, n);
        s->obj = BuiltinObjective<double>(objective, s->d0.data(), s->d1.data());
        void* p = nullptr;
        dev.check(lbfgs_b200_malloc_host(dev.ctx(), &p, sizeof(double) * size_t(n)));
        s->pinned_in = static_cast<double*>(p);
        dev.check(lbfgs_b200_malloc_host(dev.ctx(), &p, sizeof(double) * size_t(n)));
        s->pinned_out = static_cast<double*>(p);
        std::memcpy(s->pinned_in, x0_host, sizeof(double) * size_t(n));
        s->s_bt.set_hv_algorithm(hv_algo);
        s->s_br.set_hv_algorithm(hv_algo);
        s->s_nw.set_hv_algorithm(hv_algo);
        s->s_mt.set_hv_algorithm(hv_algo);
        s->s_bt.set_device_resident(resident != 0);
        s->s_br.set_device_resident(resident != 0);
        s->s_nw.set_device_resident(resident != 0);
        s->s_mt.set_device_resident(resident != 0);
        return s.release();
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return nullptr;
    }
}

void lbfgsb200_drv_session_destroy(void* handle)
{
    Session* s = static_cast<Session*>(handle);
    if (!s) return;
    lbfgs_b200_free_host(s->dev->ctx(), s->pinned_in);
    lbfgs_b200_free_host(s->dev->ctx(), s->pinned_out);
    delete s;
}

// One solve.  from_host = 1: the start point is copied host(pinned) -> device inside the call (end-to-end path);
// from_host = 0: it is copied device -> device from the resident x0.  to_host = 1: the result x is copied back to
// pinned host memory before returning.  No stream synchronisation is added beyond what minimize() itself needs,
// except for the final download.
int lbfgsb200_drv_session_solve(void* handle, int from_host, int to_host, drv_result* out)
{
    Session* s = static_cast<Session*>(handle);
    return guarded(out, [&]() {
        Device& dev = *s->dev;
        const size_t bytes = sizeof(double) * size_t(s->n);
        if (from_host) dev.check(lbfgs_b200_memcpy_h2d(dev.ctx(), s->x.data(), s->pinned_in, bytes));
        else dev.check(lbfgs_b200_memcpy_d2d(dev.ctx(), s->x.data(), s->x0.data(), bytes));
        const unsigned long long launches0 = lbfgs_b200_launch_count(dev.ctx());
        double fx = 0;
        int niter = 0;
        long nfev = 0;
        double gnorm = 0;
        switch (s->ls)
        {
        case DRV_LS_BACKTRACKING: niter = s->s_bt.minimize(s->obj, s->x, fx); nfev = s->s_bt.num_evaluations(); gnorm = s->s_bt.final_grad_norm(); break;
        case DRV_LS_BRACKETING: niter = s->s_br.minimize(s->obj, s->x, fx); nfev = s->s_br.num_evaluations(); gnorm = s->s_br.final_grad_norm(); break;
        case DRV_LS_NOCEDAL_WRIGHT: niter = s->s_nw.minimize(s->obj, s->x, fx); nfev = s->s_nw.num_evaluations(); gnorm = s->s_nw.final_grad_norm(); break;
        default: niter = s->s_mt.minimize(s->obj, s->x, fx); nfev = s->s_mt.num_evaluations(); gnorm = s->s_mt.final_grad_norm(); break;
        }
        if (to_host) dev.check(lbfgs_b200_memcpy_d2h(dev.ctx(), s->pinned_out, s->x.data(), bytes));
        out->niter = niter;
        out->nfev = nfev;
        out->fx = fx;
        out->gnorm = gnorm;
        out->launches = lbfgs_b200_launch_count(dev.ctx()) - launches0;
        out->h2d_bytes = from_host ? long(bytes) : 0;
        out->d2h_bytes = to_host ? long(bytes) : 0;
    });
}

const double* lbfgsb200_drv_session_result(void* handle) { return static_cast<Session*>(handle)->pinned_out; }

// The x the last solve left on the device -> x_host (n doubles), for a solve that ran with to_host = 0; synchronises.
int lbfgsb200_drv_session_download(void* handle, double* x_host, char* err, int errlen)
{
    try
    {
        static_cast<Session*>(handle)->x.copy_to_host(x_host);
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return -1;
    }
}

// accounting of the session's last device-resident solve (lbfgs_b200_solver_profile; sync_ms has 3 slots); returns 1 when the
// session runs the host-driven loop
int lbfgsb200_drv_session_profile(void* handle, double* kernel_ms, double* ms_by_op10, unsigned long long* rounds_by_op10, double* alg_bytes_by_op10,
                                  double* sync_ms)
{
    Session* s = static_cast<Session*>(handle);
    lbfgs_b200_solver* r = nullptr;
    switch (s->ls)
    {
    case DRV_LS_BACKTRACKING: r = s->s_bt.resident_handle(); break;
    case DRV_LS_BRACKETING: r = s->s_br.resident_handle(); break;
    case DRV_LS_NOCEDAL_WRIGHT: r = s->s_nw.resident_handle(); break;
    default: r = s->s_mt.resident_handle(); break;
    }
    if (!r) return 1;
    return lbfgs_b200_solver_profile(r, kernel_ms, ms_by_op10, rounds_by_op10, alg_bytes_by_op10, sync_ms) == LBFGS_B200_OK ? 0 : 2;
}

}  // extern "C"

extern "C" int lbfgsb200_drv_comm_init(int device_ordinal, const void* unique_id_128, int rank, int nranks, long long index_offset,
                                       char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        dev.check(lbfgs_b200_comm_init(dev.ctx(), unique_id_128, rank, nranks));
        dev.check(lbfgs_b200_set_index_offset(dev.ctx(), index_offset));
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}

extern "C" int lbfgsb200_drv_p2p_export(int device_ordinal, void* handle64, char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        dev.check(lbfgs_b200_comm_p2p_export(dev.ctx(), handle64));
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}

extern "C" int lbfgsb200_drv_p2p_attach(int device_ordinal, const void* handles, int rank, int nranks, long long index_offset,
                                        char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        dev.check(lbfgs_b200_comm_p2p_attach(dev.ctx(), handles, rank, nranks));
        dev.check(lbfgs_b200_set_index_offset(dev.ctx(), index_offset));
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}

// n-sharding: declare this rank's block [index_offset, index_offset + n_local) of a global vector of n_global coordinates
// (needed by the neighbour-coupled built-in objectives, which exchange halos; see lbfgs_b200_set_global_extent)
extern "C" int lbfgsb200_drv_set_global_extent(int device_ordinal, long long index_offset, long long n_global, char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        dev.check(lbfgs_b200_set_global_extent(dev.ctx(), index_offset, n_global));
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}


// LBFGSBSolver<double>::minimize with host buffers (More-Thuente line search, built-in objective, fused trials)
extern "C" int lbfgsb200_drv_lbfgsb_f64(int device_ordinal, int objective, const double* data0_host, const double* data1_host, long n,
                                        const drv_param* q, double* x_host, const double* lb_host, const double* ub_host,
                                        double* grad_host, double* fx_trace, long trace_cap, drv_result* out)
{
    return guarded(out, [&]() {
        const double t_begin = now();
        Device& dev = device(device_ordinal);
        typedef DeviceVector<double> Vector;
        Vector d0(dev), d1(dev), x(dev), lb(dev), ub(dev);
        if (data0_host) d0.copy_from_host(data0_host, n);
        if (data1_host) d1.copy_from_host(data1_host, n);
        x.copy_from_host(x_host, n);
        lb.copy_from_host(lb_host, n);
        ub.copy_from_host(ub_host, n);
        LBFGSBParam<double> prm;
        prm.m = q->m; prm.epsilon = q->epsilon; prm.epsilon_rel = q->epsilon_rel; prm.past = q->past; prm.delta = q->delta;
        prm.max_iterations = q->max_iterations; prm.max_submin = q->max_submin; prm.max_linesearch = q->max_linesearch;
        prm.min_step = q->min_step; prm.max_step = q->max_step; prm.ftol = q->ftol; prm.wolfe = q->wolfe;
        LBFGSBSolver<double> solver(prm);
        BuiltinObjective<double> obj(objective, d0.data(), d1.data());
        Traced<BuiltinObjective<double>, double, true> f(obj, fx_trace, trace_cap);
        double fx = 0;
        const unsigned long long launches0 = lbfgs_b200_launch_count(dev.ctx());
        const double t0 = now();
        int niter = 0;
        try { niter = solver.minimize(f, x, fx, lb, ub); }
        catch (...)
        {
            out->nfev = f.count;
            out->trace_len = f.count < trace_cap ? f.count : trace_cap;
            throw;
        }
        dev.synchronize();
        const double t1 = now();
        x.copy_to_host(x_host);
        if (grad_host) solver.final_grad().copy_to_host(grad_host);
        out->niter = niter;
        out->fx = fx;
        out->gnorm = solver.final_grad_norm();
        out->nfev = f.count;
        out->trace_len = f.count < trace_cap ? f.count : trace_cap;
        out->seconds = t1 - t0;
        out->seconds_e2e = now() - t_begin;
        out->launches = lbfgs_b200_launch_count(dev.ctx()) - launches0;
        out->h2d_bytes = 8L * n * 3;
        out->d2h_bytes = 8L * n * (grad_host ? 2 : 1);
    });
}

// Cauchy point on an explicit history (kernel-level test hook): pairs are appended with add_correction, then
// Cauchy<double>::get_cauchy_point runs.  Outputs: xcp (n), classes (n), vecc (2c), counts {nact, nfree}.
extern "C" int lbfgsb200_drv_cauchy_f64(int device_ordinal, long n, int m, int npairs, const double* S_host, const double* Y_host,
                                        const double* x_host, const double* g_host, const double* lb_host, const double* ub_host,
                                        double* xcp_host, unsigned char* cls_host, double* vecc_host, long* counts2, double* theta_out,
                                        char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        typedef DeviceVector<double> Vector;
        BFGSMat<double, true> mat;
        mat.reset(dev, n, m);
        Vector s(dev), y(dev);
        for (int k = 0; k < npairs; k++)
        {
            s.copy_from_host(S_host + size_t(k) * n, n);
            y.copy_from_host(Y_host + size_t(k) * n, n);
            mat.add_correction(s, y);
        }
        mat.refresh_middle();
        Vector x(dev), g(dev), lb(dev), ub(dev);
        x.copy_from_host(x_host, n);
        g.copy_from_host(g_host, n);
        lb.copy_from_host(lb_host, n);
        ub.copy_from_host(ub_host, n);
        const CauchyResult<double> cp = Cauchy<double>::get_cauchy_point(mat, x, g, lb, ub);
        dev.check(lbfgs_b200_memcpy_d2h(dev.ctx(), xcp_host, lbfgs_b200_box_xcp(mat.box()), sizeof(double) * size_t(n)));
        dev.check(lbfgs_b200_memcpy_d2h(dev.ctx(), cls_host, lbfgs_b200_box_classes(mat.box()), size_t(n)));
        for (size_t q = 0; q < cp.vecc.size(); q++) vecc_host[q] = cp.vecc[q];
        counts2[0] = cp.nact;
        counts2[1] = cp.nfree;
        *theta_out = mat.theta();
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}

// ----------------------------------------------------------------------------------------------------------
// Batches of independent problems (BASELINE config 5).  `nthreads` host threads, each with its own context
// (stream, reduction scratch, mailbox) and its own solver object, take problems b = t, t + nthreads, ... ;
// kernels of different problems interleave on the GPU and fill each other's launch/synchronisation gaps.
// Every problem runs exactly the single-problem code path, so its result is bit-identical to a lone solve.
// With a communicator attached to the device's driver context (n-sharded mode) use nthreads = 1.
// ----------------------------------------------------------------------------------------------------------
#include <thread>

typedef struct
{
    int status;
    int niter;
    long nfev;
    double fx;
    double gnorm;
} drv_batch_item;

namespace {

template <template <class> class LS>
void batch_worker(int dev_ordinal, bool use_shared_device, int objective, long n, int B, int first, int stride, const double* x0s,
                  const drv_param* q, int hv_algo, drv_batch_item* items, double* xs_out)
{
    typedef DeviceVector<double> Vector;
    std::unique_ptr<Device> own;
    Device* dev = nullptr;
    int next = first;   // first item this worker has not finished yet
    try
    {
        if (use_shared_device) dev = &device(dev_ordinal);
        else { own.reset(new Device(dev_ordinal)); dev = own.get(); }
        const LBFGSParam<double> prm = to_param<double>(q);
        LBFGSSolver<double, LS> solver(prm);
        solver.set_hv_algorithm(hv_algo);
        BuiltinObjective<double> obj(objective);
        Vector x(*dev);
        for (int b = first; b < B; b += stride)
        {
            drv_batch_item& it = items[b];
            try
            {
                x.copy_from_host(x0s + size_t(b) * n, n);
                double fx = 0;
                it.niter = solver.minimize(obj, x, fx);
                it.fx = fx;
                it.gnorm = solver.final_grad_norm();
                it.nfev = solver.num_evaluations();
                it.status = 0;
                if (xs_out) x.copy_to_host(xs_out + size_t(b) * n);
            }
            catch (const std::invalid_argument&) { it.status = 1; }
            catch (const std::logic_error&) { it.status = 2; }
            catch (const std::runtime_error&) { it.status = 3; }
            catch (const std::exception&) { it.status = 4; }   // e.g. std::bad_alloc from a resize: this item only
            next = b + stride;
        }
    }
    catch (...)
    {
        for (int b = next; b < B; b += stride) items[b].status = 4;   // items already processed keep their outcome
    }
}

}  // namespace

extern "C" int lbfgsb200_drv_batch_f64(int device_ordinal, int objective, long n, int B, const double* x0s_host, int ls,
                                       const drv_param* prm, int hv_algo, int nthreads, int shared_device, drv_batch_item* items,
                                       double* xs_out_host, double* seconds_out)
{
    if (nthreads < 1) nthreads = 1;
    if (shared_device) nthreads = 1;
    for (int b = 0; b < B; b++) items[b] = drv_batch_item{4, 0, 0, 0.0, 0.0};
    const double t0 = now();
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; t++)
    {
        auto fn = [=]() {
            switch (ls)
            {
            case DRV_LS_BACKTRACKING: batch_worker<LineSearchBacktracking>(device_ordinal, shared_device != 0, objective, n, B, t, nthreads, x0s_host, prm, hv_algo, items, xs_out_host); break;
            case DRV_LS_BRACKETING: batch_worker<LineSearchBracketing>(device_ordinal, shared_device != 0, objective, n, B, t, nthreads, x0s_host, prm, hv_algo, items, xs_out_host); break;
            case DRV_LS_NOCEDAL_WRIGHT: batch_worker<LineSearchNocedalWright>(device_ordinal, shared_device != 0, objective, n, B, t, nthreads, x0s_host, prm, hv_algo, items, xs_out_host); break;
            default: batch_worker<LineSearchMoreThuente>(device_ordinal, shared_device != 0, objective, n, B, t, nthreads, x0s_host, prm, hv_algo, items, xs_out_host); break;
            }
        };
        if (nthreads == 1) fn();
        else pool.emplace_back(fn);
    }
    for (auto& th : pool) th.join();
    if (seconds_out) *seconds_out = now() - t0;
    int bad = 0;
    for (int b = 0; b < B; b++) bad += items[b].status != 0;
    return bad;
}

// ----------------------------------------------------------------------------------------------------------
// The same batch as ONE persistent kernel launch (LBFGSBatchSolver, include/LBFGSBatch.h): the start points stay
// resident, solve() can be repeated (bench.py --config c5), every problem bit-identical to a lone resident solve.
// ----------------------------------------------------------------------------------------------------------
namespace {
struct BatchSession
{
    Device* dev;
    long n;
    int B, ls;
    LBFGSParam<double> prm;
    DeviceVector<double> X0, X;
    BuiltinObjective<double> obj;
    LBFGSBatchSolver<double, LineSearchBacktracking> s_bt;
    LBFGSBatchSolver<double, LineSearchBracketing> s_br;
    LBFGSBatchSolver<double, LineSearchNocedalWright> s_nw;
    LBFGSBatchSolver<double, LineSearchMoreThuente> s_mt;
    BatchSession(Device& d, long n_, int B_, int ls_, const drv_param* q, int objective) :
        dev(&d), n(n_), B(B_), ls(ls_), prm(to_param<double>(q)), X0(d), X(d), obj(objective), s_bt(prm), s_br(prm), s_nw(prm), s_mt(prm) {}
};
}  // namespace

extern "C" void* lbfgsb200_drv_batch_session_create(int device_ordinal, int objective, long n, int B, const double* x0s_host, int ls,
                                                    const drv_param* prm, char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        std::unique_ptr<BatchSession> s(new BatchSession(dev, n, B, ls, prm, objective));
        s->X0.copy_from_host(x0s_host, std::ptrdiff_t(n) * B);
        s->X.resize(std::ptrdiff_t(n) * B);
        return s.release();
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return nullptr;
    }
}
extern "C" void lbfgsb200_drv_batch_session_destroy(void* handle) { delete static_cast<BatchSession*>(handle); }

// new start points for the next solve(s), from host memory (B*n doubles): the end-to-end path of a batch
extern "C" int lbfgsb200_drv_batch_session_upload(void* handle, const double* x0s_host, char* err, int errlen)
{
    BatchSession* s = static_cast<BatchSession*>(handle);
    try
    {
        s->X0.copy_from_host(x0s_host, std::ptrdiff_t(s->n) * s->B);
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return -1;
    }
}

// One batched solve from the resident start points.  items[B]; rounds_out[B] (optional); seconds_out: host wall clock around the
// synchronised call; xs_out_host (optional, B*n): the solutions.  Returns the number of problems that did not finish cleanly.
extern "C" int lbfgsb200_drv_batch_session_solve(void* handle, drv_batch_item* items, long* rounds_out, double* xs_out_host, double* seconds_out,
                                                 char* err, int errlen)
{
    BatchSession* s = static_cast<BatchSession*>(handle);
    try
    {
        Device& dev = *s->dev;
        dev.check(lbfgs_b200_memcpy_d2d(dev.ctx(), s->X.data(), s->X0.data(), sizeof(double) * size_t(s->n) * size_t(s->B)));
        dev.synchronize();
        const double t0 = now();
        std::vector<BatchOutcome<double> > out;
        switch (s->ls)
        {
        case DRV_LS_BACKTRACKING: out = s->s_bt.minimize(s->obj, s->X, s->B); break;
        case DRV_LS_BRACKETING: out = s->s_br.minimize(s->obj, s->X, s->B); break;
        case DRV_LS_NOCEDAL_WRIGHT: out = s->s_nw.minimize(s->obj, s->X, s->B); break;
        default: out = s->s_mt.minimize(s->obj, s->X, s->B); break;
        }
        dev.synchronize();
        if (seconds_out) *seconds_out = now() - t0;
        int bad = 0;
        for (int b = 0; b < s->B; b++)
        {
            const BatchOutcome<double>& o = out[size_t(b)];
            items[b].status = o.status == 0 ? 0 : ls_error_kind(o.status);
            items[b].niter = o.niter; items[b].nfev = o.nfev; items[b].fx = o.fx; items[b].gnorm = o.gnorm;
            if (rounds_out) rounds_out[b] = o.rounds;
            bad += o.status != 0;
        }
        if (xs_out_host) s->X.copy_to_host(xs_out_host);
        return bad;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return -1;
    }
}

// accounting of the batch session's last solve (the whole batch is one kernel launch: lbfgs_b200_solver_profile)
extern "C" int lbfgsb200_drv_batch_session_profile(void* handle, double* kernel_ms, double* ms_by_op10, unsigned long long* rounds_by_op10,
                                                   double* alg_bytes_by_op10, double* sync_ms)
{
    BatchSession* s = static_cast<BatchSession*>(handle);
    lbfgs_b200_solver* r = nullptr;
    switch (s->ls)
    {
    case DRV_LS_BACKTRACKING: r = s->s_bt.solver_handle(); break;
    case DRV_LS_BRACKETING: r = s->s_br.solver_handle(); break;
    case DRV_LS_NOCEDAL_WRIGHT: r = s->s_nw.solver_handle(); break;
    default: r = s->s_mt.solver_handle(); break;
    }
    if (!r) return 1;
    return lbfgs_b200_solver_profile(r, kernel_ms, ms_by_op10, rounds_by_op10, alg_bytes_by_op10, sync_ms) == LBFGS_B200_OK ? 0 : 2;
}

// minimize() followed by final_approx_hessian() / final_approx_inverse_hessian() (reference LBFGS.h:192-197) on a built-in objective;
// resident = 1: the device-resident solve (the matrices then come from the solver's own ring), 0: the host-driven loop.
extern "C" int lbfgsb200_drv_solve_dense_f64(int device_ordinal, int objective, long n, int ls, const drv_param* q, int resident, double* x_host,
                                             double* B_out /* n*n */, double* H_out /* n*n */, int* niter_out, char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        const LBFGSParam<double> prm = to_param<double>(q);
        BuiltinObjective<double> obj(objective);
        DeviceVector<double> x(dev);
        x.copy_from_host(x_host, n);
        double fx = 0;
        SmallMatrix<double> Bm, Hm;
        int niter = 0;
        auto run = [&](auto& solver) {
            solver.set_device_resident(resident != 0);
            niter = solver.minimize(obj, x, fx);
            Bm = solver.final_approx_hessian();
            Hm = solver.final_approx_inverse_hessian();
        };
        switch (ls)
        {
        case DRV_LS_BACKTRACKING: { LBFGSSolver<double, LineSearchBacktracking> s(prm); run(s); break; }
        case DRV_LS_BRACKETING: { LBFGSSolver<double, LineSearchBracketing> s(prm); run(s); break; }
        case DRV_LS_NOCEDAL_WRIGHT: { LBFGSSolver<double, LineSearchNocedalWright> s(prm); run(s); break; }
        default: { LBFGSSolver<double, LineSearchMoreThuente> s(prm); run(s); break; }
        }
        x.copy_to_host(x_host);
        for (long i = 0; i < n * n; i++) { B_out[i] = Bm.data()[i]; H_out[i] = Hm.data()[i]; }
        if (niter_out) *niter_out = niter;
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}

// PhaseClock (include/LBFGSpp/PhaseClock.h): wall-clock accounting of the host-driven L-BFGS-B loop's phases for bench.py / profiles
extern "C" void lbfgsb200_drv_phase_enable(int on)
{
    PhaseClock::get().enabled = on != 0;
    PhaseClock::get().reset();
}
// JSON object {"phase": {"seconds": s, "calls": k}, ...} of everything recorded on this thread since the last enable; returns its length
extern "C" int lbfgsb200_drv_phase_report(char* buf, int len)
{
    std::string out = "{";
    bool first = true;
    for (const auto& kv : PhaseClock::get().acc)
    {
        char item[256];
        std::snprintf(item, sizeof(item), "%s\"%s\": {\"seconds\": %.9g, \"calls\": %ld}", first ? "" : ", ", kv.first.c_str(), kv.second.seconds, kv.second.calls);
        out += item;
        first = false;
    }
    out += "}";
    if (buf && len > 0) { std::strncpy(buf, out.c_str(), size_t(len) - 1); buf[len - 1] = 0; }
    return int(out.size());
}

// dense B or H of an explicit history (test hook for final_approx_hessian / final_approx_inverse_hessian)
extern "C" int lbfgsb200_drv_dense_f64(int device_ordinal, long n, int m, int npairs, const double* S_host, const double* Y_host,
                                       int inverse, double* out_host /* n*n row-major */, char* err, int errlen)
{
    try
    {
        Device& dev = device(device_ordinal);
        BFGSMat<double> mat;
        mat.reset(dev, n, m);
        DeviceVector<double> s(dev), y(dev);
        for (int k = 0; k < npairs; k++)
        {
            s.copy_from_host(S_host + size_t(k) * n, n);
            y.copy_from_host(Y_host + size_t(k) * n, n);
            mat.add_correction(s, y);
        }
        const SmallMatrix<double> D = mat.dense(inverse != 0);
        for (long i = 0; i < n * n; i++) out_host[i] = D.data()[i];
        return 0;
    }
    catch (const std::exception& e)
    {
        if (err && errlen > 0) { std::strncpy(err, e.what(), size_t(errlen) - 1); err[errlen - 1] = 0; }
        return 1;
    }
}

#pragma GCC visibility pop
