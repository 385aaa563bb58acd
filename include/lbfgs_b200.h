/* lbfgs_b200.h -- C ABI of liblbfgs_b200.so: the L-BFGS hot path of LBFGSpp on NVIDIA B200 (sm_100a).
 *
 * The reference (yixuan/LBFGSpp @ ebef584) has no FFI: its boundary is a C++ template API whose
 * floating-point work happens inside Eigen expressions.  This header is the contract between the
 * header-only C++ front in include/LBFGS.h (same class names / template parameters as the reference)
 * and the hand-written CUDA kernels.  Every entry point names the reference expression it replaces
 * (paths relative to the reference root).  Conventions:
 *   - plain C types only; device pointers are `void*`/typed pointers into memory obtained from
 *     lbfgs_b200_malloc (256-byte aligned) -- never host memory unless the name says `_host`;
 *   - every call returns a lbfgs_b200_status; no exception crosses the boundary; the text of the last
 *     failure is available from lbfgs_b200_last_error();
 *   - calls are stream-ordered on the context's stream; a call that returns scalars to the host
 *     (`*_host` out-parameters) synchronises the stream before returning, all others are asynchronous;
 *   - reductions are deterministic (fixed grid, fixed-order block partials, no floating-point atomics);
 *     with a communicator attached (n sharded over ranks) every reduction is summed over all ranks;
 *   - a context (and everything created from it) must be used by one host thread at a time;
 *   - there is NO CPU fallback: without a CUDA device every call fails with LBFGS_B200_ERR_CUDA.
 * `T` in {f64, f32} via the suffix.
 */
#ifndef LBFGS_B200_H
#define LBFGS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    LBFGS_B200_OK = 0,
    LBFGS_B200_ERR_INVALID = 1, /* bad argument (maps to std::invalid_argument in the C++ front) */
    LBFGS_B200_ERR_CUDA = 2,    /* CUDA runtime / driver failure, or no device (std::runtime_error) */
    LBFGS_B200_ERR_COMM = 3,    /* NCCL failure (std::runtime_error)                               */
    LBFGS_B200_ERR_ALLOC = 4    /* out of device memory (std::bad_alloc)                           */
} lbfgs_b200_status;

typedef struct lbfgs_b200_ctx lbfgs_b200_ctx;   /* device + stream + reduction scratch + communicator */
typedef struct lbfgs_b200_hist lbfgs_b200_hist; /* the S/Y ring of BFGSMat, resident in HBM           */

/* built-in device objective functions (the reference's example functors, SURVEY.md 8a row A12) */
enum {
    LBFGS_B200_OBJ_ROSENBROCK_PAIRED = 0,  /* examples/example-rosenbrock.cpp:15-27      */
    LBFGS_B200_OBJ_QUAD_SHIFT = 1,         /* examples/example-quadratic.cpp:9-19        */
    LBFGS_B200_OBJ_ROSENBROCK_CHAINED = 2, /* examples/example-rosenbrock-box.cpp:18-33  */
    LBFGS_B200_OBJ_QUAD_TRIDIAG = 3        /* f = 1/2 x'Ax - b'x, A = diag(d) + 1/2 tridiag(-1,2,-1); data0=d, data1=b */
};

/* apply_Hv algorithms */
enum {
    LBFGS_B200_HV_AUTO = 0,      /* currently GRAM                                                             */
    LBFGS_B200_HV_TWO_LOOP = 1,  /* literal two-loop recursion, one fused AXPY+dot stage kernel per history column:
                                    (8c+4) n words of traffic, 2c+1 launches, 2c collectives when sharded      */
    LBFGS_B200_HV_GRAM = 2,      /* the same recursion carried out on 2c coefficients: two passes over S,Y,
                                    (4c+3) n words, 3 launches, 1 collective; differs from TWO_LOOP by rounding */
    LBFGS_B200_HV_GRAM_UNFUSED = 3 /* GRAM, but hist_update_apply_Hv keeps the separate update kernel (s'y, y'y from
                                    its own reduction): the exact arithmetic of the device-resident solve, kept so
                                    that the two solver loops can be compared bit for bit                       */
};

/* ---------------------------------------------------------------- context, memory, communicator */
const char* lbfgs_b200_version(void);
/* stream: a cudaStream_t to run on, or NULL to let the context create its own non-blocking stream. */
lbfgs_b200_status lbfgs_b200_ctx_create(lbfgs_b200_ctx** out, int device, void* stream);
void lbfgs_b200_ctx_destroy(lbfgs_b200_ctx* ctx);
const char* lbfgs_b200_last_error(const lbfgs_b200_ctx* ctx); /* ctx may be NULL: creation errors */
void* lbfgs_b200_stream(const lbfgs_b200_ctx* ctx);
int lbfgs_b200_sm_count(const lbfgs_b200_ctx* ctx);
uint64_t lbfgs_b200_launch_count(const lbfgs_b200_ctx* ctx); /* kernels launched so far by this context */

lbfgs_b200_status lbfgs_b200_malloc(lbfgs_b200_ctx* ctx, void** dptr, size_t bytes); /* replaces Eigen resize(): LBFGS.h:40-50 */
lbfgs_b200_status lbfgs_b200_free(lbfgs_b200_ctx* ctx, void* dptr);
/* Device blocks released by lbfgs_b200_free / *_destroy stay with the context and are handed out again (exact size match): the
 * reference reallocates its work vectors and history in every minimize() (LBFGS.h:84-90, BFGSMat.h:61-67), which on the GPU would
 * cost a cudaMalloc/cudaFree pair and a device-wide synchronisation each.  lbfgs_b200_trim returns the cached blocks to the driver
 * (lbfgs_b200_ctx_destroy does so as well). */
lbfgs_b200_status lbfgs_b200_trim(lbfgs_b200_ctx* ctx);
lbfgs_b200_status lbfgs_b200_malloc_host(lbfgs_b200_ctx* ctx, void** hptr, size_t bytes); /* pinned */
lbfgs_b200_status lbfgs_b200_free_host(lbfgs_b200_ctx* ctx, void* hptr);
lbfgs_b200_status lbfgs_b200_memcpy_h2d(lbfgs_b200_ctx* ctx, void* dst, const void* src_host, size_t bytes);
lbfgs_b200_status lbfgs_b200_memcpy_d2h(lbfgs_b200_ctx* ctx, void* dst_host, const void* src, size_t bytes); /* synchronises */
lbfgs_b200_status lbfgs_b200_memcpy_d2d(lbfgs_b200_ctx* ctx, void* dst, const void* src, size_t bytes);      /* `m_xp = x`, LBFGS.h:121-122 */
lbfgs_b200_status lbfgs_b200_memset_zero(lbfgs_b200_ctx* ctx, void* dst, size_t bytes);
lbfgs_b200_status lbfgs_b200_sync(lbfgs_b200_ctx* ctx);
/* CUDA-event stopwatch on the context's stream (device time of everything enqueued in between) */
lbfgs_b200_status lbfgs_b200_timer_start(lbfgs_b200_ctx* ctx);
lbfgs_b200_status lbfgs_b200_timer_stop(lbfgs_b200_ctx* ctx, float* elapsed_ms_host); /* synchronises */
/* Optional device-time accounting per phase (0 = apply_Hv, 1 = line-search trial, 2 = history update): when
 * enabled every such call is bracketed by a CUDA event pair on the context's stream; profile_read synchronises,
 * returns the accumulated milliseconds / call count and optionally clears them. */
lbfgs_b200_status lbfgs_b200_profile_enable(lbfgs_b200_ctx* ctx, int on);
lbfgs_b200_status lbfgs_b200_profile_read(lbfgs_b200_ctx* ctx, int phase, double* total_ms_host, uint64_t* calls_host, int reset);
/* algorithmic bytes of the profiled calls: apply_Hv w*n*(4c+2), trial w*n*4 (+2 for data vectors), update w*n*6 */
lbfgs_b200_status lbfgs_b200_profile_bytes(lbfgs_b200_ctx* ctx, int phase, double* alg_bytes_host, int reset);
/* n-sharding: global index of this rank's element 0 (used by objectives that depend on the coordinate index) */
lbfgs_b200_status lbfgs_b200_set_index_offset(lbfgs_b200_ctx* ctx, int64_t offset);
/* n-sharding: offset as above plus the global vector length.  Required before a neighbour-coupled built-in objective
 * (chained Rosenbrock, tridiagonal quadratic) is evaluated on a sharded vector: those exchange one boundary coordinate per
 * side with the neighbouring ranks before every evaluation (every block but the last must hold a multiple of 4 coordinates). */
lbfgs_b200_status lbfgs_b200_set_global_extent(lbfgs_b200_ctx* ctx, int64_t offset, int64_t n_global);

/* n-sharding over GPUs (SURVEY.md 8e): rank r owns a contiguous block of every vector; all scalars replicated.
 * unique_id is NCCL's 128-byte ncclUniqueId, created on one rank and shipped to the others by the caller. */
lbfgs_b200_status lbfgs_b200_comm_unique_id(void* unique_id_128);
lbfgs_b200_status lbfgs_b200_comm_init(lbfgs_b200_ctx* ctx, const void* unique_id_128, int rank, int nranks);
int lbfgs_b200_comm_size(const lbfgs_b200_ctx* ctx);
/* In-kernel all-reduce over NVLink peer memory (one process per GPU, same node), replacing the per-reduction NCCL call:
 * every rank exports its inbox (64-byte cudaIpcMemHandle), the application gathers the nranks handles in rank order and
 * every rank attaches them.  From then on the last CTA of every reducing kernel pushes its partial sums into all peers'
 * inboxes, waits for theirs and adds them in rank order: deterministic, identical bits on all ranks, no extra launch.
 * All ranks must issue the same sequence of library calls (they do: the host logic is replicated). */
lbfgs_b200_status lbfgs_b200_comm_p2p_export(lbfgs_b200_ctx* ctx, void* ipc_handle_64);
lbfgs_b200_status lbfgs_b200_comm_p2p_attach(lbfgs_b200_ctx* ctx, const void* all_handles_nranks_x_64, int rank, int nranks);

/* ---------------------------------------------------------------- level-1 kernels (f64 / f32) */
#define LBFGS_B200_DECLARE_L1(T, SUF)                                                                          \
    /* a.dot(b)                                   LBFGS.h:123,161; every LineSearch*.h `grad.dot(drt)` */      \
    lbfgs_b200_status lbfgs_b200_dot_##SUF(lbfgs_b200_ctx*, int64_t n, const T* a, const T* b, T* out_host);   \
    /* out3 = { g.d, g.g, x.x } in one pass       LineSearchMoreThuente.h:414 + LBFGS.h:130,137 */             \
    lbfgs_b200_status lbfgs_b200_dot3_##SUF(lbfgs_b200_ctx*, int64_t n, const T* g, const T* d, const T* x,    \
                                            T* out3_host);                                                    \
    /* out = a + s*b  (out may alias a or b)      `x = xp + step*drt`, LineSearchMoreThuente.h:412 */          \
    lbfgs_b200_status lbfgs_b200_axpy_out_##SUF(lbfgs_b200_ctx*, int64_t n, const T* a, T s, const T* b,       \
                                                T* out);                                                      \
    /* out = s*a                                  `m_drt = -m_grad`, LBFGS.h:106 */                            \
    lbfgs_b200_status lbfgs_b200_scale_out_##SUF(lbfgs_b200_ctx*, int64_t n, T s, const T* a, T* out);         \
    /* built-in objective: g = grad f(x), out4 = { f(x), 0, g.g, x.x }   (user functor, LBFGS.h:69-71,91-92) */ \
    lbfgs_b200_status lbfgs_b200_objective_##SUF(lbfgs_b200_ctx*, int objective, const T* data0,               \
                                                 const T* data1, int64_t n, const T* x, T* g, T* out4_host);   \
    /* One line-search trial for a built-in objective in ONE kernel:                                           \
     *   x = xp + step*d;  g = grad f(x);  out4 = { f(x), g.d, g.g, x.x }                                      \
     * replaces LineSearchMoreThuente.h:412-414 (and the same three lines of the other three line searches)    \
     * plus the norms of LBFGS.h:130,137. */                                                                   \
    lbfgs_b200_status lbfgs_b200_trial_##SUF(lbfgs_b200_ctx*, int objective, const T* data0, const T* data1,   \
                                             int64_t n, const T* xp, const T* d, T step, T* x, T* g,          \
                                             T* out4_host);

LBFGS_B200_DECLARE_L1(double, f64)
LBFGS_B200_DECLARE_L1(float, f32)

/* ---------------------------------------------------------------- the S/Y ring (BFGSMat, L-BFGS part) */
/* elem_bytes: 8 (fp64) or 4 (fp32).  Replaces BFGSMat::reset's allocations, BFGSMat.h:61-78. */
lbfgs_b200_status lbfgs_b200_hist_create(lbfgs_b200_ctx* ctx, lbfgs_b200_hist** out, int64_t n, int m,
                                         int elem_bytes);
void lbfgs_b200_hist_destroy(lbfgs_b200_hist* h);
/* theta = 1, ncorr = 0 (no reallocation).  BFGSMat.h:61-78. */
lbfgs_b200_status lbfgs_b200_hist_reset(lbfgs_b200_hist* h);
int lbfgs_b200_hist_ncorr(const lbfgs_b200_hist* h);
int lbfgs_b200_hist_m(const lbfgs_b200_hist* h);
/* device pointers of logical column `age` (0 = newest) for inspection / tests; NULL if age >= ncorr */
const void* lbfgs_b200_hist_s_col(const lbfgs_b200_hist* h, int age);
const void* lbfgs_b200_hist_y_col(const lbfgs_b200_hist* h, int age);

#define LBFGS_B200_DECLARE_HIST(T, SUF)                                                                        \
    /* s = x - xp, y = g - gp written straight into the next ring slot, gate s'y > eps*y'y, ys, theta:         \
     * LBFGS.h:159-162 + BFGSMat::add_correction BFGSMat.h:81-97, one kernel.  sy_yy_host (2 values) optional. */ \
    lbfgs_b200_status lbfgs_b200_hist_update_##SUF(lbfgs_b200_hist* h, const T* x, const T* xp, const T* g,    \
                                                   const T* gp, T eps, int* accepted_host, T* sy_yy_host);    \
    /* add_correction(s, y) for explicit vectors (BFGSMat.h:81-97); no gate. */                                \
    lbfgs_b200_status lbfgs_b200_hist_add_##SUF(lbfgs_b200_hist* h, const T* s, const T* y);                   \
    /* res = a * H * v by the two-loop recursion, BFGSMat::apply_Hv BFGSMat.h:276-302.                         \
     * gdotres_host (optional) receives v.res, i.e. `dg = m_grad.dot(m_drt)` of LBFGS.h:123 when v = grad.     \
     * res must not alias v. */                                                                                \
    lbfgs_b200_status lbfgs_b200_hist_apply_Hv_##SUF(lbfgs_b200_hist* h, const T* v, T a, T* res, int algo,    \
                                                     T* vdotres_host);                                        \
    /* LBFGS.h:159-165 in one call: hist_update(x, xp, g, gp) followed by apply_Hv(v = g, a, res) (+ g.res).   \
     * With the Gram form the pair is formed inside the dots pass, so x, xp, g, gp are read once and no         \
     * separate update kernel runs; otherwise equivalent to the two calls.  res must not alias an input. */    \
    lbfgs_b200_status lbfgs_b200_hist_update_apply_Hv_##SUF(lbfgs_b200_hist* h, const T* x, const T* xp,       \
                                                            const T* g, const T* gp, T eps, T a, T* res,       \
                                                            int algo, int* accepted_host, T* gdotres_host);    \
    /* host copies of theta and of ys/alpha by age (newest first), for tests */                                \
    lbfgs_b200_status lbfgs_b200_hist_scalars_##SUF(lbfgs_b200_hist* h, T* theta_host, T* ys_host,             \
                                                    T* alpha_host);

LBFGS_B200_DECLARE_HIST(double, f64)
LBFGS_B200_DECLARE_HIST(float, f32)

/* ---------------------------------------------------------------- bound-constrained path (LBFGSBSolver, config 4)
 * Index sets of the reference (std::vector<int> free / active / L / U / P sets of Cauchy.h and SubspaceMin.h) are bits of
 * a per-coordinate class byte; W = [Y, theta*S] is never gathered: every W-product is a masked pass over the S/Y columns.
 * The 2m x 2m algebra (Minv, BKLDLT, the BOXCQP bookkeeping) stays on the host in the C++ front, as in the reference.
 * Replicas only: these entry points refuse a context with more than one rank.  m <= 20. */
typedef struct lbfgs_b200_box lbfgs_b200_box;   /* n-sized temporaries of Cauchy / SubspaceMin + sort buffers */
enum { LBFGS_B200_CLS_FIXED = 1, LBFGS_B200_CLS_ACT = 2, LBFGS_B200_CLS_FREE = 4,
       LBFGS_B200_SUB_L = 8, LBFGS_B200_SUB_U = 16, LBFGS_B200_SUB_P = 32 };
/* element-wise steps of SubspaceMin::subspace_minimize (SubspaceMin.h:122-302), see lbfgsb_kernels.cuh */
enum { LBFGS_B200_SUB_INIT = 0, LBFGS_B200_SUB_ACT_DIR = 1, LBFGS_B200_SUB_ADD_G = 2, LBFGS_B200_SUB_NEG_C_FREE = 3,
       LBFGS_B200_SUB_CHECK_BOUNDS = 4, LBFGS_B200_SUB_CLASSIFY = 5, LBFGS_B200_SUB_LU_VEC = 6, LBFGS_B200_SUB_RHS_P = 7,
       LBFGS_B200_SUB_FREE_VEC = 8, LBFGS_B200_SUB_MULTIPLIERS = 9, LBFGS_B200_SUB_CONVERGED = 10,
       LBFGS_B200_SUB_WRITE_DRT = 11 };
/* work vectors of the box workspace, for lbfgs_b200_box_vector() */
enum { LBFGS_B200_BOXV_VECC = 0, LBFGS_B200_BOXV_VECY = 1, LBFGS_B200_BOXV_LAMBDA = 2, LBFGS_B200_BOXV_MU = 3,
       LBFGS_B200_BOXV_TMP = 4, LBFGS_B200_BOXV_TMP2 = 5, LBFGS_B200_BOXV_YFB = 6, LBFGS_B200_BOXV_DVEC = 7,
       LBFGS_B200_BOXV_BRK = 8, LBFGS_B200_BOXV_XCP = 9 };

lbfgs_b200_status lbfgs_b200_box_create(lbfgs_b200_hist* h, lbfgs_b200_box** out);
void lbfgs_b200_box_destroy(lbfgs_b200_box* b);
const void* lbfgs_b200_box_xcp(const lbfgs_b200_box* b);                 /* generalized Cauchy point (device, n)   */
const unsigned char* lbfgs_b200_box_classes(const lbfgs_b200_box* b);    /* class bytes (device, n)                */
void* lbfgs_b200_box_vector(lbfgs_b200_box* b, int which);               /* LBFGS_B200_BOXV_* (device, n)          */

#define LBFGS_B200_DECLARE_BOX(T, SUF)                                                                         \
    /* x = x.cwiseMax(lb).cwiseMin(ub)                                   force_bounds, LBFGSB.h:55-58 */        \
    lbfgs_b200_status lbfgs_b200_box_clamp_##SUF(lbfgs_b200_ctx*, int64_t n, T* x, const T* lb, const T* ub);  \
    /* max_i |clamp(x - g) - x|                                          proj_grad_norm, LBFGSB.h:62-65 */      \
    lbfgs_b200_status lbfgs_b200_box_proj_grad_norm_##SUF(lbfgs_b200_ctx*, int64_t n, const T* x, const T* g,  \
                                                          const T* lb, const T* ub, T* out_host);              \
    /* out2 = { g.d , largest feasible step along d }                    LBFGSB.h:176 + max_step_size :68-86 */ \
    lbfgs_b200_status lbfgs_b200_box_dir_info_##SUF(lbfgs_b200_ctx*, int64_t n, const T* x, const T* d,        \
                                                    const T* g, const T* lb, const T* ub, T* out2_host);       \
    /* raw[2c] = { y_age.v (c), s_age.v (c) }        apply_Wtv / apply_WtPv without theta, BFGSMat.h:315-320,382-433 */ \
    lbfgs_b200_status lbfgs_b200_hist_wt_dot_##SUF(lbfgs_b200_hist*, const T* v, T* raw_host);                 \
    /* c x c Gram blocks by age (row-major, any may be NULL): s_i.y_j, s_i.s_j, y_i.y_j; ys[c]; theta  (the material   \
     * of m_permMinv, BFGSMat.h:99-146) */                                                                     \
    lbfgs_b200_status lbfgs_b200_hist_gram_##SUF(lbfgs_b200_hist*, T* SY_host, T* SS_host, T* YY_host,         \
                                                 T* ys_host, T* theta_host);                                   \
    /* out_i = a0*v0_i + sum_j cy_j*y_j[i] + cs_j*s_j[i] on rows with (cls_i & mask) != 0 (cls NULL: all rows);        \
     * coef_host = { cy by age (c), cs by age (c) }.    apply_PtWMv / apply_PtBQv / solve_PtBP tail, BFGSMat.h:435-615 */ \
    lbfgs_b200_status lbfgs_b200_hist_lincomb_##SUF(lbfgs_b200_hist*, lbfgs_b200_box*, T a0, const T* v0,      \
                                                    const T* coef_host, const unsigned char* cls, int mask,    \
                                                    T* out);                                                   \
    /* G[(2c)x(2c)] = sum over rows with (cls & mask) of r r', r = (y_0[i]..,s_0[i]..) by age.  WP'WP, BFGSMat.h:529-565 */ \
    lbfgs_b200_status lbfgs_b200_hist_masked_gram_##SUF(lbfgs_b200_hist*, lbfgs_b200_box*,                     \
                                                        const unsigned char* cls, int mask, T* G_host);        \
    /* Cauchy.h:111-129: breakpoints, d = -g on movable coordinates, class bytes.                                      \
     * out5 = { #fixed, #never-bounded, #with a finite breakpoint, d.d, smallest breakpoint } */                       \
    lbfgs_b200_status lbfgs_b200_box_cauchy_breaks_##SUF(lbfgs_b200_box*, const T* x, const T* g, const T* lb, \
                                                         const T* ub, T* out5_host);                           \
    /* Cauchy.h:132-256: sort the breakpoints, prefix sums, first segment holding its one-dimensional minimiser.       \
     * Mmat_host [2c][2c] (B = theta I - W M W'), p0_host = W'd [2c].                                                  \
     * out = { t_cross, tfinal, f', f'', all-crossed flag, W'(xcp - x0) [2c] } */                                      \
    lbfgs_b200_status lbfgs_b200_box_cauchy_sweep_##SUF(lbfgs_b200_box*, const T* g, const T* Mmat_host,       \
                                                        const T* p0_host, T theta, T gt, int64_t nord,         \
                                                        int64_t nfree_inf, T* out_host);                       \
    /* Cauchy.h:205-216,268-283: xcp and the ACT / FREE classes from (t_cross, tfinal); counts2 = { #act, #free } */   \
    lbfgs_b200_status lbfgs_b200_box_cauchy_build_##SUF(lbfgs_b200_box*, const T* x, const T* lb, const T* ub, \
                                                        T t_cross, T tfinal, T* counts2_host);                 \
    /* one element-wise step (LBFGS_B200_SUB_*) of SubspaceMin.h:122-302; reducing steps return 3 counters */          \
    lbfgs_b200_status lbfgs_b200_box_sub_step_##SUF(lbfgs_b200_box*, int op, int flag, const T* x0,            \
                                                    const T* g, const T* lb, const T* ub, T* drt, T theta,     \
                                                    T* out3_host);

LBFGS_B200_DECLARE_BOX(double, f64)
LBFGS_B200_DECLARE_BOX(float, f32)

/* ---------------------------------------------------------------- device-resident solve (built-in objectives)
 * LBFGSSolver<Scalar, LineSearch>::minimize() (reference LBFGS.h:78-173) as ONE persistent cooperative kernel launch, for one problem
 * or for a batch of B independent problems of the same shape (BASELINE config 5).  One CTA per SM stays resident for the whole
 * solve; the work proceeds in rounds of one streaming pass per running problem (first evaluation / line-search trial /
 * pair-forming dots [S Y]'[g s y] / combination d = -H g fused with the first trial of the next search) separated by one grid-wide
 * synchronisation in which CTA 0 sums the CTAs' partial sums in a fixed order, exchanges them with the other ranks when n is
 * sharded (ONE exchange per round for all running problems: a B-vector all-reduce per dot) and runs every problem's scalar logic:
 * the line-search state machines (include/LBFGSpp/LineSearchCore.h, the code the host front uses), the convergence tests of
 * LBFGS.h:137-154, the curvature gate of :161, the ring bookkeeping of BFGSMat.h:81-97 and the buffer rotation.  The host is not
 * involved between launch and completion.  Reductions are deterministic and a problem's result does not depend on what else is
 * in the batch: every problem of a batch is bit-identical to the same problem solved alone.
 * When n is sharded the in-kernel NVLink exchange must be attached (lbfgs_b200_comm_p2p_*); neighbour-coupled objectives then
 * also need lbfgs_b200_set_global_extent (their boundary coordinates travel with the sums). */
typedef struct lbfgs_b200_solver lbfgs_b200_solver;
typedef struct {             /* LBFGSParam (reference Param.h:67-219); doubles for both precisions */
    int m;
    double epsilon, epsilon_rel;
    int past;
    double delta;
    int max_iterations;
    int linesearch;
    int max_linesearch;
    double min_step, max_step, ftol, wolfe;
} lbfgs_b200_param;
typedef struct {
    int status;              /* 0, or a LBFGSpp::LineSearchError code (>= 16) = the exception the reference would throw */
    int niter;               /* return value of minimize()                                                          */
    long long nfev;          /* objective evaluations                                                               */
    double fx, gnorm;
    long long rounds;        /* streaming passes (= grid-wide synchronisations) this problem took part in           */
} lbfgs_b200_outcome;
enum { LBFGS_B200_LS_BACKTRACKING = 0, LBFGS_B200_LS_BRACKETING = 1, LBFGS_B200_LS_NOCEDAL_WRIGHT = 2, LBFGS_B200_LS_MORE_THUENTE = 3 };

lbfgs_b200_status lbfgs_b200_solver_create(lbfgs_b200_ctx* ctx, int64_t n, int m, int elem_bytes, lbfgs_b200_solver** out);
/* batch problems of n coordinates each (n = this rank's block when sharded), all with history size m */
lbfgs_b200_status lbfgs_b200_solver_create_batch(lbfgs_b200_ctx* ctx, int64_t n, int m, int elem_bytes, int batch, lbfgs_b200_solver** out);
void lbfgs_b200_solver_destroy(lbfgs_b200_solver* s);
int lbfgs_b200_solver_batch(const lbfgs_b200_solver* s);
/* Accounting of the last solve.  kernel_ms: device time of the one kernel (CUDA events around its launch).  The arrays have 10 slots
 * indexed by the pass a round ran: 0 = rounds in which the problems of a batch ran different passes, 1 FIRST, 2 TRIAL, 3 DOTS_FORM,
 * 4 DOTS_PLAIN, 5 COMBINE, 6 COMBINE_TRIAL, 7 RESTORE, 8 MATERIALIZE (9 unused).  ms_by_op10: the kernel's time split by round (CTA 0's cycle counter scaled
 * to kernel_ms; includes each round's synchronisation); alg_bytes_by_op10: algorithmic bytes of those passes (whole vectors read and
 * written: FIRST 3n, TRIAL 4n, DOTS_FORM (2c+4)n, DOTS_PLAIN (2c+1)n, COMBINE (2c+2)n, COMBINE_TRIAL (2c+3)n words or (2c+5)n when the first trial's x, g are stored, MATERIALIZE 4n words, + the objective's
 * data vectors per evaluation); sync_ms[3]: { the part of kernel_ms between CTA 0's arrival at a grid barrier and its release, the part of that spent waiting for
 * the last CTA to arrive, the part spent in the cross-rank exchange }. */
lbfgs_b200_status lbfgs_b200_solver_profile(const lbfgs_b200_solver* s, double* kernel_ms, double* ms_by_op10, unsigned long long* rounds_by_op10,
                                            double* alg_bytes_by_op10, double* sync_ms);
const void* lbfgs_b200_solver_final_grad(const lbfgs_b200_solver* s);   /* device pointer (problem 0), valid until the next minimize */
const void* lbfgs_b200_solver_final_grad_of(const lbfgs_b200_solver* s, int problem);
lbfgs_b200_hist* lbfgs_b200_solver_history(lbfgs_b200_solver* s);       /* the S/Y ring of problem 0 as left by the last solve   */
lbfgs_b200_hist* lbfgs_b200_solver_history_of(lbfgs_b200_solver* s, int problem);
/* x_inout: device vector (start point in, solution out).  trace_host (optional): f of every evaluation.
 * data0/data1 (the tridiagonal quadratic's d and b): device vectors, 16-byte aligned.  They are read by bulk copies of whole 256-byte
 * lines, so each must stay readable up to n rounded up to a multiple of 256 bytes (32 fp64 / 64 fp32 elements); the values past n
 * are never used.  Memory from lbfgs_b200_malloc(n * elem_bytes) satisfies both.  A misaligned pointer fails with
 * LBFGS_B200_ERR_INVALID, as does a configuration whose passes do not fit the kernel's staging ring (LBFGS_B200_STAGES). */
lbfgs_b200_status lbfgs_b200_solver_minimize_f64(lbfgs_b200_solver* s, int objective, const double* data0, const double* data1,
                                                 const lbfgs_b200_param* prm, int line_search, double* x_inout,
                                                 double* trace_host, long long trace_cap, lbfgs_b200_outcome* out);
lbfgs_b200_status lbfgs_b200_solver_minimize_f32(lbfgs_b200_solver* s, int objective, const float* data0, const float* data1,
                                                 const lbfgs_b200_param* prm, int line_search, float* x_inout,
                                                 double* trace_host, long long trace_cap, lbfgs_b200_outcome* out);
/* Batch: problem b starts from x_inout + b*ldx (device) and leaves its solution there; data0/data1 (optional) per problem at
 * data + b*ldd (ldd = 0: shared by all problems; otherwise ldd >= n and ldd * elem_bytes a multiple of 16, else
 * LBFGS_B200_ERR_INVALID).  The padded tail above applies to every problem's vectors: a buffer of (batch - 1) * ldd elements plus n
 * rounded up to 256 bytes is enough.  outs[batch]. */
lbfgs_b200_status lbfgs_b200_solver_minimize_batch_f64(lbfgs_b200_solver* s, int objective, const double* data0, const double* data1,
                                                       int64_t ldd, const lbfgs_b200_param* prm, int line_search, double* x_inout,
                                                       int64_t ldx, lbfgs_b200_outcome* outs);
lbfgs_b200_status lbfgs_b200_solver_minimize_batch_f32(lbfgs_b200_solver* s, int objective, const float* data0, const float* data1,
                                                       int64_t ldd, const lbfgs_b200_param* prm, int line_search, float* x_inout,
                                                       int64_t ldx, lbfgs_b200_outcome* outs);

#ifdef __cplusplus
}
#endif
#endif /* LBFGS_B200_H */
