// persist.cuh -- the device-resident L-BFGS solve: LBFGSSolver::minimize() (reference LBFGS.h:78-173) for built-in objectives as
// ONE persistent cooperative kernel launch, for one problem or for a batch of B independent problems (BASELINE config 5).
// Included by persist_f64.cu / persist_f32.cu.
//
// The kernel is a "phase machine".  One CTA per SM (768 threads), all co-resident (cooperative launch).  Work proceeds in ROUNDS;
// in a round every problem that is still running executes the ONE streaming pass its state asks for:
//     FIRST          g = grad f(x0), d = -g                      ; {f, g.g, x.x}                            LBFGS.h:91-108
//     TRIAL          x = xp + step*d, g = grad f(x)              ; {f, g.d, g.g, x.x}                       LineSearch*.h trial, LBFGS.h:130,137
//     DOTS_FORM      s = x - xp, y = g - gp -> free ring slot    ; [S Y]'[g s y] (6 dots per column pair)   LBFGS.h:159-162, BFGSMat.h:85-92 + apply_Hv pass 1
//     DOTS_PLAIN     (pair rejected by the curvature gate)       ; [S Y]'g over the old history
//     COMBINE        coefficient recursion (every CTA, shared memory) ; d = cv*g + sum cy_j y_j + cs_j s_j ; {g.d}   BFGSMat.h:283-301 in Gram form
//     COMBINE_TRIAL  COMBINE + the first trial of the next line search in the same pass: the reference restarts every search
//                    at step = 1 (LBFGS.h:168), so x1 = x + d, g1 = grad f(x1) ; {g.d, f1, g1.d, g1.g1, x1.x1}
//     RESTORE        x = xp, g = gp (a search that never improved on its start point; LineSearchMoreThuente.h:602-614)
//     MATERIALIZE    x = xp + step*d, g = grad f(x) for a trial whose sums are already known: optional policy in which the fused first trial
//                    does not store x1, g1 while first trials keep being rejected (see digest_trial; off by default)
// Every CTA owns the same contiguous chunk (granularity: the block length of the tiled history) of EVERY vector in EVERY pass, so a CTA only ever reads vector
// elements it wrote itself (halo coordinates excepted, those are read through L2) and streams long contiguous runs.  Between rounds there is one
// grid-wide synchronisation: CTAs deposit their partial sums in fixed slots, CTA 0 adds them in a fixed order (deterministic: no
// floating-point atomics, result independent of which other problems are in flight), exchanges them with the other ranks when
// n is sharded (ONE exchange per round carrying the sums of all running problems = "one all-reduce of a B-vector per dot"), runs
// each problem's scalar logic -- line-search state machine (the cores of include/LBFGSpp/LineSearchCore.h, the same code the host
// front uses), convergence tests (LBFGS.h:137-154), curvature gate (:161), ring bookkeeping (BFGSMat.h:81-97), buffer rotation
// (pointer swaps) -- and publishes one 128-byte descriptor per problem that tells every CTA what the next round does.  The host is
// not involved between launch and completion: 1 launch per minimize(), 2 + (T - 1) rounds per iteration with T line-search trials.
//
// Data movement: ALL operands of the dots and combination passes -- the right-hand vectors and the 2c history columns, which live in
// a tiled layout (PHist) so that the columns of a tile are one or two contiguous runs -- are staged into shared memory by TMA bulk
// copies (cp.async.bulk + mbarrier) in a two-stage ring of ~90 KB stages: the bytes in flight per SM are set by the ring, not by
// registers.  The trial pass streams through registers (256-bit loads / stores).  Vectors owned by the solver are padded to whole
// 256-byte lines, so every tile -- the ragged end of a vector included -- is a legal bulk copy; lanes past n are masked in the
// arithmetic.  The coefficient recursion of a combination pass runs from a scratch area of its own while the pass's first tiles
// are in flight.  DESIGN.md section 10 has what was measured about the limits of this arrangement.
#pragma once

#include "../../include/LBFGSpp/LineSearchCore.h"
#include "persist_geometry.h"

namespace lb {

constexpr int kMaxPast = 64;
constexpr int kPThreads = kGramMaxThreads;   // 768: one CTA per SM
constexpr int kPWarps = kPThreads / 32;
static_assert(kPStageBytes == kGramStages * 4 * kGramTE * 8, "the staging ring is the Gram kernels' three stages of four fp64 tiles");
constexpr int kPCache = 4;                   // problems whose leader-side state is kept in shared memory

enum { POP_IDLE = 0, POP_FIRST = 1, POP_TRIAL = 2, POP_DOTS_FORM = 3, POP_DOTS_PLAIN = 4, POP_COMBINE = 5, POP_COMBINE_TRIAL = 6, POP_RESTORE = 7,
       POP_MATERIALIZE = 8 };
constexpr int kPOps = 10;   // accounting slots (ops + the "mixed" bucket 0)
constexpr int kPGramScratch = 1024;   // doubles

// ---- the S/Y history of the solve: tiled layout ---------------------------------------------------------------------------------
// H[block][slot][S|Y][BT]: all ring slots of one block of BT coordinates lie next to each other (BT = the largest power of two for
// which two stages of 2m+4 rows fit the kernel's shared memory: 512 for fp64 m = 10).  A pass over a tile then needs the right-hand
// vectors plus ONE or TWO bulk copies of 8..90 KB for all history columns (the live slots form a cyclic range of the ring), instead
// of one 4 KB copy per column: measured, the per-copy cost of 22 separate copies was ~15 % of the combination pass, and 42 copies of
// 2 KB at m = 20 made it 2.8x slower per byte.  The new pair of an iteration is written as one 2*BT run per block.
template <class T> struct PHist
{
    T* H;
    int bt_log, M;
    int64_t bstride;      // elements per block: M * 2 * BT
    __device__ __forceinline__ int BT() const { return 1 << bt_log; }
    __device__ __forceinline__ T* s_at(int slot, int64_t i) const { return H + (i >> bt_log) * bstride + ((int64_t)slot << (bt_log + 1)) + (i & (BT() - 1)); }
    __device__ __forceinline__ T* y_at(int slot, int64_t i) const { return s_at(slot, i) + BT(); }
};

// ---- per-problem state (device memory; the leader CTA's working copy) ----------------------------------------------------------
template <class T> struct PState
{
    // vectors (rotate by pointer swap)
    T *x, *xp, *g, *gp, *drt, *x_lo, *g_lo;
    // history storage (fixed for the duration of the kernel: other CTAs read these fields with ordinary loads)
    PHist<T> hist;              // the S/Y ring, tiled (see PHist)
    T *ys, *alpha, *theta;
    T *SY[2], *YY[2], *SS[2];
    const T *data0, *data1;
    double* raw;               // [pstride] reduced values of the last round
    double* halo;              // kHaloDoubles (neighbour-coupled objectives under n-sharding)
    // ring geometry
    int head, ncorr, M, m, gram_cur, pending;
    // what the next round does
    int op, c_round;
    // options (LBFGSParam)
    T epsilon, epsilon_rel, delta, max_step, eps_gate;
    int past, max_iterations, ls_kind, fuse_first_trial;
    LBFGSpp::LineSearchOptions<T> ls_opt;
    // line-search state
    LBFGSpp::BacktrackingCore<T> bt;
    LBFGSpp::BracketingCore<T> br;
    LBFGSpp::NocedalWrightCore<T> nw;
    LBFGSpp::MoreThuenteCore<T> mt;
    int have_lo;
    T lo_gg, lo_xx, start_gg, start_xx;
    // the fused first trial of a search may be "virtual": evaluated and reduced, but x1 / g1 not stored
    int first_store;            // policy for the next COMBINE_TRIAL pass: 1 = store x1, g1
    int adaptive_first_store;   // 1: first_store follows the fate of the last first trial (accepted -> store); 0: always store
    int lo_virtual;             // the best-so-far point (x_lo, g_lo) is the virtual first trial: materialise it at lo_step if needed
    T lo_step;
    int after_materialize;      // what MATERIALIZE was for: 1 = the accepted trial, 2 = the best-so-far point
    // iteration scalars
    T fx, dg, gg, xx, gnorm, step;
    int k;
    long long nfev;
    int status;     // 0 ok, otherwise a LineSearchError code
    int finished;
    int niter;      // return value of minimize()
    T fx_hist[kMaxPast];
    double* trace;              // optional: f of every evaluation
    long long trace_cap;
    long long rounds;           // rounds this problem took part in
};

// what every CTA needs to know about a problem's next round: one 128-byte line, written by the leader, read through L2
template <class T> struct alignas(128) PRound
{
    T *x, *xp, *g, *gp, *drt;
    T step;
    int op, c_round, head, pending, gram_cur, store_first;
};

struct alignas(128) PCtl
{
    unsigned arrive;            // grid barrier: arrivals so far (monotonic); a cache line of its own
    unsigned pad0[31];
    unsigned release;           // grid barrier: last episode released by the leader; bit 31 = nothing left to do
    unsigned pad1[31];
    int abort;                  // watchdog tripped (a wait exceeded its budget): everybody leaves
    int nactive;                // problems still running
    unsigned long long epoch;   // cross-rank exchange sequence number (continues the context's)
    unsigned long long rounds;
    // accounting by CTA 0 (clock64 cycles of its SM): wall time of the rounds by the op they ran (bucket 0: rounds in which
    // problems ran different ops), the part of it spent between CTA 0's own arrival and the release (waiting for the slowest
    // CTA + the leader's work), and the algorithmic n-words of the passes (what the design has to move, see words_of)
    long long cyc_op[kPOps];
    long long cyc_sync;
    long long cyc_wait_all;     // of cyc_sync: from CTA 0's own arrival until the last CTA has arrived
    long long cyc_exchange;     // of cyc_sync: the cross-rank exchange (push, wait for every peer's flag, rank-ordered sums)
    unsigned long long n_op[kPOps];
    double words_op[kPOps];
};
constexpr unsigned kPStopBit = 0x80000000u;

template <class T> struct PArgs
{
    PState<T>* probs;
    PRound<T>* rounds;
    int B;
    PCtl* ctl;
    double* partials;           // [B][pstride][G]
    int pstride;
    int64_t n;
    int grain;                  // chunk boundaries are multiples of this many elements (= the history's block length)
    const XComm* xc;
    int64_t index_offset, n_global;
    long long wait_cycles;      // watchdog budget of a grid-barrier wait (clock64 ticks); cross-rank waits get 4x, the release wait 6x
    int tune;                   // 4 = the trial pass stores x, g with L2 evict-first: +3 % on that pass at n = 1e7 (set by the host when the vectors cannot stay
                                // in L2 anyway; LBFGS_B200_TUNE overrides).  Measured and dropped: unrolling the pass 4x (no change), prefetching its inputs
                                // into L2 (-5 %), a grid-stride instead of a chunked sweep (+1 %)
};

template <class V> __device__ __forceinline__ V ldv(const V* p) { return *reinterpret_cast<const volatile V*>(p); }

template <class T> __device__ __forceinline__ T& ls_step_ref(PState<T>* st)
{
    switch (st->ls_kind)
    {
    case 0: return st->bt.step;
    case 1: return st->br.step;
    case 2: return st->nw.step;
    default: return st->mt.step;
    }
}
template <class T> __device__ __forceinline__ int ls_init(PState<T>* st, T fx, T dg, T step, T step_max)
{
    switch (st->ls_kind)
    {
    case 0: return st->bt.init(st->ls_opt, fx, dg, step, step_max);
    case 1: return st->br.init(st->ls_opt, fx, dg, step, step_max);
    case 2: return st->nw.init(st->ls_opt, fx, dg, step, step_max);
    default: return st->mt.init(st->ls_opt, fx, dg, step, step_max);
    }
}
template <class T> __device__ __forceinline__ int ls_advance(PState<T>* st, T fx, T dg, bool& keep)
{
    switch (st->ls_kind)
    {
    case 0: return st->bt.advance(fx, dg, keep);
    case 1: return st->br.advance(fx, dg, keep);
    case 2: return st->nw.advance(fx, dg, keep);
    default: return st->mt.advance(fx, dg, keep);
    }
}
template <class T> __device__ __forceinline__ void ls_best(PState<T>* st, T& fx, T& dg)
{
    switch (st->ls_kind)
    {
    case 0: fx = st->bt.best_fx; dg = st->bt.best_dg; break;
    case 1: fx = st->br.best_fx; dg = st->br.best_dg; break;
    case 2: fx = st->nw.best_fx; dg = st->nw.best_dg; break;
    default: fx = st->mt.best_fx; dg = st->mt.best_dg; break;
    }
}
template <class P> __device__ __forceinline__ void dswap(P& a, P& b) { P t = a; a = b; b = t; }
__device__ __forceinline__ int slot_by_age(int head, int M, int age) { return ((head - 1 - age) % M + M) % M; }

// ---- objectives as the persistent kernel builds them ------------------------------------------------------------------------
template <class T, class OBJ> struct PObjMaker;
template <class T> struct PObjMaker<T, RosenbrockPaired<T> >
{ static __device__ RosenbrockPaired<T> make(const PArgs<T>& a, const T*, const T*, const double*) { return RosenbrockPaired<T>{a.n}; } };
template <class T> struct PObjMaker<T, QuadShift<T> >
{ static __device__ QuadShift<T> make(const PArgs<T>& a, const T*, const T*, const double*) { return QuadShift<T>{a.n, a.index_offset}; } };
template <class T> struct PObjMaker<T, RosenbrockChained<T> >
{ static __device__ RosenbrockChained<T> make(const PArgs<T>& a, const T*, const T*, const double* halo)
  { return RosenbrockChained<T>{a.n, a.index_offset, a.n_global, halo}; } };
template <class T> struct PObjMaker<T, QuadTridiag<T> >
{ static __device__ QuadTridiag<T> make(const PArgs<T>& a, const T* d0, const T* d1, const double* halo)
  { return QuadTridiag<T>{a.n, d0, d1, a.index_offset, a.n_global, halo}; } };

// ---- shared memory of the kernel ----------------------------------------------------------------------------------------------
struct PShared
{
    uint64_t full_bar[kPMaxStages];
    double red[kPWarps][3 * kGramVals];     // block reduction scratch (dots: ROUNDS*6 values per warp)
    double coef[2 * kMaxM + 2];             // combination coefficients {cv, cy[c], cs[c]} (stored as T)
    const void* vecs[2 * kMaxM + 2];        // combination pass: the staged vectors {g, (x), y_0.., s_0..} in coefficient order
    unsigned char slots[kMaxM];             // by age: packed row of the column in the staged history block
    unsigned char slotid[kMaxM];            // by age: physical ring slot
    double margin[2][2 * kMaxM + 2];        // neighbour-coupled combination pass: products of the element on either side of a tile
    double carry[2];                        // ... and x1 of the last element of the previous tile (two slots, alternating)
    unsigned char ops[4096];                // this round's op of every problem
};

// Ownership.  CTA i owns the contiguous chunk [c0, c1) of every vector (boundaries on multiples of the history's block length, the
// chunks differ by at most one block) in EVERY pass: a CTA only ever reads what it wrote itself, and every CTA streams long contiguous
// runs of each vector (measured faster than dealing 2048-element blocks round-robin: 14.3 vs 15.1 ms per config-2 solve).
struct Own
{
    int64_t n;
    int G, cta;
    int64_t c0, c1;
    __device__ __forceinline__ Own(int64_t n_, int G_, int cta_, int grain) : n(n_), G(G_), cta(cta_)
    {
        const int64_t units = (n + grain - 1) / grain;
        const int64_t K = units < G ? units : G;
        if (cta >= K) { c0 = c1 = 0; return; }
        c0 = ((units * cta) / K) * grain;
        c1 = ((units * (cta + 1)) / K) * grain;
        if (c1 > n) c1 = n;
    }
    // tiles of TE elements: number owned, first element and length of the t-th (the last one may be shorter)
    __device__ __forceinline__ int64_t ntiles(int TE) const { return (c1 - c0 + TE - 1) / TE; }
    __device__ __forceinline__ int64_t start(int64_t t, int TE) const { return c0 + t * TE; }
    __device__ __forceinline__ int len(int64_t t, int TE) const
    {
        const int64_t rest = c1 - start(t, TE);
        return rest <= 0 ? 0 : (rest < TE ? (int)rest : TE);
    }
};

// block-wide sums of NV per-thread values -> dst[k * G] (this CTA's slot of value k).  All threads call.
template <int NV> __device__ __forceinline__ void block_sums(const double (&acc)[NV], PShared& sh, double* dst, int G)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();   // sh.red may still be read from the previous use
#pragma unroll
    for (int k = 0; k < NV; k++)
    {
        const double w = warp_sum(acc[k]);
        if (lane == 0) sh.red[warp][k] = w;
    }
    __syncthreads();
    if (threadIdx.x < NV)
    {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kPWarps; w++) t += sh.red[w][threadIdx.x];
        dst[(size_t)threadIdx.x * G] = t;
    }
}

// ---- FIRST / TRIAL -------------------------------------------------------------------------------------------------------------
// MODE 0: FIRST (evaluate at x, write g and d = -g) ; MODE 1: TRIAL (x = xp + step*d, write x and g).  Operands stream through
// registers with 256-bit loads/stores (a shared-memory staged variant measured slower for this 1:1 read/write pass).
template <class T, class OBJ, int MODE>
__device__ __forceinline__ void p_trial(const OBJ& obj, const Own& own, const T* __restrict__ xp, const T* __restrict__ d, T step,
                                        T* __restrict__ x, T* __restrict__ g, T* __restrict__ dout, PShared& sh, double* dst, int G, int tune)
{
    T acc[4] = {T(0), T(0), T(0), T(0)};
    const int64_t n = own.n;
    const int64_t p1 = (own.c1 + 3) >> 2;
    const bool evict_first = (tune & 4) != 0;
    auto body = [&](int64_t q) {
        const int64_t i0 = q << 2;
        const int cnt = (n - i0 >= 4) ? 4 : int(n - i0);
        T xv[4], dv[4] = {T(0), T(0), T(0), T(0)}, gv[4];
        T xl = T(0), xr = T(0);
        if (MODE == 1)
        {
            const Pack<T> px = load4<T, Hint::Stream, true>(xp, i0, cnt), pd = load4<T, Hint::Stream, true>(d, i0, cnt);
#pragma unroll
            for (int k = 0; k < 4; k++) { dv[k] = pd.v[k]; xv[k] = px.v[k] + step * pd.v[k]; }
            if constexpr (OBJ::kHalo)
            {
                if (i0 > 0) xl = __ldcg(xp + i0 - 1) + step * __ldcg(d + i0 - 1);
                else if (obj.halo && obj.gofs > 0) xl = T(ldv(obj.halo + kHaloLeftA)) + step * T(ldv(obj.halo + kHaloLeftB));
                if (i0 + 4 < n) xr = __ldcg(xp + i0 + 4) + step * __ldcg(d + i0 + 4);
                else if (obj.halo && i0 + 4 == n && obj.gofs + n < obj.n_glob) xr = T(ldv(obj.halo + kHaloRightA)) + step * T(ldv(obj.halo + kHaloRightB));
            }
        }
        else
        {
            const Pack<T> px = load4<T, Hint::Stream, true>(x, i0, cnt);
#pragma unroll
            for (int k = 0; k < 4; k++) xv[k] = px.v[k];
            if constexpr (OBJ::kHalo)
            {
                if (i0 > 0) xl = __ldcg(x + i0 - 1);
                else if (obj.halo && obj.gofs > 0) xl = T(ldv(obj.halo + kHaloLeftA));
                if (i0 + 4 < n) xr = __ldcg(x + i0 + 4);
                else if (obj.halo && i0 + 4 == n && obj.gofs + n < obj.n_glob) xr = T(ldv(obj.halo + kHaloRightA));
            }
        }
        acc[0] += obj.eval(i0, cnt, xv, xl, xr, gv);
        Pack<T> pg, po;
#pragma unroll
        for (int k = 0; k < 4; k++)
        {
            acc[1] += gv[k] * dv[k];
            acc[2] += gv[k] * gv[k];
            acc[3] += (k < cnt) ? xv[k] * xv[k] : T(0);
            pg.v[k] = gv[k];
            po.v[k] = (MODE == 1) ? xv[k] : T(-1) * gv[k];
        }
        T* const out0 = (MODE == 1) ? x : dout;
        if (evict_first) { store4<T, Hint::Stream, true>(out0, i0, cnt, po); store4<T, Hint::Stream, true>(g, i0, cnt, pg); }
        else { store4<T, Hint::Plain, true>(out0, i0, cnt, po); store4<T, Hint::Plain, true>(g, i0, cnt, pg); }
    };
#pragma unroll 2
    for (int64_t q = (own.c0 >> 2) + threadIdx.x; q < p1; q += kPThreads) body(q);
    const double dacc[4] = {(double)acc[0], (double)acc[1], (double)acc[2], (double)acc[3]};
    block_sums<4>(dacc, sh, dst, G);
}

// Neighbour-coupled objectives (chained Rosenbrock, tridiagonal quadratic): the same pass with its inputs staged tile by tile through
// shared memory by bulk copies, every tile with one 16-byte granule of margin on either side, so that x_{i-1} and x_{i+1} of a pack
// come from the tile instead of from single-word L2 loads per pack (3x faster on config 3).  Only the two ends of the GLOBAL vector
// take their neighbours from the halo record (n-sharding) or as 0.

template <class T, class OBJ, int MODE>
__device__ __forceinline__ void p_trial_halo(const OBJ& obj, const Own& own, const T* __restrict__ xp, const T* __restrict__ d, T step,
                                             T* __restrict__ x, T* __restrict__ g, T* __restrict__ dout, T* tiles, PShared& sh, unsigned& phase_bits,
                                             double* dst, int G)
{
    constexpr int NIN = (MODE == 1) ? 2 : 1;                         // xp, d  /  x
    constexpr int DV = OBJ::kDataVectors;                            // the objective's data vectors are staged with them
    constexpr int NVEC = NIN + DV;
    constexpr int PAD = 16 / (int)sizeof(T);                         // margin in elements = one 16-byte granule
    constexpr int TS = kTrialTE + 2 * PAD;                           // staged elements per vector per tile
    constexpr int STAGES = trial_halo_stages((int)sizeof(T), NIN, DV);   // (kTrialTE: with the margins, six fp64 (xp, d) tiles fit the ring)
    static_assert(STAGES >= 1, "a trial tile must fit the staging ring");
    const int tid = threadIdx.x, lane = tid & 31;
    uint64_t* full_bar = sh.full_bar;
    const T* in0 = (MODE == 1) ? xp : x;
    const int64_t n = own.n;
    const int64_t ntl = own.ntiles(kTrialTE);
    const int64_t n_pad = (n + 31) & ~int64_t(31);                   // the vectors are allocated in whole 256-byte lines

    auto stage_tile = [&](int64_t t, int stage) {
        if (tid != 0) return;
        T* dstt = tiles + (size_t)stage * NVEC * TS;
        const int64_t e0 = own.start(t, kTrialTE);
        const int64_t lo = e0 >= PAD ? e0 - PAD : 0;                 // first element copied
        int64_t hi = e0 + ((own.len(t, kTrialTE) + 31) & ~31) + PAD; // one past the last element copied
        if (hi > n_pad) hi = n_pad;
        const unsigned bytes = (unsigned)(hi - lo) * (unsigned)sizeof(T);
        const int shift = (int)(lo - (e0 - PAD));                    // 0, or PAD at the very start of the vector
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&full_bar[stage], bytes * NVEC);
        tma_load_1d(dstt + shift, in0 + lo, bytes, &full_bar[stage]);
        if (MODE == 1) tma_load_1d(dstt + TS + shift, d + lo, bytes, &full_bar[stage]);
        if constexpr (DV == 2)
        {
            tma_load_1d(dstt + (size_t)NIN * TS + shift, obj.diag + lo, bytes, &full_bar[stage]);
            tma_load_1d(dstt + (size_t)(NIN + 1) * TS + shift, obj.rhs + lo, bytes, &full_bar[stage]);
        }
    };

    T acc[4] = {T(0), T(0), T(0), T(0)};
    __syncthreads();   // the tile area is free
    int64_t next_tile = 0;
    for (int s = 0; s < STAGES; s++, next_tile++)
        if (next_tile < ntl) stage_tile(next_tile, s);
    int stage = 0;
    for (int64_t t = 0; t < ntl; t++)
    {
        mbar_wait(&full_bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        const T* ta = tiles + (size_t)stage * NVEC * TS + PAD;       // element 0 of the tile
        const T* tb = ta + TS;
        const int64_t e0 = own.start(t, kTrialTE);
        const int len = own.len(t, kTrialTE);
        for (int off = tid * 4; off < len; off += kPThreads * 4)
        {
            const int64_t i0 = e0 + off;
            const int cnt = (len - off >= 4) ? 4 : (len - off);
            T xv[4], dv[4] = {T(0), T(0), T(0), T(0)}, gv[4];
            T xl = T(0), xr = T(0);
            const Pack<T> pa = lds_pack(ta + off, lane);
            if (MODE == 1)
            {
                const Pack<T> pb = lds_pack(tb + off, lane);
#pragma unroll
                for (int k = 0; k < 4; k++) { dv[k] = (k < cnt) ? pb.v[k] : T(0); xv[k] = (k < cnt) ? pa.v[k] + step * pb.v[k] : T(0); }
                if (i0 > 0) xl = ta[off - 1] + step * tb[off - 1];
                else if (obj.halo && obj.gofs > 0) xl = T(ldv(obj.halo + kHaloLeftA)) + step * T(ldv(obj.halo + kHaloLeftB));
                if (i0 + 4 < n) xr = ta[off + 4] + step * tb[off + 4];
                else if (obj.halo && i0 + 4 == n && obj.gofs + n < obj.n_glob) xr = T(ldv(obj.halo + kHaloRightA)) + step * T(ldv(obj.halo + kHaloRightB));
            }
            else
            {
#pragma unroll
                for (int k = 0; k < 4; k++) xv[k] = (k < cnt) ? pa.v[k] : T(0);
                if (i0 > 0) xl = ta[off - 1];
                else if (obj.halo && obj.gofs > 0) xl = T(ldv(obj.halo + kHaloLeftA));
                if (i0 + 4 < n) xr = ta[off + 4];
                else if (obj.halo && i0 + 4 == n && obj.gofs + n < obj.n_glob) xr = T(ldv(obj.halo + kHaloRightA));
            }
            if constexpr (DV == 2) acc[0] += obj.staged(ta + (size_t)NIN * TS, ta + (size_t)(NIN + 1) * TS, e0).eval(i0, cnt, xv, xl, xr, gv);
            else acc[0] += obj.eval(i0, cnt, xv, xl, xr, gv);
            Pack<T> pg, po;
#pragma unroll
            for (int k = 0; k < 4; k++)
            {
                acc[1] += gv[k] * dv[k];
                acc[2] += gv[k] * gv[k];
                acc[3] += (k < cnt) ? xv[k] * xv[k] : T(0);
                pg.v[k] = gv[k];
                po.v[k] = (MODE == 1) ? xv[k] : T(-1) * gv[k];
            }
            if (MODE == 1) store4<T, Hint::Plain, true>(x, i0, cnt, po);
            else store4<T, Hint::Plain, true>(dout, i0, cnt, po);
            store4<T, Hint::Plain, true>(g, i0, cnt, pg);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (next_tile < ntl) stage_tile(next_tile, stage);
        next_tile++;
        stage = (stage + 1 == STAGES) ? 0 : stage + 1;
    }
    const double dacc[4] = {(double)acc[0], (double)acc[1], (double)acc[2], (double)acc[3]};
    block_sums<4>(dacc, sh, dst, G);
}

// ---- RESTORE --------------------------------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ void p_restore(const Own& own, const T* __restrict__ xp, const T* __restrict__ gp, T* __restrict__ x, T* __restrict__ g)
{
    const int64_t n = own.n;
    const int64_t p1 = (own.c1 + 3) >> 2;
    for (int64_t q = (own.c0 >> 2) + threadIdx.x; q < p1; q += kPThreads)
    {
        const int64_t i0 = q << 2;
        const int cnt = (n - i0 >= 4) ? 4 : int(n - i0);
        store4<T, Hint::Plain, true>(x, i0, cnt, load4<T, Hint::Stream, true>(xp, i0, cnt));
        store4<T, Hint::Plain, true>(g, i0, cnt, load4<T, Hint::Stream, true>(gp, i0, cnt));
    }
}

// the `cnt` slots of the ring that end just below `end` (cyclically), as <= 2 ascending runs of slots; packed row of a slot
struct SlotRuns
{
    int a0, a1, b0, b1;   // run A = [a0, a1), run B = [b0, b1) (empty when b0 == b1); rows: A first, then B
    __device__ __forceinline__ SlotRuns(int end, int cnt, int M)
    {
        if (cnt <= end) { a0 = end - cnt; a1 = end; b0 = b1 = 0; }
        else { a0 = 0; a1 = end; b0 = M - (cnt - end); b1 = M; }
    }
    __device__ __forceinline__ int row_of(int slot) const { return (slot >= a0 && slot < a1) ? slot - a0 : (a1 - a0) + (slot - b0); }
};

// 16-byte units (2 doubles / 4 floats): the granularity of the staged passes
template <class T> struct alignas(16) Unit { T v[16 / sizeof(T)]; };
template <class T> __device__ __forceinline__ Unit<T> lds_unit(const T* p)
{
    Unit<T> u;
    *reinterpret_cast<float4*>(u.v) = *reinterpret_cast<const float4*>(p);
    return u;
}
template <class T> __device__ __forceinline__ void st_unit(T* base, int64_t i0, int cnt, const Unit<T>& u)
{
    constexpr int EPT = 16 / (int)sizeof(T);
    if (cnt >= EPT) { *reinterpret_cast<float4*>(base + i0) = *reinterpret_cast<const float4*>(u.v); return; }
#pragma unroll
    for (int k = 0; k < EPT; k++)
        if (k < cnt) base[i0 + k] = u.v[k];
}
template <class T> __device__ __forceinline__ void mask_unit(Unit<T>& u, int cnt)
{
#pragma unroll
    for (int k = 0; k < 16 / (int)sizeof(T); k++) u.v[k] = (k < cnt) ? u.v[k] : T(0);
}

// copies of one tile: `nrhs` right-hand vectors (sh.vecs[0..nrhs), round_up(len, 32) elements each) + the history runs of block
// `blk`; one lane per copy.  Returns nothing; the stage's barrier has been told the byte count.
template <class T>
__device__ __forceinline__ void stage_tiled(T* dstt, int TE, int nrhs, int64_t e0, int len, const PHist<T>& h, const SlotRuns& runs, PShared& sh,
                                            uint64_t* bar)
{
    const int tid = threadIdx.x;
    if (tid >= 32) return;
    const unsigned rbytes = (unsigned)((len + 31) & ~31) * (unsigned)sizeof(T);
    const unsigned abytes = (unsigned)(runs.a1 - runs.a0) * 2u * (unsigned)TE * (unsigned)sizeof(T);
    const unsigned bbytes = (unsigned)(runs.b1 - runs.b0) * 2u * (unsigned)TE * (unsigned)sizeof(T);
    if (tid == 0)
    {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy accesses of this stage before the copies that overwrite it
        mbar_expect_tx(bar, rbytes * (unsigned)nrhs + abytes + bbytes);
    }
    __syncwarp();
    const T* blk = h.H + (e0 >> h.bt_log) * h.bstride;
    if (tid < nrhs) tma_load_1d(dstt + (size_t)tid * TE, static_cast<const T*>(sh.vecs[tid]) + e0, rbytes, bar);
    else if (tid == nrhs && abytes) tma_load_1d(dstt + (size_t)nrhs * TE, blk + (size_t)runs.a0 * 2 * TE, abytes, bar);
    else if (tid == nrhs + 1 && bbytes) tma_load_1d(dstt + (size_t)(nrhs + 2 * (runs.a1 - runs.a0)) * TE, blk + (size_t)runs.b0 * 2 * TE, bbytes, bar);
}

// ---- DOTS -----------------------------------------------------------------------------------------------------------------------
// [S Y]'[v s_new y_new] over this CTA's chunk, one block (tile) at a time, everything staged by bulk copies.  FORM: the newest pair
// is formed on the fly from (x, xp, v = g, gp) -- s = x - xp, y = g - gp, identical in every warp that needs them -- takes part as
// column 0 and is written to ring slot `new_slot` by the warps that own column 0.  Column j (by age) belongs to warp group j, whose
// `split` warps share the tile's units.  PLAIN: s.v and y.v over the old history only.
template <class T> struct PDots
{
    int64_t n;
    PHist<T> h;
    int c;               // columns taking part (FORM: including the new pair)
    int end, cnt_old;    // the old columns: the cnt_old slots below `end`
    int new_slot, split, cols_per_round;
};

template <class T, int ROUNDS, bool FORM>
__device__ __forceinline__ void p_dots(const PDots<T>& a, const Own& own, T* tiles, PShared& sh, unsigned& phase_bits, double* dst, int G)
{
    constexpr int EPT = 16 / (int)sizeof(T);
    constexpr int NRHS = FORM ? 4 : 1;                           // staged right-hand vectors: g (, x, gp, xp)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int TE = a.h.BT();
    const int my_col = warp / a.split, my_part = warp % a.split;
    const int upp = (TE / EPT) / a.split;                        // units of a tile per warp of a column group
    const SlotRuns runs(a.end, a.cnt_old, a.h.M);
    const int nrows = NRHS + 2 * a.cnt_old;
    const int stages = dots_stages((int)sizeof(T), TE, FORM, a.cnt_old);   // >= 1: checked by the host before the launch
    const int64_t ntl = own.ntiles(TE);
    uint64_t* full_bar = sh.full_bar;

    T acc[ROUNDS][kGramVals];
#pragma unroll
    for (int r = 0; r < ROUNDS; r++)
#pragma unroll
        for (int k = 0; k < kGramVals; k++) acc[r][k] = T(0);

    __syncthreads();   // sh.vecs / sh.slots are in place and the staging ring is free
    int64_t next_tile = 0;
    for (int s = 0; s < stages; s++, next_tile++)
        if (next_tile < ntl) stage_tiled<T>(tiles + (size_t)s * nrows * TE, TE, NRHS, own.start(next_tile, TE), own.len(next_tile, TE), a.h, runs, sh, &full_bar[s]);
    int stage = 0;
    for (int64_t t = 0; t < ntl; t++)
    {
        mbar_wait(&full_bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        const T* base = tiles + (size_t)stage * nrows * TE;
        const T* hist = base + (size_t)NRHS * TE;
        const int64_t e0 = own.start(t, TE);
        const int len = own.len(t, TE);
#pragma unroll
        for (int r = 0; r < ROUNDS; r++)
        {
            const int j = r * a.cols_per_round + my_col;
            if (my_col < a.cols_per_round && j < a.c)
            {
                const bool is_new = FORM && j == 0;
                const T* srow = hist + (size_t)2 * (is_new ? 0 : sh.slots[j]) * TE;     // sh.slots[j]: packed row of the column of age j
                const T* yrow = srow + TE;
                T* s_new = a.h.s_at(a.new_slot < 0 ? 0 : a.new_slot, e0);
                for (int u = my_part * upp + lane; u < (my_part + 1) * upp; u += 32)
                {
                    const int off = u * EPT;
                    const int cnt = len - off;
                    if (cnt <= 0) break;
                    Unit<T> ug = lds_unit<T>(base + off), us, uy, usn, uyn;
                    if constexpr (FORM)
                    {
                        const Unit<T> ux = lds_unit<T>(base + TE + off), ugp = lds_unit<T>(base + 2 * TE + off), uxp = lds_unit<T>(base + 3 * TE + off);
#pragma unroll
                        for (int k = 0; k < EPT; k++) { usn.v[k] = ux.v[k] - uxp.v[k]; uyn.v[k] = ug.v[k] - ugp.v[k]; }
                        if (cnt < EPT) { mask_unit(usn, cnt); mask_unit(uyn, cnt); }
                    }
                    bool loaded = false;
                    if constexpr (FORM)
                    {
                        if (is_new)
                        {
                            us = usn; uy = uyn;
                            st_unit<T>(s_new, off, cnt, usn);
                            st_unit<T>(s_new + TE, off, cnt, uyn);
                            loaded = true;
                        }
                    }
                    if (!loaded) { us = lds_unit<T>(srow + off); uy = lds_unit<T>(yrow + off); }
                    if (cnt < EPT) { mask_unit(ug, cnt); mask_unit(us, cnt); mask_unit(uy, cnt); }
#pragma unroll
                    for (int k = 0; k < EPT; k++)
                    {
                        acc[r][0] += us.v[k] * ug.v[k];
                        acc[r][1] += uy.v[k] * ug.v[k];
                    }
                    if constexpr (FORM)
                    {
#pragma unroll
                        for (int k = 0; k < EPT; k++)
                        {
                            acc[r][2] += us.v[k] * uyn.v[k];
                            acc[r][3] += uy.v[k] * uyn.v[k];
                            acc[r][4] += uy.v[k] * usn.v[k];
                            acc[r][5] += us.v[k] * usn.v[k];
                        }
                    }
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (next_tile < ntl) stage_tiled<T>(tiles + (size_t)stage * nrows * TE, TE, NRHS, own.start(next_tile, TE), own.len(next_tile, TE), a.h, runs, sh, &full_bar[stage]);
        next_tile++;
        stage = (stage + 1 == stages) ? 0 : stage + 1;
    }

    // block reduction: lanes -> warp, then the `split` warps of a column; value (j, k) -> dst[(j*6 + k) * G]
#pragma unroll
    for (int r = 0; r < ROUNDS; r++)
#pragma unroll
        for (int k = 0; k < kGramVals; k++)
        {
            const double w = warp_sum((double)acc[r][k]);
            if (lane == 0) sh.red[warp][r * kGramVals + k] = w;
        }
    __syncthreads();
    const int nvals = a.c * kGramVals;
    for (int idx = tid; idx < nvals; idx += kPThreads)
    {
        const int j = idx / kGramVals, k = idx % kGramVals;
        const int r = j / a.cols_per_round, col = j % a.cols_per_round;
        double t = 0.0;
        for (int p = 0; p < a.split; p++) t += sh.red[col * a.split + p][r * kGramVals + k];
        dst[(size_t)idx * G] = t;
    }
}

// how the warps of the dots pass share the columns: `split` warps per column pair, cols_per_round column pairs at a time
__device__ __forceinline__ void dots_geometry(int c, int units, int& split, int& cols_per_round)
{
    split = 8;
    while (split > 1 && (c * split > kGramMaxWarps || units / split < 32)) split >>= 1;
    cols_per_round = c < kGramMaxWarps / split ? c : kGramMaxWarps / split;
}

// ---- COMBINE (+ first trial) ---------------------------------------------------------------------------------------------------
// d = cv*v + sum_j cy_j*y_j + cs_j*s_j ; FUSE: x1 = xc + d, g1 = grad f(x1) written to (x1_out, g1_out) and the four trial sums.
// Staged rows of a tile: v, (xc,) then the history block's live slots; sh.slots[j] = packed row of the pair of age j.  A thread owns
// one 16-byte unit of the tile and adds the terms in the order the recursion would (y newest -> oldest, then s oldest -> newest), with
// the operand loads of 8 columns in flight before their multiply-adds retire (the pass is bound by shared-memory latency otherwise).
// HALO (neighbour-coupled objectives, one GPU): x1 goes back into the staged x row, two spare warps form d and x1 of the element on
// either side of the tile from global memory with the very arithmetic of the tile that owns it, and after a barrier the objective
// takes x1_{i-1}, x1_{i+1} from shared memory.
// `between` (all threads) runs after the bulk copies of the first tiles have been issued and before anything reads the coefficients:
// the coefficient recursion overlaps the latency of those copies when it has a scratch area of its own.
template <class T, class OBJ, bool FUSE, bool HALO, class Between>
__device__ __forceinline__ void p_combine(const OBJ& obj, const Own& own, const PHist<T>& h, int c, int end, T* tiles, T* __restrict__ res,
                                          T* __restrict__ x1_out, T* __restrict__ g1_out, PShared& sh, unsigned& phase_bits, double* dst, int G,
                                          Between between)
{
    constexpr int EPT = 16 / (int)sizeof(T);
    constexpr int DV = HALO ? OBJ::kDataVectors : 0;              // HALO: the objective's data vectors ride in the stage as well
    constexpr int NRHS = (FUSE ? 2 : 1) + DV;                     // v (, xc) (, data0, data1)
    constexpr int PAD = EPT;                                      // HALO: room for x1 of the neighbouring element on either side of the x row
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int TE = h.BT();
    const SlotRuns runs(end, c, h.M);
    const int nrows = NRHS + 2 * c;
    const size_t stage_elems = (size_t)nrows * TE + (HALO ? 2 * PAD : 0);
    const int stages = combine_stages((int)sizeof(T), TE, c, FUSE, HALO, DV);   // >= 1: checked by the host before the launch
    const int64_t n = own.n;
    const int64_t ntl = own.ntiles(TE);
    const T* s_coef = reinterpret_cast<const T*>(sh.coef);
    uint64_t* full_bar = sh.full_bar;
    // HALO: the x row is staged one granule into the stage (row 1 starts at TE + PAD), everything after it shifts by 2*PAD
    auto stage_one = [&](int64_t t, int s) {
        T* dstt = tiles + (size_t)s * stage_elems;
        if (!HALO) { stage_tiled<T>(dstt, TE, NRHS, own.start(t, TE), own.len(t, TE), h, runs, sh, &full_bar[s]); return; }
        if (tid >= 32) return;
        const int64_t e0 = own.start(t, TE);
        const int len = own.len(t, TE);
        const unsigned rbytes = (unsigned)((len + 31) & ~31) * (unsigned)sizeof(T);
        const unsigned abytes = (unsigned)(runs.a1 - runs.a0) * 2u * (unsigned)TE * (unsigned)sizeof(T);
        const unsigned bbytes = (unsigned)(runs.b1 - runs.b0) * 2u * (unsigned)TE * (unsigned)sizeof(T);
        if (tid == 0)
        {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(&full_bar[s], rbytes * (unsigned)NRHS + abytes + bbytes);
        }
        __syncwarp();
        const T* blk = h.H + (e0 >> h.bt_log) * h.bstride;
        T* hist = dstt + (size_t)NRHS * TE + 2 * PAD;
        if (tid == 0) tma_load_1d(dstt, static_cast<const T*>(sh.vecs[0]) + e0, rbytes, &full_bar[s]);
        else if (tid == 1) tma_load_1d(dstt + TE + PAD, static_cast<const T*>(sh.vecs[1]) + e0, rbytes, &full_bar[s]);
        else if (tid == 2 && abytes) tma_load_1d(hist, blk + (size_t)runs.a0 * 2 * TE, abytes, &full_bar[s]);
        else if (tid == 3 && bbytes) tma_load_1d(hist + (size_t)2 * (runs.a1 - runs.a0) * TE, blk + (size_t)runs.b0 * 2 * TE, bbytes, &full_bar[s]);
        else if (tid >= 4 && tid < 4 + DV) tma_load_1d(dstt + (size_t)(tid - 2) * TE + 2 * PAD, static_cast<const T*>(sh.vecs[tid - 2]) + e0, rbytes, &full_bar[s]);
    };

    T acc[5] = {T(0), T(0), T(0), T(0), T(0)};
    T pre[5] = {T(0), T(0), T(0), T(0), T(0)};   // HALO, right-margin warp: operands of the element after the current tile
    __syncthreads();   // sh.vecs / sh.slots are in place and the staging ring is free
    int64_t next_tile = 0;
    for (int s = 0; s < stages; s++, next_tile++)
        if (next_tile < ntl) stage_one(next_tile, s);
    between();         // (ends with a barrier: sh.coef is in place)
    const T cv = s_coef[0];
    int stage = 0;
    for (int64_t t = 0; t < ntl; t++)
    {
        mbar_wait(&full_bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        T* base = tiles + (size_t)stage * stage_elems;                          // row 0: v
        T* xrow = base + TE + (HALO ? PAD : 0);                                   // row 1: xc (FUSE)
        const T* hist = base + (size_t)NRHS * TE + (HALO ? 2 * PAD : 0);
        const int len = own.len(t, TE);
        const int64_t e0 = own.start(t, TE);
        // d of one unit: the arithmetic every owner of an element uses
        auto direction = [&](int off, T (&r)[EPT], Unit<T>& uv) {
            uv = lds_unit<T>(base + off);
#pragma unroll
            for (int k = 0; k < EPT; k++) r[k] = cv * uv.v[k];
#pragma unroll 8
            for (int j = 0; j < c; j++)                        // y terms newest -> oldest
            {
                const Unit<T> uy = lds_unit<T>(hist + ((size_t)2 * sh.slots[j] + 1) * TE + off);
                const T cy = s_coef[1 + j];
#pragma unroll
                for (int k = 0; k < EPT; k++) r[k] += cy * uy.v[k];
            }
#pragma unroll 8
            for (int j = c - 1; j >= 0; j--)                   // s terms oldest -> newest
            {
                const Unit<T> us = lds_unit<T>(hist + (size_t)2 * sh.slots[j] * TE + off);
                const T cs = s_coef[1 + c + j];
#pragma unroll
                for (int k = 0; k < EPT; k++) r[k] += cs * us.v[k];
            }
        };
        if constexpr (!HALO)
        {
            for (int off = tid * EPT; off < len; off += kPThreads * EPT)
            {
                const int cnt = (len - off >= EPT) ? EPT : (len - off);
                T r[EPT];
                Unit<T> uv;
                direction(off, r, uv);
                Unit<T> out;
#pragma unroll
                for (int k = 0; k < EPT; k++)
                {
                    out.v[k] = r[k];
                    acc[0] += (k < cnt) ? uv.v[k] * r[k] : T(0);
                }
                const int64_t i0 = e0 + off;
                st_unit<T>(res, i0, cnt, out);
                if constexpr (FUSE)
                {
                    const Unit<T> ux = lds_unit<T>(xrow + off);
                    T xv[4] = {T(0), T(0), T(0), T(0)}, gv[4];
#pragma unroll
                    for (int k = 0; k < EPT; k++) xv[k] = (k < cnt) ? ux.v[k] + T(1) * r[k] : T(0);
                    acc[1] += obj.eval(i0, cnt, xv, T(0), T(0), gv);
                    Unit<T> ug, uo;
#pragma unroll
                    for (int k = 0; k < EPT; k++)
                    {
                        acc[2] += (k < cnt) ? gv[k] * r[k] : T(0);
                        acc[3] += (k < cnt) ? gv[k] * gv[k] : T(0);
                        acc[4] += (k < cnt) ? xv[k] * xv[k] : T(0);
                        ug.v[k] = gv[k];
                        uo.v[k] = xv[k];
                    }
                    if (x1_out != nullptr)
                    {
                        st_unit<T>(x1_out, i0, cnt, uo);
                        st_unit<T>(g1_out, i0, cnt, ug);
                    }
                }
            }
        }
        else
        {
            // ---- phase 1: d and x1 of the tile's units (one per thread: a tile has at most 512 units) ----
            const int off = tid * EPT;
            const bool mine = off < len;
            const int64_t i0 = e0 + off;
            const int cnt = mine ? ((len - off >= EPT) ? EPT : (len - off)) : 0;
            T r[EPT];
#pragma unroll
            for (int k = 0; k < EPT; k++) r[k] = T(0);
            if (mine)
            {
                Unit<T> uv;
                direction(off, r, uv);
                Unit<T> out;
#pragma unroll
                for (int k = 0; k < EPT; k++)
                {
                    out.v[k] = r[k];
                    acc[0] += (k < cnt) ? uv.v[k] * r[k] : T(0);
                }
                st_unit<T>(res, i0, cnt, out);
                const Unit<T> ux = lds_unit<T>(xrow + off);
                Unit<T> u1;
#pragma unroll
                for (int k = 0; k < EPT; k++) u1.v[k] = (k < cnt) ? ux.v[k] + T(1) * r[k] : T(0);
                *reinterpret_cast<float4*>(xrow + off) = *reinterpret_cast<const float4*>(u1.v);
            }
            // the element on either side of the tile.  Left: the previous tile of this chunk left its last x1 in sh.carry (only a chunk's
            // first tile asks global memory).  Right: warp kPWarps-1 holds the operands of the element after the tile (fetched through
            // L2 one tile ahead: other CTAs wrote them in earlier rounds), multiplies them by their coefficients in parallel and lane 0
            // adds the products in the owner's order -- the owner's arithmetic, bit for bit.
            if (warp == kPWarps - 2 && lane == 0 && t > 0) xrow[-1] = *reinterpret_cast<const T*>(&sh.carry[(t - 1) & 1]);
            if (warp >= kPWarps - 2 && (warp == kPWarps - 1 || t == 0))
            {
                const bool left = warp == kPWarps - 2;
                const int64_t im = left ? e0 - 1 : e0 + len;
                T* scratch = reinterpret_cast<T*>(sh.margin[left ? 0 : 1]);
                auto fetch = [&](int64_t i, T (&dstv)[5]) {
#pragma unroll
                    for (int w = 0; w < 5; w++)
                    {
                        const int q = lane + 32 * w;
                        T val = T(0);
                        if (i >= 0 && i < n && q < 2 * c + 2)
                        {
                            if (q == 0) val = __ldcg(static_cast<const T*>(sh.vecs[0]) + i);
                            else if (q == 1) val = __ldcg(static_cast<const T*>(sh.vecs[1]) + i);
                            else if (q < 2 + c) val = __ldcg(h.y_at(sh.slotid[q - 2], i));          // y of age q-2
                            else val = __ldcg(h.s_at(sh.slotid[q - 2 - c], i));                      // s of age q-2-c
                        }
                        dstv[w] = val;
                    }
                };
                if (left || t == 0) fetch(im, pre);        // (the right-margin warp fetched this tile's element during the previous tile)
                if (im >= 0 && im < n)
                {
#pragma unroll
                    for (int w = 0; w < 5; w++)
                    {
                        const int q = lane + 32 * w;
                        if (q < 2 * c + 2)
                            scratch[q] = (q == 0) ? cv * pre[w] : (q == 1) ? pre[w] : (q < 2 + c) ? s_coef[1 + (q - 2)] * pre[w] : s_coef[1 + c + (q - 2 - c)] * pre[w];
                    }
                    __syncwarp();
                    if (lane == 0)
                    {
                        T rm = scratch[0];
                        for (int j = 0; j < c; j++) rm += scratch[2 + j];
                        for (int j = c - 1; j >= 0; j--) rm += scratch[2 + c + j];
                        xrow[left ? -1 : len] = scratch[1] + T(1) * rm;
                    }
                }
                if (!left && t + 1 < ntl) fetch(own.start(t + 1, TE) + own.len(t + 1, TE), pre);   // next tile's right neighbour, in flight meanwhile
            }
            if (mine && off + EPT >= len) *reinterpret_cast<T*>(&sh.carry[t & 1]) = xrow[len - 1];   // (this thread wrote it above; two slots: the next tile reads the other one)
            __syncthreads();
            // ---- phase 2: the objective at x1 with its neighbours from shared memory ----
            if (mine)
            {
                T xv[4] = {T(0), T(0), T(0), T(0)}, gv[4];
                const Unit<T> u1 = lds_unit<T>(xrow + off);
#pragma unroll
                for (int k = 0; k < EPT; k++) xv[k] = u1.v[k];
                const T xl = (i0 > 0) ? xrow[off - 1] : T(0);
                const T right = (i0 + EPT < n) ? xrow[off + EPT] : T(0);
                T xr = T(0);
                if (EPT < 4) xv[EPT < 4 ? EPT : 3] = right; else xr = right;
                if constexpr (DV == 2) acc[1] += obj.staged(base + 2 * (size_t)TE + 2 * PAD, base + 3 * (size_t)TE + 2 * PAD, e0).eval(i0, cnt, xv, xl, xr, gv);
                else acc[1] += obj.eval(i0, cnt, xv, xl, xr, gv);
                Unit<T> ug, uo;
#pragma unroll
                for (int k = 0; k < EPT; k++)
                {
                    acc[2] += (k < cnt) ? gv[k] * r[k] : T(0);
                    acc[3] += (k < cnt) ? gv[k] * gv[k] : T(0);
                    acc[4] += (k < cnt) ? xv[k] * xv[k] : T(0);
                    ug.v[k] = gv[k];
                    uo.v[k] = xv[k];
                }
                if (x1_out != nullptr)
                {
                    st_unit<T>(x1_out, i0, cnt, uo);
                    st_unit<T>(g1_out, i0, cnt, ug);
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (next_tile < ntl) stage_one(next_tile, stage);
        next_tile++;
        stage = (stage + 1 == stages) ? 0 : stage + 1;
    }
    if (FUSE)
    {
        const double dacc[5] = {(double)acc[0], (double)acc[1], (double)acc[2], (double)acc[3], (double)acc[4]};
        block_sums<5>(dacc, sh, dst, G);
    }
    else
    {
        const double dacc[1] = {(double)acc[0]};
        block_sums<1>(dacc, sh, dst, G);
    }
}

// ---- waits with a watchdog ----------------------------------------------------------------------------------------------------
constexpr long long kPWaitCycles = 6000000000ll;   // default watchdog budget, ~3 s at 2 GHz: far beyond any legitimate wait (LBFGS_B200_WATCHDOG_SCALE multiplies it, e.g. under compute-sanitizer)

__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned* p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// ---- the leader's work between two rounds ------------------------------------------------------------------------------------
template <class T> __device__ __forceinline__ void record_eval(PState<T>* st, T fx)
{
    if (st->trace && st->nfev < st->trace_cap) st->trace[st->nfev] = (double)fx;
    st->nfev++;
}
template <class T> __device__ __forceinline__ void finish(PState<T>* st, int niter, int status = 0)
{
    st->finished = 1;
    st->niter = niter;
    if (status) st->status = status;
    st->op = POP_IDLE;
}

// LBFGS.h:137-154 after an accepted / best-so-far point: returns true when the solve is over
template <class T> __device__ __forceinline__ bool converged_after_search(PState<T>* st)
{
    const int k = st->k;
    st->gnorm = sqrt(st->gg);
    if (st->gnorm <= st->epsilon || st->gnorm <= st->epsilon_rel * sqrt(st->xx)) { finish(st, k); return true; }
    if (st->past > 0)
    {
        const T fxd = st->fx_hist[k % st->past];
        const T fx = st->fx;
        const T afx = fx < T(0) ? -fx : fx, afxd = fxd < T(0) ? -fxd : fxd;
        T big = afx < afxd ? afxd : afx;       // std::max(abs(fx), abs(fxd))
        big = big < T(1) ? T(1) : big;         // std::max(., 1)
        const T diff = (fxd - fx) < T(0) ? -(fxd - fx) : (fxd - fx);
        if (k >= st->past && diff <= st->delta * big) { finish(st, k); return true; }
        st->fx_hist[k % st->past] = fx;
    }
    if (st->max_iterations != 0 && k >= st->max_iterations) { finish(st, k); return true; }
    return false;
}

// after a search has produced its point in (x, g): convergence tests, then on to the pair-forming dots
template <class T> __device__ __forceinline__ void after_search(PState<T>* st)
{
    if (converged_after_search(st)) return;
    st->op = POP_DOTS_FORM;
    st->c_round = st->ncorr < st->m ? st->ncorr + 1 : st->m;
}

// the trial at ls_step_ref(st) has been evaluated: {fx, dg, gg, xx}.  Sets the next op.  `is_virtual`: the fused first trial
// whose x1 / g1 were not stored (they are x = xp + 1*d and its gradient: a MATERIALIZE pass recomputes them bit for bit if the
// search turns out to need them).  Adaptive policy (off by default, LBFGS_B200_VIRTUAL_FIRST_TRIAL=1): store the next first trial
// iff this one was accepted.  Measured on config 2 (3 of 21 first trials accepted): 0.25 ms saved in the combination passes,
// 0.20 ms spent on the three MATERIALIZE rounds -- a wash at n = 1e7 and a loss at n = 1e6, hence off.
template <class T> __device__ __forceinline__ void digest_trial(PState<T>* st, T fx, T dg, T gg, T xx, bool is_first, bool is_virtual)
{
    record_eval(st, fx);
    bool keep = false;
    const T step_tried = ls_step_ref(st);
    const int rc = ls_advance(st, fx, dg, keep);
    if (is_first && st->adaptive_first_store) st->first_store = (rc == LBFGSpp::LSC_ACCEPT) ? 1 : 0;
    if (keep)
    {
        if (is_virtual) { st->lo_virtual = 1; st->lo_step = step_tried; }
        else
        {
            dswap(st->x, st->x_lo);
            dswap(st->g, st->g_lo);
            st->lo_virtual = 0;
        }
        st->have_lo = 1;
        st->lo_gg = gg;
        st->lo_xx = xx;
    }
    if (rc == LBFGSpp::LSC_EVALUATE) { st->op = POP_TRIAL; st->step = ls_step_ref(st); return; }
    if (rc == LBFGSpp::LSC_ACCEPT)
    {
        st->fx = fx; st->dg = dg; st->gg = gg; st->xx = xx;
        if (is_virtual) { st->op = POP_MATERIALIZE; st->step = step_tried; st->after_materialize = 1; return; }
    }
    else if (rc == LBFGSpp::LSC_TAKE_BEST)
    {
        T bf, bd;
        ls_best(st, bf, bd);
        st->fx = bf;
        st->dg = bd;
        if (st->have_lo)
        {
            st->gg = st->lo_gg;
            st->xx = st->lo_xx;
            if (st->lo_virtual) { st->op = POP_MATERIALIZE; st->step = st->lo_step; st->after_materialize = 2; return; }
            dswap(st->x, st->x_lo);
            dswap(st->g, st->g_lo);
        }
        else
        {
            st->gg = st->start_gg;
            st->xx = st->start_xx;
            st->op = POP_RESTORE;   // no trial ever improved on the start point: copy xp/gp back, then carry on
            return;
        }
    }
    else { finish(st, st->k, rc); return; }
    after_search(st);
}

// top of an iteration (LBFGS.h:121-127): the search is armed, the current point becomes the previous one
template <class T> __device__ __forceinline__ bool begin_search(PState<T>* st, T step)
{
    // the search validates its inputs before anything moves (the reference throws before touching x): on failure x stays the
    // current point
    const int rc = ls_init(st, st->fx, st->dg, step, st->max_step);
    if (rc != 0) { finish(st, st->k, rc); return false; }
    dswap(st->xp, st->x);
    dswap(st->gp, st->g);
    st->have_lo = 0;
    st->lo_virtual = 0;
    st->start_gg = st->gg;
    st->start_xx = st->xx;
    st->op = POP_TRIAL;
    st->step = ls_step_ref(st);
    return true;
}

template <class T> __device__ void advance_problem(PState<T>* st, const double* vals)
{
    st->rounds++;
    switch (st->op)
    {
    case POP_FIRST:
    {
        const T fx = (T)vals[0], gg = (T)vals[2], xx = (T)vals[3];
        st->nfev = 0;
        record_eval(st, fx);
        st->fx = fx; st->gg = gg; st->xx = xx;
        st->k = 1;
        if (st->past > 0) st->fx_hist[0] = fx;
        st->gnorm = sqrt(gg);
        if (st->gnorm <= st->epsilon || st->gnorm <= st->epsilon_rel * sqrt(xx)) { finish(st, 1); return; }
        st->dg = -gg;                       // grad . (-grad)
        begin_search(st, T(1) / st->gnorm); // LBFGS.h:108
        return;
    }
    case POP_TRIAL:
        digest_trial(st, (T)vals[0], (T)vals[1], (T)vals[2], (T)vals[3], false, false);
        return;
    case POP_RESTORE:
    case POP_MATERIALIZE:       // (x, g) now hold the search's point; its sums were digested before
        after_search(st);
        return;
    case POP_DOTS_FORM:
    {
        // curvature gate on the pair's own dots (age-0 column: [2] = s'y, [3] = y'y), LBFGS.h:161; commit = BFGSMat.h:89-97
        const T sy = (T)vals[2], yy = (T)vals[3];
        if (sy > st->eps_gate * yy)
        {
            st->ys[st->head] = sy;
            *st->theta = yy / sy;
            st->pending = st->head;
            st->head = (st->head + 1) % st->M;
            st->ncorr = st->c_round;
            st->op = st->fuse_first_trial ? POP_COMBINE_TRIAL : POP_COMBINE;
        }
        else if (st->ncorr > 0) { st->op = POP_DOTS_PLAIN; st->c_round = st->ncorr; }
        else { st->op = st->fuse_first_trial ? POP_COMBINE_TRIAL : POP_COMBINE; st->c_round = 0; }
        return;
    }
    case POP_DOTS_PLAIN:
        st->op = st->fuse_first_trial ? POP_COMBINE_TRIAL : POP_COMBINE;
        return;
    case POP_COMBINE:
    case POP_COMBINE_TRIAL:
    {
        const bool fused = st->op == POP_COMBINE_TRIAL;
        const bool stored = st->first_store != 0;      // what this pass was told (the policy flag changes in digest_trial)
        if (st->pending >= 0) { st->gram_cur = 1 - st->gram_cur; st->pending = -1; }
        st->dg = (T)vals[0];                // LBFGS.h:123 for the next pass
        st->k += 1;
        if (!begin_search(st, T(1))) return;   // LBFGS.h:168
        // the pass already evaluated x + 1*d into the buffers that the rotation just made (x, g)
        if (fused && ls_step_ref(st) == T(1)) digest_trial(st, (T)vals[1], (T)vals[2], (T)vals[3], (T)vals[4], true, !stored);
        return;
    }
    default: return;
    }
}

// n-words a pass has to move (reads + writes of whole vectors): the roofline numerator of the persistent kernel
__device__ __forceinline__ double words_of(int op, int c, int data_vectors, int store_first)
{
    switch (op)
    {
    case POP_FIRST: return 3.0 + data_vectors;              // R x ; W g, d
    case POP_TRIAL: case POP_MATERIALIZE: return 4.0 + data_vectors;   // R xp, d ; W x, g
    case POP_RESTORE: return 4.0;                           // R xp, gp ; W x, g
    case POP_DOTS_FORM: return 2.0 * c + 4.0;               // R x, xp, g, gp, 2(c-1) columns ; W s, y
    case POP_DOTS_PLAIN: return 2.0 * c + 1.0;              // R g, 2c columns
    case POP_COMBINE: return 2.0 * c + 2.0;                 // R g, 2c columns ; W d
    case POP_COMBINE_TRIAL: return 2.0 * c + 3.0 + (store_first ? 2.0 : 0.0) + data_vectors;   // R g, x, 2c columns ; W d (, x1, g1)
    default: return 0.0;
    }
}

template <class T> __device__ __forceinline__ int nvals_of(const PState<T>* st)
{
    switch (st->op)
    {
    case POP_FIRST: case POP_TRIAL: case POP_MATERIALIZE: return 4;
    case POP_DOTS_FORM: case POP_DOTS_PLAIN: return st->c_round * kGramVals;
    case POP_COMBINE: return 1;
    case POP_COMBINE_TRIAL: return 5;
    default: return 0;
    }
}

// Fixed-order sums of the CTAs' partials of every running problem into raw[], (optional) cross-rank exchange, scalar logic,
// publication of the next round's descriptors.  Called by all threads of CTA 0 once every CTA has arrived.  Returns (in every
// thread) the number of problems still running.
template <class T, bool HALO>
__device__ int leader_round(const PArgs<T>& a, int G, PShared& sh, PState<T>* cache)
{
    const int tid = threadIdx.x;
    // the leader's working copies: the first kPCache problems live in shared memory for the duration of the kernel
    auto state_of = [&](int b) -> PState<T>* { return b < kPCache ? cache + b : a.probs + b; };
    // 1. local sums: 16 threads per value (CTAs s, s+16, ... then a fixed shuffle tree), 48 values per sweep
    for (int b = 0; b < a.B; b++)
    {
        PState<T>* st = state_of(b);
        const int op = st->op;           // the pass this problem just ran (advance_problem below moves it on)
        if (op == POP_IDLE) continue;
        const int nv = nvals_of(st);
        const double* part = a.partials + (size_t)b * a.pstride * G;
        for (int v0 = 0; v0 < nv; v0 += kPThreads / 16)
        {
            const int v = v0 + tid / 16, sub = tid & 15;
            double t = 0.0;
            if (v < nv)
                for (int cta = sub; cta < G; cta += 16) t += __ldcg(part + (size_t)v * G + cta);
            t += __shfl_xor_sync(0xffffffffu, t, 8);
            t += __shfl_xor_sync(0xffffffffu, t, 4);
            t += __shfl_xor_sync(0xffffffffu, t, 2);
            t += __shfl_xor_sync(0xffffffffu, t, 1);
            if (v < nv && sub == 0) st->raw[v] = t;
        }
    }
    __syncthreads();
    // 2. n sharded over ranks: ONE exchange for all running problems (sums in rank order: identical bits on every rank)
    if (a.xc != nullptr)
    {
        const long long t_x0 = clock64();
        const XComm* xc = a.xc;
        const int me = xc->rank, R = xc->nranks;
        const unsigned long long epoch = a.ctl->epoch + 1ull;
        const int slot = (int)(epoch % kXRing);
        const unsigned tag = (unsigned)epoch;
        auto give_up = [&]() {
            if (clock64() - t_x0 > 4 * a.wait_cycles || ldv(&a.ctl->abort)) { a.ctl->abort = 1; return true; }
            return false;
        };
        // payload layout: problem after problem, nv sums then (HALO) 4 gathered boundary values.  Every value goes to every rank
        // (this one included) as two tagged 8-byte words: the receiver needs no flag and the sender no fence.
        int ofs = 0;
        for (int b = 0; b < a.B; b++)
        {
            PState<T>* st = state_of(b);
            const int op = st->op;
            if (op == POP_IDLE) continue;
            const int nv = nvals_of(st);
            for (int r = tid; r < R * nv; r += kPThreads)
                ll_push(xc->inbox[r / nv]->ll[slot][me][ofs + r % nv], st->raw[r % nv], tag);
            ofs += nv;
            if (HALO)
            {
                // boundary coordinates for the neighbours' next evaluations: the next search starts from the current x along drt
                if (tid < 4 * R)
                {
                    const int k = tid & 3;
                    const T* src = (k & 1) ? st->drt : st->x;
                    const double val = (double)__ldcg(src + ((k & 2) ? a.n - 1 : 0));
                    ll_push(xc->inbox[tid >> 2]->ll[slot][me][ofs + k], val, tag);
                }
                ofs += 4;
            }
        }
        __syncthreads();   // (raw[] is about to be overwritten with the global sums)
        ofs = 0;
        for (int b = 0; b < a.B; b++)
        {
            PState<T>* st = state_of(b);
            const int op = st->op;
            if (op == POP_IDLE) continue;
            const int nv = nvals_of(st);
            for (int k = tid; k < nv; k += kPThreads)
            {
                double t = 0.0;
                for (int r = 0; r < R; r++)           // rank order: identical bits on every rank
                {
                    double v = 0.0;
                    ll_pull(xc->inbox[me]->ll[slot][r][ofs + k], tag, v, give_up);
                    t += v;
                }
                st->raw[k] = t;
            }
            ofs += nv;
            if (HALO)
            {
                if ((op == POP_FIRST || op == POP_COMBINE || op == POP_COMBINE_TRIAL) && tid < 8)
                {
                    const int side = tid >> 2, k = tid & 3;       // side 0: left neighbour, 1: right neighbour
                    const int nb = side == 0 ? me - 1 : me + 1;
                    double v = 0.0;
                    if (nb >= 0 && nb < R) ll_pull(xc->inbox[me]->ll[slot][nb][ofs + k], tag, v, give_up);
                    st->halo[4 + 4 * side + k] = v;
                }
                ofs += 4;
            }
        }
        __syncthreads();
        if (tid == 0) { a.ctl->epoch = epoch; a.ctl->cyc_exchange += clock64() - t_x0; }
    }
    // 3. scalar logic, one thread per problem; the outcome goes into the problem's round descriptor
    int still = 0;
    for (int b0 = 0; b0 < a.B; b0 += kPThreads)
    {
        const int b = b0 + tid;
        int running = 0;
        if (b < a.B && state_of(b)->op != POP_IDLE)
        {
            PState<T>* st = state_of(b);
            advance_problem(st, st->raw);
            PRound<T>* rd = a.rounds + b;
            rd->x = st->x; rd->xp = st->xp; rd->g = st->g; rd->gp = st->gp; rd->drt = st->drt;
            rd->step = st->step;
            rd->c_round = st->c_round; rd->head = st->head; rd->pending = st->pending; rd->gram_cur = st->gram_cur;
            rd->store_first = st->first_store;
            rd->op = st->op;
            running = st->op != POP_IDLE;
        }
        still += __syncthreads_count(running);
    }
    if (tid == 0) { a.ctl->nactive = still; a.ctl->rounds++; }
    return still;
}

// exchange-only prelude for neighbour-coupled objectives under n-sharding: the first evaluation needs the neighbours' boundary
// coordinates of x0 (later rounds piggyback the boundaries of (x, drt) on the sums, see leader_round).  All threads of CTA 0.
template <class T> __device__ void leader_halo_prelude(const PArgs<T>& a)
{
    const int tid = threadIdx.x;
    const XComm* xc = a.xc;
    const int me = xc->rank, R = xc->nranks;
    const unsigned long long epoch = a.ctl->epoch + 1ull;
    const int slot = (int)(epoch % kXRing);
    const unsigned tag = (unsigned)epoch;
    const long long t_x0 = clock64();
    auto give_up = [&]() {
        if (clock64() - t_x0 > 4 * a.wait_cycles || ldv(&a.ctl->abort)) { a.ctl->abort = 1; return true; }
        return false;
    };
    for (int b = 0; b < a.B; b++)
    {
        PState<T>* st = a.probs + b;
        if (tid < 4 * R)
        {
            const int k = tid & 3;
            const double val = (k & 1) ? 0.0 : (double)__ldcg(st->x + ((k & 2) ? a.n - 1 : 0));
            ll_push(xc->inbox[tid >> 2]->ll[slot][me][4 * b + k], val, tag);
        }
    }
    for (int b = 0; b < a.B; b++)
    {
        PState<T>* st = a.probs + b;
        if (tid < 8)
        {
            const int side = tid >> 2, k = tid & 3;
            const int nb = side == 0 ? me - 1 : me + 1;
            double v = 0.0;
            if (nb >= 0 && nb < R) ll_pull(xc->inbox[me]->ll[slot][nb][4 * b + k], tag, v, give_up);
            st->halo[4 + 4 * side + k] = v;
        }
    }
    __syncthreads();
    if (tid == 0) a.ctl->epoch = epoch;
}

// ---- the kernel ----------------------------------------------------------------------------------------------------------------
template <class T, class OBJ, int ROUNDS>
__global__ void __launch_bounds__(kPThreads, 1) k_persist(PArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char p_smem[];
    T* tiles = reinterpret_cast<T*>(p_smem);      // the staging ring of the dots / combination passes
    __shared__ PShared sh;
    const int tid = threadIdx.x, G = gridDim.x, cta = blockIdx.x;
    const Own own(a.n, G, cta, a.grain);
    if (tid == 0)
    {
        for (int s = 0; s < kPMaxStages; s++) mbar_init(&sh.full_bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned phase_bits = 0;
    unsigned episode = 0;    // grid-barrier episodes so far
    constexpr bool HALO = OBJ::kHalo;
    constexpr int kDataVectors = OBJ::kDataVectors;
    long long t_last = clock64(), t_arrive = 0;   // CTA 0, thread 0: accounting (PCtl::cyc_*)
    int acct_bucket = 0;
    double acct_words = 0.0;
    __shared__ unsigned s_release;
    __shared__ __align__(16) double s_gram[kPGramScratch];   // the coefficient recursion's own scratch (c <= 21: it then runs while the first tiles of the pass are in flight)
    __shared__ PState<T> s_state[kPCache];     // CTA 0: working copies of the first problems' states (scalar logic at shared-memory latency)
    const int ncache = a.B < kPCache ? a.B : kPCache;
    if (cta == 0)
    {
        const unsigned* src = reinterpret_cast<const unsigned*>(a.probs);
        unsigned* dstw = reinterpret_cast<unsigned*>(s_state);
        for (int w = tid; w < (int)(sizeof(PState<T>) / 4) * ncache; w += kPThreads) dstw[w] = src[w];
        __syncthreads();
    }

    // Grid-wide barrier.  Arrival: the CTA's partial sums are written, bar.sync, thread 0 fences and counts in.  Between the last
    // arrival and the release CTA 0 runs `leader_work` (all its threads; returns true when nothing is left to do).  Returns that
    // verdict in every thread of every CTA (it travels in bit 31 of the release word).
    auto grid_barrier = [&](auto leader_work) -> bool {
        episode++;
        asm volatile("fence.proxy.async;" ::: "memory");   // this round's generic-proxy stores before later bulk (async-proxy) reads
        if (HALO) __threadfence();                           // boundary coordinates are read by the neighbouring CTA next round
        __syncthreads();
        if (tid == 0) { __threadfence(); atomicAdd(&a.ctl->arrive, 1u); }
        if (cta == 0)
        {
            if (tid == 0)
            {
                const long long t_start = clock64();
                t_arrive = t_start;
                while (ld_acquire_gpu_u32(&a.ctl->arrive) != episode * (unsigned)G)
                    if (clock64() - t_start > a.wait_cycles || ldv(&a.ctl->abort)) { a.ctl->abort = 1; break; }
                a.ctl->cyc_wait_all += clock64() - t_start;
            }
            __syncthreads();
            const bool stop = leader_work();
            __syncthreads();
            if (tid == 0)
            {
                const long long now = clock64();
                a.ctl->cyc_op[acct_bucket] += now - t_last;
                a.ctl->cyc_sync += now - t_arrive;
                a.ctl->n_op[acct_bucket] += 1ull;
                a.ctl->words_op[acct_bucket] += acct_words;
                t_last = now;
                st_release_gpu_u32(&a.ctl->release, episode | (stop ? kPStopBit : 0u));
            }
        }
        if (tid == 0)
        {
            const long long t_start = clock64();
            unsigned v;
            while (((v = ld_acquire_gpu_u32(&a.ctl->release)) & ~kPStopBit) < episode)
                if (clock64() - t_start > 6 * a.wait_cycles || ldv(&a.ctl->abort)) { a.ctl->abort = 1; v = kPStopBit; break; }
            s_release = v;
        }
        __syncthreads();
        return (s_release & kPStopBit) != 0u;
    };

    if (HALO && a.xc != nullptr)
        if (grid_barrier([&]() { leader_halo_prelude<T>(a); return ldv(&a.ctl->abort) != 0; })) return;

    for (;;)
    {
        // this round's op of every problem (the descriptors were published before the release that let us through)
        if (a.B > 1)
        {
            for (int b = tid; b < a.B; b += kPThreads) sh.ops[b] = (unsigned char)ldv(&a.rounds[b].op);
            __syncthreads();
        }
        acct_bucket = -1;
        acct_words = 0.0;
        for (int b = 0; b < a.B; b++)
        {
            const PRound<T>* rd = a.rounds + b;
            if (a.B > 1 && sh.ops[b] == POP_IDLE) continue;
            // a single problem: the op travels with the rest of the descriptor, and all its fields are requested before the first one is
            // looked at (one trip to L2 per round instead of two)
            const int op = (a.B > 1) ? (int)sh.ops[b] : ldv(&rd->op);
            const PState<T>* st = a.probs + b;     // fields that are fixed for the duration of the kernel only
            T* const vx = ldv(&rd->x); T* const vxp = ldv(&rd->xp); T* const vg = ldv(&rd->g); T* const vgp = ldv(&rd->gp); T* const vd = ldv(&rd->drt);
            const T step = ldv(&rd->step);
            const int c_round = ldv(&rd->c_round), head = ldv(&rd->head), pending = ldv(&rd->pending), gram_cur = ldv(&rd->gram_cur);
            const int store_first = ldv(&rd->store_first);
            if (op == POP_IDLE) continue;
            acct_bucket = (acct_bucket == -1 || acct_bucket == op) ? op : 0;
            acct_words += words_of(op, c_round, kDataVectors, store_first);
            double* dst = a.partials + (size_t)b * a.pstride * G + cta;
            const OBJ obj = PObjMaker<T, OBJ>::make(a, st->data0, st->data1, (HALO && a.xc != nullptr) ? st->halo : nullptr);
            switch (op)
            {
            case POP_FIRST:
                if constexpr (HALO) p_trial_halo<T, OBJ, 0>(obj, own, nullptr, nullptr, T(0), vx, vg, vd, tiles, sh, phase_bits, dst, G);
                else p_trial<T, OBJ, 0>(obj, own, nullptr, nullptr, T(0), vx, vg, vd, sh, dst, G, a.tune);
                break;
            case POP_TRIAL:
            case POP_MATERIALIZE:
                if constexpr (HALO) p_trial_halo<T, OBJ, 1>(obj, own, vxp, vd, step, vx, vg, nullptr, tiles, sh, phase_bits, dst, G);
                else p_trial<T, OBJ, 1>(obj, own, vxp, vd, step, vx, vg, nullptr, sh, dst, G, a.tune);
                break;
            case POP_RESTORE:
                p_restore<T>(own, vxp, vgp, vx, vg);
                break;
            case POP_DOTS_FORM:
            case POP_DOTS_PLAIN:
            {
                const bool form = op == POP_DOTS_FORM;
                PDots<T> d;
                d.n = a.n; d.h = st->hist; d.c = c_round;
                d.end = head;                                   // the old columns: the slots below the free slot `head`
                d.cnt_old = form ? c_round - 1 : c_round;
                d.new_slot = form ? head : -1;
                dots_geometry(d.c, d.h.BT() / (16 / (int)sizeof(T)), d.split, d.cols_per_round);
                __syncthreads();   // sh.slots / sh.vecs may still be read by the previous problem's pass
                {
                    const SlotRuns runs(d.end, d.cnt_old, d.h.M);
                    // age j (FORM: j >= 1) -> packed row of its slot in the staged block
                    if (tid < d.c && !(form && tid == 0))
                        sh.slots[tid] = (unsigned char)runs.row_of(slot_by_age(head, d.h.M, form ? tid - 1 : tid));
                    if (tid == 0) { sh.vecs[0] = vg; sh.vecs[1] = vx; sh.vecs[2] = vgp; sh.vecs[3] = vxp; }
                }
                if (form) p_dots<T, ROUNDS, true>(d, own, tiles, sh, phase_bits, dst, G);
                else p_dots<T, ROUNDS, false>(d, own, tiles, sh, phase_bits, dst, G);
                break;
            }
            case POP_COMBINE:
            case POP_COMBINE_TRIAL:
            {
                GramSolveArgs<T> g;
                g.c = c_round;
                g.M = st->hist.M; g.new_slot = pending; g.with_v = 1; g.a = T(-1);
                g.raw = st->raw;
                const int in = gram_cur, out = (g.new_slot >= 0) ? 1 - in : in;
                g.SY_in = st->SY[in]; g.YY_in = st->YY[in]; g.SS_in = st->SS[in];
                g.SY_out = st->SY[out]; g.YY_out = st->YY[out]; g.SS_out = st->SS[out];
                g.ys = st->ys; g.alpha = st->alpha; g.theta = st->theta;
                g.ov_slot = -1; g.ov_theta_on = 0;
                for (int age = 0; age < g.c; age++) g.slots[age] = (unsigned char)slot_by_age(head, g.M, age);
                __syncthreads();   // the tile area / tables may still be in use by the previous problem's pass
                // per age: packed row of the column in a staged block, and its ring slot
                const bool fuse = op == POP_COMBINE_TRIAL;
                {
                    const SlotRuns runs(head, g.c, g.M);
                    for (int j = tid; j < g.c; j += kPThreads)
                    {
                        sh.slots[j] = (unsigned char)runs.row_of(g.slots[j]);
                        sh.slotid[j] = g.slots[j];
                    }
                    if (tid == 0) { sh.vecs[0] = vg; sh.vecs[1] = vx; sh.vecs[2] = st->data0; sh.vecs[3] = st->data1; }
                }
                // the coefficient recursion (every CTA; CTA 0 also writes the folded Gram matrices back) and its 2c+1 results into sh.coef
                const bool own_scratch = gram_solve_smem_elems(g.c) * sizeof(T) <= sizeof(s_gram);
                auto solve_into = [&](T* scratch) {
                    gram_solve_in_smem<T>(g, scratch, cta == 0);
                    const T* s_coef = scratch + 2 * g.c * g.c;
                    T* keep = reinterpret_cast<T*>(sh.coef);
                    for (int q = tid; q < 2 * g.c + 1; q += kPThreads) keep[q] = s_coef[q];
                    __syncthreads();
                };
                if (!own_scratch) solve_into(tiles);   // a long history: the staging ring is the scratch, the copies start afterwards
                auto between = [&]() { if (own_scratch) solve_into(reinterpret_cast<T*>(s_gram)); };
                if (fuse) p_combine<T, OBJ, true, OBJ::kHalo>(obj, own, st->hist, g.c, head, tiles, vd, store_first ? vxp : nullptr, store_first ? vgp : nullptr, sh, phase_bits, dst, G, between);
                else p_combine<T, OBJ, false, false>(obj, own, st->hist, g.c, head, tiles, vd, nullptr, nullptr, sh, phase_bits, dst, G, between);
                break;
            }
            default: break;
            }
        }
        if (acct_bucket < 0) acct_bucket = 0;
        if (grid_barrier([&]() { return leader_round<T, HALO>(a, G, sh, s_state) == 0 || ldv(&a.ctl->abort) != 0; })) break;
    }
    if (cta == 0)
    {
        __syncthreads();
        const unsigned* src = reinterpret_cast<const unsigned*>(s_state);
        unsigned* dstw = reinterpret_cast<unsigned*>(a.probs);
        for (int w = tid; w < (int)(sizeof(PState<T>) / 4) * ncache; w += kPThreads) dstw[w] = src[w];
    }
}

}  // namespace lb
