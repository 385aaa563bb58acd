// persist_host.cuh -- host side of the device-resident solve (persist.cuh): solver handle, state upload, ONE cooperative launch per
// minimize() (single problem or batch), C ABI.  Included at the end of lbfgs_b200.cu.
#pragma once

struct lbfgs_b200_solver
{
    lbfgs_b200_ctx* ctx = nullptr;
    int64_t n = 0;
    int m = 0, elem = 8, B = 1;
    // the S/Y rings, tiled: H[problem][block][slot][S|Y][BT] (lb::PHist); small per-problem arrays in one slab each
    void* d_hist = nullptr;
    int bt_log = 9, M = 0;
    size_t hist_elems = 0;                // elements of one problem's tiled ring
    void* d_small = nullptr;              // [B][ ys M | alpha M | theta 1 (padded to 4) | SY,YY,SS x2: 6 M^2 ]
    size_t small_elems = 0;
    std::vector<int> ring_head, ring_ncorr, ring_gram_cur;   // ring state after the last solve (for the export below)
    std::vector<lbfgs_b200_hist*> exported;                   // column-major copies made on request (lbfgs_b200_solver_history_of)
    std::vector<char> export_fresh;
    void* vec_slab = nullptr;             // [B][7][vec_elems] : x, xp, g, gp, drt, x_lo, g_lo
    size_t vec_elems = 0;                 // n rounded up to a whole number of 256-byte lines
    void* d_state = nullptr;              // PState<T>[B]
    void* d_rounds = nullptr;             // PRound<T>[B]
    lb::PCtl* d_ctl = nullptr;
    double* d_partials = nullptr;         // [B][pstride][sm_count]
    double* d_raw = nullptr;              // [B][pstride]
    double* d_halo = nullptr;             // [B][kHaloDoubles]
    int pstride = 0;
    double* d_trace = nullptr;
    long long trace_cap = 0;
    std::vector<void*> final_g, final_x;  // device pointers of each problem's final gradient / point (inside vec_slab)
    std::vector<unsigned char> h_state;   // host copy of the states
    std::vector<unsigned char> h_rounds;  // host image of the initial round descriptors
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    float last_kernel_ms = 0.f;           // device time of the last solve's kernel (CUDA events around the launch)
    lb::PCtl last_ctl{};                  // its accounting
};

template <class T> static void* persist_kernel_for(int objective, int rounds)
{
    using namespace lb;
#define LB_PK(OBJ) (rounds <= 1 ? (void*)k_persist<T, OBJ, 1> : rounds == 2 ? (void*)k_persist<T, OBJ, 2> : (void*)k_persist<T, OBJ, 3>)
    switch (objective)
    {
    case LBFGS_B200_OBJ_ROSENBROCK_PAIRED: return LB_PK(RosenbrockPaired<T>);
    case LBFGS_B200_OBJ_QUAD_SHIFT: return LB_PK(QuadShift<T>);
    case LBFGS_B200_OBJ_ROSENBROCK_CHAINED: return LB_PK(RosenbrockChained<T>);
    case LBFGS_B200_OBJ_QUAD_TRIDIAG: return LB_PK(QuadTridiag<T>);
    }
#undef LB_PK
    return nullptr;
}

// x_inout: B vectors of n elements, `ldx` elements apart (device).  data0/data1: nullptr, or per-problem vectors `ldd` apart (ldd = 0:
// every problem shares the same data).  outs: B outcomes.  trace_host: only with B == 1.
template <class T>
static lbfgs_b200_status solver_minimize(lbfgs_b200_solver* s, int objective, const T* data0, const T* data1, int64_t ldd, const lbfgs_b200_param* prm,
                                         int ls_kind, T* x_inout, int64_t ldx, double* trace_host, long long trace_cap, lbfgs_b200_outcome* outs)
{
    using namespace lb;
    lbfgs_b200_ctx* ctx = s->ctx;
    const int B = s->B;
    REQUIRE(ctx, s->elem == (int)sizeof(T), "solver element size mismatch");
    REQUIRE(ctx, prm && outs && x_inout, "solver_minimize: NULL argument");
    REQUIRE(ctx, prm->m == s->m, "solver was created for m = %d, called with m = %d", s->m, prm->m);
    REQUIRE(ctx, ls_kind >= 0 && ls_kind <= 3, "unknown line search %d", ls_kind);
    REQUIRE(ctx, prm->past <= kMaxPast, "past > %d is not supported by the device-resident solve", kMaxPast);
    REQUIRE(ctx, ctx->nranks == 1 || ctx->x_active, "the device-resident solve needs the in-kernel exchange (comm_p2p) when sharded");
    REQUIRE(ctx, B == 1 || ldx >= s->n, "solver_minimize: the batch stride of x is shorter than n");
    REQUIRE(ctx, trace_host == nullptr || B == 1, "solver_minimize: traces are recorded for single problems only");
    const bool coupled = objective == LBFGS_B200_OBJ_ROSENBROCK_CHAINED || objective == LBFGS_B200_OBJ_QUAD_TRIDIAG;
    if (objective == LBFGS_B200_OBJ_ROSENBROCK_PAIRED) REQUIRE(ctx, s->n % 2 == 0, "paired Rosenbrock needs an even n");
    if (objective == LBFGS_B200_OBJ_QUAD_TRIDIAG) REQUIRE(ctx, data0 && data1, "quad_tridiag needs data0 = diag, data1 = rhs");
    // the data vectors are read by 16-byte bulk copies, from data + b*ldd on for problem b (lbfgs_b200.h)
    REQUIRE(ctx, (uintptr_t)data0 % 16 == 0 && (uintptr_t)data1 % 16 == 0, "solver_minimize: data0 / data1 must be 16-byte aligned");
    REQUIRE(ctx, ldd == 0 || (ldd >= s->n && (ldd * (int64_t)sizeof(T)) % 16 == 0),
            "solver_minimize: the batch stride of the data vectors must be 0 (shared) or >= n and a multiple of 16 bytes (got %lld)", (long long)ldd);
    int64_t n_global = s->n, index_offset = ctx->index_offset;
    if (ctx->nranks > 1 && coupled)
    {
        REQUIRE(ctx, ctx->n_global > 0, "a neighbour-coupled objective under n-sharding needs lbfgs_b200_set_global_extent()");
        REQUIRE(ctx, ctx->index_offset + s->n <= ctx->n_global, "local block exceeds the global extent");
        REQUIRE(ctx, ctx->rank == ctx->nranks - 1 || s->n % 4 == 0, "every block but the last must hold a multiple of 4 coordinates");
        n_global = ctx->n_global;
    }
    else if (coupled) index_offset = 0;
    if (ctx->x_active) REQUIRE(ctx, (size_t)B * (s->pstride + 4) <= (size_t)kXMaxVals, "batch of %d problems with m = %d exceeds the exchange buffer", B, s->m);
    {
        // every staged pass must fit at least one tile into the staging ring, or it would wait for a copy that was never issued
        const int data_vectors = objective == LBFGS_B200_OBJ_QUAD_TRIDIAG ? 2 : 0;
        const int stages = persist_min_stages(s->m, s->elem, 1 << s->bt_log, coupled, data_vectors);
        REQUIRE(ctx, stages >= 1, "solver_minimize: with history blocks of %d elements (LBFGS_B200_STAGES) a pass of m = %d does not fit the staging ring",
                1 << s->bt_log, s->m);
    }
    const int rounds = (s->m + kGramMaxWarps - 1) / kGramMaxWarps;   // column pairs per round of the dots pass: at most one per warp
    void* kernel = persist_kernel_for<T>(objective, rounds);
    if (!kernel) return fail(ctx, LBFGS_B200_ERR_INVALID, "unknown objective id %d", objective);

    if (trace_host && trace_cap > s->trace_cap)
    {
        pool_free(ctx, s->d_trace);
        s->d_trace = nullptr;
        CU(ctx, pool_alloc(ctx, (void**)&s->d_trace, sizeof(double) * (size_t)trace_cap));
        s->trace_cap = trace_cap;
    }

    // ---- states ----
    s->h_state.assign(sizeof(PState<T>) * (size_t)B, 0);
    PState<T>* hs = reinterpret_cast<PState<T>*>(s->h_state.data());
    const size_t vb = sizeof(T) * (size_t)s->n;
    for (int b = 0; b < B; b++)
    {
        PState<T>& p = hs[b];
        T* base = static_cast<T*>(s->vec_slab) + (size_t)b * 7 * s->vec_elems;
        p.x = base; p.xp = base + s->vec_elems; p.g = base + 2 * s->vec_elems; p.gp = base + 3 * s->vec_elems;
        p.drt = base + 4 * s->vec_elems; p.x_lo = base + 5 * s->vec_elems; p.g_lo = base + 6 * s->vec_elems;
        p.hist.H = static_cast<T*>(s->d_hist) + (size_t)b * s->hist_elems;
        p.hist.bt_log = s->bt_log; p.hist.M = s->M; p.hist.bstride = (int64_t)s->M * 2 * ((int64_t)1 << s->bt_log);
        T* small = static_cast<T*>(s->d_small) + (size_t)b * s->small_elems;
        const size_t mm = (size_t)s->M * s->M;
        p.ys = small; p.alpha = small + s->M; p.theta = small + 2 * s->M;
        for (int k = 0; k < 2; k++) { p.SY[k] = small + 2 * s->M + 4 + (3 * k + 0) * mm; p.YY[k] = small + 2 * s->M + 4 + (3 * k + 1) * mm; p.SS[k] = small + 2 * s->M + 4 + (3 * k + 2) * mm; }
        p.data0 = data0 ? data0 + (size_t)b * ldd : nullptr;
        p.data1 = data1 ? data1 + (size_t)b * ldd : nullptr;
        p.raw = s->d_raw + (size_t)b * s->pstride;
        p.halo = s->d_halo + (size_t)b * kHaloDoubles;
        p.head = 0; p.ncorr = 0; p.M = s->M; p.m = s->m; p.gram_cur = 0; p.pending = -1;
        p.op = POP_FIRST; p.c_round = 0;
        p.epsilon = (T)prm->epsilon; p.epsilon_rel = (T)prm->epsilon_rel; p.delta = (T)prm->delta; p.max_step = (T)prm->max_step;
        p.eps_gate = std::numeric_limits<T>::epsilon();
        p.past = prm->past; p.max_iterations = prm->max_iterations; p.ls_kind = ls_kind;
        // the first trial of every search rides on the combination pass; a neighbour-coupled objective needs its neighbours' x + d,
        // which only exist on this rank when n is not sharded
        p.fuse_first_trial = (coupled && ctx->nranks > 1) ? 0 : 1;
        p.adaptive_first_store = (getenv("LBFGS_B200_VIRTUAL_FIRST_TRIAL") && atoi(getenv("LBFGS_B200_VIRTUAL_FIRST_TRIAL")) != 0) ? 1 : 0;
        p.first_store = p.adaptive_first_store ? 0 : 1;
        p.ls_opt.linesearch = (ls_kind == 3) ? 3 : prm->linesearch;
        p.ls_opt.max_linesearch = prm->max_linesearch;
        p.ls_opt.min_step = (T)prm->min_step; p.ls_opt.max_step = (T)prm->max_step; p.ls_opt.ftol = (T)prm->ftol; p.ls_opt.wolfe = (T)prm->wolfe;
        p.trace = trace_host ? s->d_trace : nullptr;
        p.trace_cap = trace_host ? trace_cap : 0;
        CU(ctx, cudaMemcpyAsync(p.x, x_inout + (size_t)b * ldx, vb, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    s->h_rounds.assign(sizeof(PRound<T>) * (size_t)B, 0);
    PRound<T>* hr = reinterpret_cast<PRound<T>*>(s->h_rounds.data());
    for (int b = 0; b < B; b++)
    {
        const PState<T>& p = hs[b];
        hr[b].x = p.x; hr[b].xp = p.xp; hr[b].g = p.g; hr[b].gp = p.gp; hr[b].drt = p.drt;
        hr[b].step = T(0); hr[b].op = p.op; hr[b].c_round = 0; hr[b].head = 0; hr[b].pending = -1; hr[b].gram_cur = p.gram_cur; hr[b].store_first = p.first_store;
    }
    // BFGSMat::reset (BFGSMat.h:61-78): no pairs, theta = 1, Gram matrices cleared
    CU(ctx, cudaMemsetAsync(s->d_small, 0, sizeof(T) * s->small_elems * (size_t)B, ctx->stream));
    {
        static const T one = T(1);
        for (int b = 0; b < B; b++) CU(ctx, cudaMemcpyAsync(hs[b].theta, &one, sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    }
    CU(ctx, cudaMemcpyAsync(s->d_state, hs, sizeof(PState<T>) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(s->d_rounds, hr, sizeof(PRound<T>) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    PCtl hc{};
    hc.nactive = B;
    hc.epoch = ctx->x_epoch;
    CU(ctx, cudaMemcpyAsync(s->d_ctl, &hc, sizeof(hc), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemsetAsync(s->d_halo, 0, sizeof(double) * kHaloDoubles * (size_t)B, ctx->stream));

    // ---- one cooperative launch: one CTA per SM (fewer when the vector has fewer tiles than SMs) ----
    const int64_t units = (s->n + ((int64_t)1 << s->bt_log) - 1) >> s->bt_log;
    const int grid = (int)(units < ctx->sm_count ? (units < 1 ? 1 : units) : ctx->sm_count);
    const size_t smem = (size_t)kPStageBytes;
    CU(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kPThreads, smem));
    REQUIRE(ctx, per_sm >= 1, "the persistent solve kernel does not fit on an SM of this device");
    PArgs<T> a{};
    a.probs = static_cast<PState<T>*>(s->d_state); a.rounds = static_cast<PRound<T>*>(s->d_rounds); a.B = B; a.ctl = s->d_ctl; a.partials = s->d_partials; a.pstride = s->pstride;
    a.n = s->n; a.grain = 1 << s->bt_log; a.xc = ctx->x_active ? ctx->x_comm : nullptr;
    a.index_offset = index_offset; a.n_global = n_global;
    a.wait_cycles = kPWaitCycles;
    if (const char* e = getenv("LBFGS_B200_WATCHDOG_SCALE")) { const long long k = atoll(e); if (k >= 1 && k <= 100000) a.wait_cycles *= k; }
    a.tune = ((size_t)s->n * sizeof(T) * 4 > ((size_t)96 << 20)) ? 4 : 0;     // x, xp, g, d of one problem exceed what L2 can hold between rounds
    if (const char* e = getenv("LBFGS_B200_TUNE")) a.tune = atoi(e);
    void* kargs[] = {&a};
    CU(ctx, cudaEventRecord(s->ev0, ctx->stream));
    CU(ctx, cudaLaunchCooperativeKernel(kernel, dim3((unsigned)grid), dim3(kPThreads), kargs, smem, ctx->stream));
    CU(ctx, cudaEventRecord(s->ev1, ctx->stream));
    ctx->launches++;
    CU(ctx, cudaMemcpyAsync(hs, s->d_state, sizeof(PState<T>) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(&hc, s->d_ctl, sizeof(hc), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->x_epoch = hc.epoch;
    s->last_ctl = hc;
    CU(ctx, cudaEventElapsedTime(&s->last_kernel_ms, s->ev0, s->ev1));
    if (hc.abort) return fail(ctx, LBFGS_B200_ERR_CUDA, "the persistent solve gave up waiting at a grid / cross-rank barrier after %llu rounds (watchdog)", hc.rounds);

    // the states tell where the results live after all the pointer rotations
    for (int b = 0; b < B; b++)
    {
        const PState<T>& p = hs[b];
        CU(ctx, cudaMemcpyAsync(x_inout + (size_t)b * ldx, p.x, vb, cudaMemcpyDeviceToDevice, ctx->stream));
        s->final_g[b] = p.g;
        s->final_x[b] = p.x;
        s->ring_head[b] = p.head; s->ring_ncorr[b] = p.ncorr; s->ring_gram_cur[b] = p.gram_cur;
        s->export_fresh[b] = 0;
        outs[b].status = p.status;
        outs[b].niter = p.niter;
        outs[b].nfev = p.nfev;
        outs[b].fx = (double)p.fx;
        outs[b].gnorm = (double)p.gnorm;
        outs[b].rounds = p.rounds;
    }
    if (trace_host)
    {
        const long long cnt = hs[0].nfev < trace_cap ? hs[0].nfev : trace_cap;
        CU(ctx, cudaMemcpyAsync(trace_host, s->d_trace, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return LBFGS_B200_OK;
}

// The ring of problem b as an ordinary (column-major) lbfgs_b200_hist, for final_approx_hessian() and inspection: made on request,
// refreshed after every solve.  nullptr on failure (the context holds the message).
template <class T> __global__ void k_untile_history(lb::PHist<T> h, int64_t n, int64_t ld, T* __restrict__ S, T* __restrict__ Y)
{
    const int slot = blockIdx.y;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        S[(int64_t)slot * ld + i] = *h.s_at(slot, i);
        Y[(int64_t)slot * ld + i] = *h.y_at(slot, i);
    }
}
#if defined(LBFGS_B200_PERSIST_F64)
template <class T> static lbfgs_b200_hist* export_history(lbfgs_b200_solver* s, int b)
{
    lbfgs_b200_ctx* ctx = s->ctx;
    lbfgs_b200_hist*& h = s->exported[(size_t)b];
    if (h && s->export_fresh[(size_t)b]) return h;
    if (!h && lbfgs_b200_hist_create(ctx, &h, s->n, s->m, s->elem) != LBFGS_B200_OK) return nullptr;
    lb::PHist<T> ph;
    ph.H = static_cast<T*>(s->d_hist) + (size_t)b * s->hist_elems;
    ph.bt_log = s->bt_log; ph.M = s->M; ph.bstride = (int64_t)s->M * 2 * ((int64_t)1 << s->bt_log);
    const dim3 grid((unsigned)std::min<int64_t>((s->n + 255) / 256, 4 * ctx->sm_count), (unsigned)s->M);
    k_untile_history<T><<<grid, 256, 0, ctx->stream>>>(ph, s->n, h->ld, static_cast<T*>(h->S), static_cast<T*>(h->Y));
    const T* small = static_cast<const T*>(s->d_small) + (size_t)b * s->small_elems;
    const size_t mm = (size_t)s->M * s->M;
    cudaMemcpyAsync(h->ys, small, sizeof(T) * s->M, cudaMemcpyDeviceToDevice, ctx->stream);
    cudaMemcpyAsync(h->alpha, small + s->M, sizeof(T) * s->M, cudaMemcpyDeviceToDevice, ctx->stream);
    cudaMemcpyAsync(h->theta, small + 2 * s->M, sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream);
    for (int k = 0; k < 2; k++)
    {
        cudaMemcpyAsync(h->SY[k], small + 2 * s->M + 4 + (3 * k + 0) * mm, sizeof(T) * mm, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaMemcpyAsync(h->YY[k], small + 2 * s->M + 4 + (3 * k + 1) * mm, sizeof(T) * mm, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaMemcpyAsync(h->SS[k], small + 2 * s->M + 4 + (3 * k + 2) * mm, sizeof(T) * mm, cudaMemcpyDeviceToDevice, ctx->stream);
    }
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess) { fail(ctx, LBFGS_B200_ERR_CUDA, "exporting the solver's history failed"); return nullptr; }
    h->head = s->ring_head[(size_t)b]; h->ncorr = s->ring_ncorr[(size_t)b]; h->gram_cur = s->ring_gram_cur[(size_t)b]; h->pending = -1;
    s->export_fresh[(size_t)b] = 1;
    return h;
}
#endif

extern "C" {

#ifdef LBFGS_B200_PERSIST_F64
lbfgs_b200_status lbfgs_b200_solver_create_batch(lbfgs_b200_ctx* ctx, int64_t n, int m, int elem_bytes, int batch, lbfgs_b200_solver** out)
{
    REQUIRE(ctx, ctx && out, "solver_create: NULL argument");
    *out = nullptr;
    REQUIRE(ctx, batch >= 1 && batch <= 4096, "solver_create: 1 <= batch <= 4096 (got %d)", batch);
    REQUIRE(ctx, n >= 1 && m >= 1 && m <= 64, "solver_create: need n >= 1 and 1 <= m <= 64 (got n=%lld m=%d)", (long long)n, m);
    REQUIRE(ctx, elem_bytes == 8 || elem_bytes == 4, "solver_create: elem_bytes must be 8 or 4");
    lbfgs_b200_solver* s = new (std::nothrow) lbfgs_b200_solver();
    if (!s) return fail(ctx, LBFGS_B200_ERR_ALLOC, "out of host memory");
    s->ctx = ctx; s->n = n; s->m = m; s->elem = elem_bytes; s->B = batch;
    s->final_g.assign((size_t)batch, nullptr);
    s->final_x.assign((size_t)batch, nullptr);
    s->M = m + 1;
    // block length of the tiled history: the largest power of two for which two stages of 2m+4 rows fit the kernel's staging ring
    {
        int want_stages = 2;
        if (const char* e = getenv("LBFGS_B200_STAGES")) { const int v = atoi(e); if (v >= 1 && v <= lb::kPMaxStages) want_stages = v; }
        const int bt = lb::persist_block_len(m, elem_bytes, want_stages);
        s->bt_log = 0;
        while ((1 << s->bt_log) < bt) s->bt_log++;
    }
    const int64_t nblocks = (n + ((int64_t)1 << s->bt_log) - 1) >> s->bt_log;
    s->hist_elems = (size_t)nblocks * s->M * 2 * ((size_t)1 << s->bt_log);
    s->small_elems = (size_t)2 * s->M + 4 + 6 * (size_t)s->M * s->M;
    s->ring_head.assign((size_t)batch, 0); s->ring_ncorr.assign((size_t)batch, 0); s->ring_gram_cur.assign((size_t)batch, 0);
    s->exported.assign((size_t)batch, nullptr); s->export_fresh.assign((size_t)batch, 0);
    cudaError_t e = cudaSuccess;
    s->vec_elems = (((size_t)n * elem_bytes + 255) & ~size_t(255)) / elem_bytes;
    s->pstride = ((m * lb::kGramVals > 8 ? m * lb::kGramVals : 8) + 7) & ~7;
    const size_t state_bytes = (elem_bytes == 8 ? sizeof(lb::PState<double>) : sizeof(lb::PState<float>)) * (size_t)batch;
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->vec_slab, (size_t)batch * 7 * s->vec_elems * elem_bytes);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_hist, (size_t)batch * s->hist_elems * elem_bytes);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_small, (size_t)batch * s->small_elems * elem_bytes);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_state, state_bytes);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_rounds, (elem_bytes == 8 ? sizeof(lb::PRound<double>) : sizeof(lb::PRound<float>)) * (size_t)batch);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_ctl, sizeof(lb::PCtl));
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_partials, sizeof(double) * (size_t)batch * s->pstride * ctx->sm_count);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_raw, sizeof(double) * (size_t)batch * s->pstride);
    if (e == cudaSuccess) e = pool_alloc(ctx, (void**)&s->d_halo, sizeof(double) * (size_t)batch * lb::kHaloDoubles);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
    if (e != cudaSuccess)
    {
        lbfgs_b200_solver_destroy(s);
        return fail(ctx, e == cudaErrorMemoryAllocation ? LBFGS_B200_ERR_ALLOC : LBFGS_B200_ERR_CUDA, "solver_create: %s", cudaGetErrorString(e));
    }
    *out = s;
    return LBFGS_B200_OK;
}

lbfgs_b200_status lbfgs_b200_solver_create(lbfgs_b200_ctx* ctx, int64_t n, int m, int elem_bytes, lbfgs_b200_solver** out)
{
    return lbfgs_b200_solver_create_batch(ctx, n, m, elem_bytes, 1, out);
}

void lbfgs_b200_solver_destroy(lbfgs_b200_solver* s)
{
    if (!s) return;
    if (s->ctx && s->ctx->stream) cudaStreamSynchronize(s->ctx->stream);   // the events below must not be in use
    for (void* p : {(void*)s->vec_slab, (void*)s->d_state, (void*)s->d_rounds, (void*)s->d_ctl, (void*)s->d_partials, (void*)s->d_raw, (void*)s->d_halo,
                    (void*)s->d_trace, (void*)s->d_hist, (void*)s->d_small})
        pool_free(s->ctx, p);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    for (lbfgs_b200_hist* h : s->exported) lbfgs_b200_hist_destroy(h);
    delete s;
}

int lbfgs_b200_solver_batch(const lbfgs_b200_solver* s) { return s ? s->B : 0; }
lbfgs_b200_status lbfgs_b200_solver_profile(const lbfgs_b200_solver* s, double* kernel_ms, double* ms_by_op10, unsigned long long* rounds_by_op10,
                                            double* alg_bytes_by_op10, double* sync_ms)
{
    if (!s) return LBFGS_B200_ERR_INVALID;
    const lb::PCtl& c = s->last_ctl;
    long long total = 0;
    for (int k = 0; k < lb::kPOps; k++) total += c.cyc_op[k];
    const double scale = total > 0 ? (double)s->last_kernel_ms / (double)total : 0.0;   // CTA 0's cycles -> share of the event-timed kernel
    if (kernel_ms) *kernel_ms = s->last_kernel_ms;
    for (int k = 0; k < lb::kPOps; k++)
    {
        if (ms_by_op10) ms_by_op10[k] = scale * (double)c.cyc_op[k];
        if (rounds_by_op10) rounds_by_op10[k] = c.n_op[k];
        if (alg_bytes_by_op10) alg_bytes_by_op10[k] = c.words_op[k] * (double)s->n * (double)s->elem;
    }
    if (sync_ms) { sync_ms[0] = scale * (double)c.cyc_sync; sync_ms[1] = scale * (double)c.cyc_wait_all; sync_ms[2] = scale * (double)c.cyc_exchange; }
    return LBFGS_B200_OK;
}
const void* lbfgs_b200_solver_final_grad(const lbfgs_b200_solver* s) { return s ? s->final_g[0] : nullptr; }
const void* lbfgs_b200_solver_final_grad_of(const lbfgs_b200_solver* s, int b) { return (s && b >= 0 && b < s->B) ? s->final_g[(size_t)b] : nullptr; }
lbfgs_b200_hist* lbfgs_b200_solver_history_of(lbfgs_b200_solver* s, int b)
{
    if (!s || b < 0 || b >= s->B) return nullptr;
    if (s->elem == 8) return export_history<double>(s, b);
    return export_history<float>(s, b);
}
lbfgs_b200_hist* lbfgs_b200_solver_history(lbfgs_b200_solver* s) { return lbfgs_b200_solver_history_of(s, 0); }

lbfgs_b200_status lbfgs_b200_solver_minimize_f64(lbfgs_b200_solver* s, int objective, const double* data0, const double* data1,
                                                 const lbfgs_b200_param* prm, int line_search, double* x_inout, double* trace_host,
                                                 long long trace_cap, lbfgs_b200_outcome* out)
{
    if (!s || !s->ctx) return LBFGS_B200_ERR_INVALID;
    if (s->B != 1) return fail(s->ctx, LBFGS_B200_ERR_INVALID, "solver_minimize: the solver holds a batch of %d problems, use solver_minimize_batch", s->B);
    return solver_minimize<double>(s, objective, data0, data1, 0, prm, line_search, x_inout, s->n, trace_host, trace_cap, out);
}
lbfgs_b200_status lbfgs_b200_solver_minimize_batch_f64(lbfgs_b200_solver* s, int objective, const double* data0, const double* data1, int64_t ldd,
                                                       const lbfgs_b200_param* prm, int line_search, double* x_inout, int64_t ldx,
                                                       lbfgs_b200_outcome* outs)
{
    if (!s || !s->ctx) return LBFGS_B200_ERR_INVALID;
    return solver_minimize<double>(s, objective, data0, data1, ldd, prm, line_search, x_inout, ldx, nullptr, 0, outs);
}
#endif  // LBFGS_B200_PERSIST_F64

#ifdef LBFGS_B200_PERSIST_F32
lbfgs_b200_status lbfgs_b200_solver_minimize_f32(lbfgs_b200_solver* s, int objective, const float* data0, const float* data1,
                                                 const lbfgs_b200_param* prm, int line_search, float* x_inout, double* trace_host,
                                                 long long trace_cap, lbfgs_b200_outcome* out)
{
    if (!s || !s->ctx) return LBFGS_B200_ERR_INVALID;
    if (s->B != 1) return fail(s->ctx, LBFGS_B200_ERR_INVALID, "solver_minimize: the solver holds a batch of %d problems, use solver_minimize_batch", s->B);
    return solver_minimize<float>(s, objective, data0, data1, 0, prm, line_search, x_inout, s->n, trace_host, trace_cap, out);
}
lbfgs_b200_status lbfgs_b200_solver_minimize_batch_f32(lbfgs_b200_solver* s, int objective, const float* data0, const float* data1, int64_t ldd,
                                                       const lbfgs_b200_param* prm, int line_search, float* x_inout, int64_t ldx,
                                                       lbfgs_b200_outcome* outs)
{
    if (!s || !s->ctx) return LBFGS_B200_ERR_INVALID;
    return solver_minimize<float>(s, objective, data0, data1, ldd, prm, line_search, x_inout, ldx, nullptr, 0, outs);
}

#endif  // LBFGS_B200_PERSIST_F32

}  // extern "C"
