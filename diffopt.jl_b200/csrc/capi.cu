// C-ABI entry points: ctx lifetime + the QuadraticProgram batch calls (include/diffopt_b200.h).
#include "common.cuh"

int32_t qp_batch_launch_generic(diffopt_b200_ctx* ctx, const QpSolveArgs& a);
int32_t qp_batch_launch_tuned(diffopt_b200_ctx* ctx, const QpSolveArgs& a, bool* handled);

extern "C" {

int32_t diffopt_b200_version(void) { return 100; }

int32_t diffopt_b200_create(int32_t device, diffopt_b200_ctx** out) {
    if (!out) return -1;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) return -2;  // no CUDA device: there is no CPU fallback
    if (device < 0 || device >= count) return -1;
    DeviceGuard guard_(device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -2;
    if (prop.major != 10) return -4;  // this library only carries sm_100a code
    diffopt_b200_ctx* ctx = new diffopt_b200_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess) {
        delete ctx;
        return -2;
    }
    *out = ctx;
    return 0;
}

static void release_csr(CsrDev& c) {
    c.rowptr.release(); c.colind.release(); c.val.release();
    c.t_rowptr.release(); c.t_colind.release(); c.t_val.release();
    c.blk.release(); c.t_blk.release();
    for (DevBuf* b : {&c.sval, &c.scol, &c.spos, &c.t_sval, &c.t_scol, &c.t_spos}) b->release(); c.cblk.release(); c.t_cblk.release(); c.gblk.release(); c.t_gblk.release();
}

}  // extern "C"

void conic_state_release(ConicState& c) {
    release_csr(c.A);
    for (DevBuf* b : {&c.b, &c.c, &c.x, &c.s, &c.y, &c.v, &c.vp, &c.row_kind, &c.nn_scale, &c.soc_off, &c.soc_dim,
                      &c.soc_case, &c.soc_nx, &c.psd_off, &c.psd_d, &c.psd_uoff, &c.psd_U, &c.psd_Bm, &c.psd_ident,
                      &c.psd_work, &c.psd_lam, &c.psd_loff, &c.psd_tri, &c.psd_toff, &c.w1, &c.w2, &c.w3, &c.exp_off,
                      &c.exp_neg, &c.blk3, &c.pow_off, &c.pow_neg, &c.pow_alpha})
        b->release();
}

extern "C" {

int32_t diffopt_b200_destroy(diffopt_b200_ctx* ctx) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& b : ctx->in) b.release();
    for (auto& b : ctx->out) b.release();
    ctx->info.release();
    ctx->qp_fb.release();
    ctx->qp_max.release();
    ctx->qp_sticky.release();
    if (ctx->qp_hmax_host) cudaFreeHost(ctx->qp_hmax_host);
    for (cudaEvent_t ev : ctx->qp_hmax_ev)
        if (ev) cudaEventDestroy(ev);
    QpBatchState& q = ctx->qp;
    q.Q.release(); q.G.release(); q.A.release(); q.h.release(); q.z.release(); q.lam.release(); q.nu.release();
    for (DevBuf* b : {&ctx->qpf.f, &ctx->qpf.fb, &ctx->qpf.gin, &ctx->qpf.gout}) b->release();
    conic_state_release(ctx->conic);
    LsqrWork& l = ctx->lsqr;
    for (DevBuf* b : {&l.u, &l.v, &l.w, &l.x, &l.tmp, &l.scal}) b->release();
    release_csr(ctx->lsqr_mat);
    sparse_mf_release(ctx);
    conic_batch_release(ctx);
    nccl_release(ctx);
    ctx->qp_unpacked[0].release();
    ctx->qp_unpacked[1].release();
    for (DevBuf& b : ctx->qp_coo) b.release();
    ctx->qp_scratch.release();
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

const char* diffopt_b200_last_error(diffopt_b200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
int64_t diffopt_b200_launch_count(diffopt_b200_ctx* ctx) { return ctx ? ctx->launches : 0; }
void* diffopt_b200_stream(diffopt_b200_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
double diffopt_b200_last_kernel_ms(diffopt_b200_ctx* ctx) { return ctx ? ctx->last_ms : 0.0; }

int32_t diffopt_b200_host_alloc(void** ptr, int64_t bytes) {
    if (!ptr || bytes < 0) return -1;
    cudaError_t e = cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault);
    return e == cudaSuccess ? 0 : -100 - (int32_t)e;
}
int32_t diffopt_b200_host_free(void* ptr) {
    cudaError_t e = cudaFreeHost(ptr);
    return e == cudaSuccess ? 0 : -100 - (int32_t)e;
}

}  // extern "C"

int32_t qp_batch_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a) {
    bool handled = false;
    int32_t rc = qp_batch_launch_tuned(ctx, a, &handled);
    if (handled) return rc;
    ctx->qp_last_kernel = 0;
    return qp_batch_launch_generic(ctx, a);
}

// Scan info[] (device) after the solve: returns first failing instance + 1, or 0.
int32_t finish_info(diffopt_b200_ctx* ctx, int64_t B, int* dinfo, int32_t* info_user, int memspace,
                           std::vector<int>& hinfo) {
    hinfo.resize((size_t)B);
    cudaError_t e = cudaMemcpyAsync(hinfo.data(), dinfo, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream);
    if (e != cudaSuccess) return -100 - (int32_t)e;
    e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        ctx->err = std::string("kernel failed: ") + cudaGetErrorString(e);
        return -100 - (int32_t)e;
    }
    int32_t rc = 0;
    for (int64_t b = 0; b < B; ++b)
        if (hinfo[(size_t)b] != 0) {
            rc = (int32_t)(b + 1);
            break;
        }
    if (info_user && memspace == DIFFOPT_B200_HOST) memcpy(info_user, hinfo.data(), sizeof(int) * (size_t)B);
    return rc;
}

int32_t qp_solve_common(diffopt_b200_ctx* ctx, QpSolveArgs a, double* fwd_user, double* rev_user, int32_t* info_user, int memspace,
                        bool async) {
    const int64_t B = a.B;
    const int N = a.n + a.m + a.p;
    void *dfwd = nullptr, *drev = nullptr;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], fwd_user, sizeof(double) * B * N, memspace, &dfwd));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[1], rev_user, sizeof(double) * B * N, memspace, &drev));
    int* dinfo;
    if (info_user && memspace == DIFFOPT_B200_DEVICE) {
        dinfo = info_user;
    } else {
        DO_CUDA(ctx, ctx->info.reserve(sizeof(int) * (size_t)B));
        dinfo = ctx->info.as<int>();
    }
    a.fwd = (double*)dfwd;
    a.rev = (double*)drev;
    a.info = dinfo;
    if (async) {
        if (!ctx->qp_sticky.ptr) {
            DO_CUDA(ctx, ctx->qp_sticky.reserve(sizeof(unsigned long long)));
            DO_CUDA(ctx, cudaMemsetAsync(ctx->qp_sticky.ptr, 0xFF, sizeof(unsigned long long), ctx->stream));
        }
        a.sticky = ctx->qp_sticky.as<unsigned long long>();
        a.call_seq = ctx->async_calls++;
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int32_t rc = qp_batch_launch(ctx, a);
    if (rc != 0) return rc;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, stage_out_finish(ctx, dfwd, fwd_user, sizeof(double) * B * N, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, drev, rev_user, sizeof(double) * B * N, memspace));
    if (async) {  // status is collected by diffopt_b200_synchronize
        ctx->async_pending = true;
        return 0;
    }
    std::vector<int> hinfo;
    rc = finish_info(ctx, B, dinfo, info_user, memspace, hinfo);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return rc;
}

static int32_t check_shape(diffopt_b200_ctx* ctx, int64_t B, int n, int m, int p) {
    if (B < 0 || n <= 0 || m < 0 || p < 0) BAD_ARG(ctx, "qp_batch: need B >= 0, n > 0, m >= 0, p >= 0");
    return 0;
}

extern "C" {

int32_t diffopt_b200_qp_batch_solve(diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
                                    const double* Q, const double* G, const double* A, const double* h,
                                    const double* z, const double* lam, const double* nu, const double* dQ,
                                    const double* dq, const double* dG, const double* dh, const double* dA,
                                    const double* db, const double* dl_dz, double* fwd_out, double* rev_out,
                                    int32_t* info, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (int32_t rc = check_shape(ctx, B, n, m, p)) return rc;
    if (B == 0) return 0;
    if (!Q || !z || (m > 0 && (!G || !h || !lam)) || (p > 0 && (!A || !nu)))
        BAD_ARG(ctx, "qp_batch_solve: Q, z (and G, h, lam when m > 0; A, nu when p > 0) are required");
    if (rev_out && !dl_dz) BAD_ARG(ctx, "qp_batch_solve: rev_out requested without dl_dz");
    if (!fwd_out && !rev_out) BAD_ARG(ctx, "qp_batch_solve: nothing to compute (fwd_out and rev_out are NULL)");
    QpSolveArgs a{};
    a.B = B; a.n = n; a.m = m; a.p = p;
    const size_t d = sizeof(double);
    const void* ptr;
#define STAGE(slot, field, src, count)                                                   \
    DO_CUDA(ctx, stage_in(ctx, ctx->in[slot], src, d * (size_t)B * (size_t)(count), memspace, &ptr)); \
    a.field = (const double*)ptr;
    STAGE(0, Q, Q, (size_t)n * n)
    STAGE(1, G, G, (size_t)m * n)
    STAGE(2, A, A, (size_t)p * n)
    STAGE(3, h, h, m)
    STAGE(4, z, z, n)
    STAGE(5, lam, lam, m)
    STAGE(6, nu, nu, p)
    if (fwd_out) {
        STAGE(7, dQ, dQ, (size_t)n * n)
        STAGE(8, dq, dq, n)
        STAGE(9, dG, dG, (size_t)m * n)
        STAGE(10, dh, dh, m)
        STAGE(11, dA, dA, (size_t)p * n)
        STAGE(12, db, db, p)
    }
    if (rev_out) { STAGE(13, seed, dl_dz, n) }
    return qp_solve_common(ctx, a, fwd_out, rev_out, info, memspace, false);
}

int32_t diffopt_b200_qp_batch_solve_async(diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
                                          const double* Q, const double* G, const double* A, const double* h,
                                          const double* z, const double* lam, const double* nu, const double* dQ,
                                          const double* dq, const double* dG, const double* dh, const double* dA,
                                          const double* db, const double* dl_dz, double* fwd_out, double* rev_out,
                                          int32_t* info) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (int32_t rc = check_shape(ctx, B, n, m, p)) return rc;
    if (B == 0) return 0;
    if (!Q || !z || (m > 0 && (!G || !h || !lam)) || (p > 0 && (!A || !nu)))
        BAD_ARG(ctx, "qp_batch_solve_async: Q, z (and G, h, lam when m > 0; A, nu when p > 0) are required");
    if (rev_out && !dl_dz) BAD_ARG(ctx, "qp_batch_solve_async: rev_out requested without dl_dz");
    if (!fwd_out && !rev_out) BAD_ARG(ctx, "qp_batch_solve_async: nothing to compute (fwd_out and rev_out are NULL)");
    QpSolveArgs a{};
    a.B = B; a.n = n; a.m = m; a.p = p;
    a.Q = Q; a.G = G; a.A = A; a.h = h; a.z = z; a.lam = lam; a.nu = nu;
    if (fwd_out) { a.dQ = dQ; a.dq = dq; a.dG = dG; a.dh = dh; a.dA = dA; a.db = db; }
    if (rev_out) a.seed = dl_dz;
    return qp_solve_common(ctx, a, fwd_out, rev_out, info, DIFFOPT_B200_DEVICE, true);
}

int32_t diffopt_b200_qp_batch_last_stats(diffopt_b200_ctx* ctx, int64_t* out3) {
    if (!ctx || !out3) return -1;
    DeviceGuard guard_(ctx->device);
    out3[0] = 0;
    out3[1] = ctx->qp_last_hint;
    out3[2] = ctx->qp_last_kernel;
    if (ctx->qp_last_kernel == 3) out3[0] = ctx->qpf.nrej;
    if (ctx->qp_last_kernel == 2 && ctx->qp_fb.ptr) {
        int nfb = 0;
        DO_CUDA(ctx, cudaMemcpyAsync(&nfb, ctx->qp_fb.ptr, sizeof nfb, cudaMemcpyDeviceToHost, ctx->stream));
        DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        out3[0] = nfb;
    }
    return 0;
}

int32_t diffopt_b200_synchronize(diffopt_b200_ctx* ctx) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    int32_t rc = 0;
    if (ctx->async_pending && ctx->qp_sticky.ptr) {
        unsigned long long first_bad = ~0ull;
        DO_CUDA(ctx, cudaMemcpyAsync(&first_bad, ctx->qp_sticky.ptr, sizeof first_bad, cudaMemcpyDeviceToHost, ctx->stream));
        DO_CUDA(ctx, cudaMemsetAsync(ctx->qp_sticky.ptr, 0xFF, sizeof first_bad, ctx->stream));
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            ctx->err = std::string("kernel failed: ") + cudaGetErrorString(e);
            return -100 - (int32_t)e;
        }
        if (first_bad != ~0ull) {
            rc = (int32_t)(first_bad & 0xFFFFFFFFull);
            char msg[128];
            snprintf(msg, sizeof msg, "singular KKT matrix: instance %d of stream-ordered call %u since the last synchronize",
                     rc, (unsigned)(first_bad >> 32));
            ctx->err = msg;
        }
        ctx->async_pending = false;
        ctx->async_calls = 0;
    } else {
        DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return rc;
}

int32_t diffopt_b200_qp_batch_setup(diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
                                    const double* Q, const double* G, const double* A, const double* h,
                                    const double* z, const double* lam, const double* nu, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (int32_t rc = check_shape(ctx, B, n, m, p)) return rc;
    if (!Q || !z || (m > 0 && (!G || !h || !lam)) || (p > 0 && (!A || !nu)))
        BAD_ARG(ctx, "qp_batch_setup: Q, z (and G, h, lam when m > 0; A, nu when p > 0) are required");
    QpBatchState& s = ctx->qp;
    s.valid = false;
    ctx->qpf.valid = false;
    s.B = B; s.n = n; s.m = m; s.p = p;
    const size_t d = sizeof(double);
    cudaMemcpyKind kind = memspace == DIFFOPT_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
#define KEEP(buf, src, count)                                                                   \
    {                                                                                           \
        size_t bytes = d * (size_t)B * (size_t)(count);                                         \
        DO_CUDA(ctx, s.buf.reserve(bytes ? bytes : 8));                                         \
        if (bytes) DO_CUDA(ctx, cudaMemcpyAsync(s.buf.ptr, src, bytes, kind, ctx->stream));     \
    }
    KEEP(Q, Q, (size_t)n * n)
    KEEP(G, G, (size_t)m * n)
    KEEP(A, A, (size_t)p * n)
    KEEP(h, h, m)
    KEEP(z, z, n)
    KEEP(lam, lam, m)
    KEEP(nu, nu, p)
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    s.valid = true;
    return 0;
}

}  // extern "C"

void fill_from_state(const QpBatchState& s, QpSolveArgs& a) {
    a.B = s.B; a.n = s.n; a.m = s.m; a.p = s.p;
    a.Q = s.Q.as<double>();
    a.G = s.m ? s.G.as<double>() : nullptr;
    a.A = s.p ? s.A.as<double>() : nullptr;
    a.h = s.h.as<double>(); a.z = s.z.as<double>(); a.lam = s.lam.as<double>(); a.nu = s.nu.as<double>();
}

extern "C" {

int32_t diffopt_b200_qp_batch_reverse(diffopt_b200_ctx* ctx, const double* dl_dz, double* rev_out, int32_t* info,
                                      int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!ctx->qp.valid) BAD_ARG(ctx, "qp_batch_reverse: call qp_batch_setup first");
    if (!dl_dz || !rev_out) BAD_ARG(ctx, "qp_batch_reverse: dl_dz and rev_out are required");
    if (ctx->qp.B == 0) return 0;
    QpSolveArgs a{};
    fill_from_state(ctx->qp, a);
    const void* ptr;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[13], dl_dz, sizeof(double) * a.B * a.n, memspace, &ptr));
    a.seed = (const double*)ptr;
    return qp_solve_common(ctx, a, nullptr, rev_out, info, memspace, false);
}

int32_t diffopt_b200_qp_batch_forward(diffopt_b200_ctx* ctx, const double* dQ, const double* dq, const double* dG,
                                      const double* dh, const double* dA, const double* db, double* fwd_out,
                                      int32_t* info, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!ctx->qp.valid) BAD_ARG(ctx, "qp_batch_forward: call qp_batch_setup first");
    if (!fwd_out) BAD_ARG(ctx, "qp_batch_forward: fwd_out is required");
    if (ctx->qp.B == 0) return 0;
    QpSolveArgs a{};
    fill_from_state(ctx->qp, a);
    const int64_t B = a.B;
    const int n = a.n, m = a.m, p = a.p;
    const size_t d = sizeof(double);
    const void* ptr;
    STAGE(7, dQ, dQ, (size_t)n * n)
    STAGE(8, dq, dq, n)
    STAGE(9, dG, dG, (size_t)m * n)
    STAGE(10, dh, dh, m)
    STAGE(11, dA, dA, (size_t)p * n)
    STAGE(12, db, db, p)
    return qp_solve_common(ctx, a, fwd_out, nullptr, info, memspace, false);
}

int32_t diffopt_b200_qp_batch_param_grads(diffopt_b200_ctx* ctx, const double* rev, int32_t reduce_over_batch,
                                          double* dQ, double* dq, double* dG, double* dh, double* dA, double* db,
                                          int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    QpBatchState& s = ctx->qp;
    if (!s.valid) BAD_ARG(ctx, "qp_batch_param_grads: call qp_batch_setup first");
    if (!rev) BAD_ARG(ctx, "qp_batch_param_grads: rev is required");
    if (s.B == 0) return 0;
    const int64_t B = s.B;
    const int n = s.n, m = s.m, p = s.p, N = n + m + p;
    const size_t d = sizeof(double);
    const int64_t mult = reduce_over_batch ? 1 : B;
    const void* drev;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[14], rev, d * B * N, memspace, &drev));
    double* outs[6] = {dQ, dq, dG, dh, dA, db};
    size_t cnt[6] = {(size_t)n * n, (size_t)n, (size_t)m * n, (size_t)m, (size_t)p * n, (size_t)p};
    void* dev[6];
    for (int i = 0; i < 6; ++i)
        DO_CUDA(ctx, stage_out_prepare(ctx->out[2 + i], outs[i], d * mult * cnt[i], memspace, &dev[i]));
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int32_t rc = qp_param_grads_launch(ctx, B, n, m, p, s.z.as<double>(), s.lam.as<double>(), s.nu.as<double>(),
                                       (const double*)drev, reduce_over_batch, (double*)dev[0], (double*)dev[1],
                                       (double*)dev[2], (double*)dev[3], (double*)dev[4], (double*)dev[5]);
    if (rc) return rc;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    for (int i = 0; i < 6; ++i) DO_CUDA(ctx, stage_out_finish(ctx, dev[i], outs[i], d * mult * cnt[i], memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}

}  // extern "C"
