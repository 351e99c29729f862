// Many sensitivity directions per call against the current conic_setup (diffopt_b200_conic_forward_multi /
// _reverse_multi): right-hand sides for k directions assembled on the device in the interleaved [group][N][KB] layout of
// lsqr_multi_kernel (lsqr.cu), one LSQR launch for all of them, outputs transposed back to the caller's [k][.] layout.
// Every sum is formed in a fixed order: direction j gives the same bits whatever the other directions hold.
#include <cmath>
#include <vector>

#include "lsqr.cuh"

namespace {

constexpr int CM_THREADS = 256;

// fixed-order CTA sum of v (every thread gets the total); red: CM_THREADS / 32 doubles
__device__ __forceinline__ double cm_block_sum(double v, double* red) {
    for (int q = 16; q > 0; q >>= 1) v += __shfl_xor_sync(0xffffffffu, v, q);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < CM_THREADS / 32; ++w) s += red[w];
    return s;
}

// Forward right-hand sides, rows 0 .. n+m-1 of g_j = [dA_j' vp + dc_j; -dA_j x + db_j]: entry r of direction j sums its
// gather list (gptr / gidx / gval, built on the host in triplet order: rows r < n read vp, the others -x) in order.
__global__ void __launch_bounds__(CM_THREADS) conic_fwd_rhs_multi_kernel(int n, int m, int k, int KB, const long long* __restrict__ gptr,
                                                                         const int* __restrict__ gidx, const double* __restrict__ gval,
                                                                         const double* __restrict__ db, const double* __restrict__ dc,
                                                                         const double* __restrict__ x, const double* __restrict__ vp,
                                                                         double* rhs) {
    const int R = n + m, N = R + 1;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < (long long)k * R; e += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(e / R), r = (int)(e - (long long)j * R);
        double t = 0.0;
        if (gptr)
            for (long long p = gptr[e]; p < gptr[e + 1]; ++p) t += r < n ? gval[p] * vp[gidx[p]] : -gval[p] * x[gidx[p]];
        if (r < n) {
            if (dc) t += dc[(size_t)j * n + r];
        } else if (db) {
            t += db[(size_t)j * m + (r - n)];
        }
        rhs[((size_t)(j / KB) * N + r) * KB + j % KB] = t;
    }
}

// One CTA per direction: last entry -dc_j'x - db_j'vp of the forward right-hand side and ||g_j||^2
__global__ void __launch_bounds__(CM_THREADS) conic_fwd_rhs_multi_finish(int n, int m, int KB, const double* __restrict__ db,
                                                                         const double* __restrict__ dc, const double* __restrict__ x,
                                                                         const double* __restrict__ vp, double* rhs, double* norm2) {
    __shared__ double red[CM_THREADS / 32];
    const int j = blockIdx.x, N = n + m + 1;
    double* g = rhs + (size_t)(j / KB) * N * KB + j % KB;
    double acc = 0.0;
    if (dc)
        for (int i = threadIdx.x; i < n; i += CM_THREADS) acc -= dc[(size_t)j * n + i] * x[i];
    if (db)
        for (int i = threadIdx.x; i < m; i += CM_THREADS) acc -= db[(size_t)j * m + i] * vp[i];
    const double last = cm_block_sum(acc, red);
    double nn = 0.0;
    for (int i = threadIdx.x; i < n + m; i += CM_THREADS) nn += g[(size_t)i * KB] * g[(size_t)i * KB];
    nn = cm_block_sum(nn, red);
    if (threadIdx.x == 0) {
        g[(size_t)(N - 1) * KB] = last;
        norm2[j] = nn + last * last;
    }
}

// One CTA per direction: reverse right-hand side [dx_j; 0; -x'dx_j] (ConicProgram.jl:363-367) and its squared norm
__global__ void __launch_bounds__(CM_THREADS) conic_rev_rhs_multi_kernel(int n, int m, int KB, const double* __restrict__ seeds,
                                                                         const double* __restrict__ x, double* rhs, double* norm2) {
    __shared__ double red[CM_THREADS / 32];
    const int j = blockIdx.x, N = n + m + 1;
    const double* dx = seeds + (size_t)j * n;
    double* g = rhs + (size_t)(j / KB) * N * KB + j % KB;
    double acc = 0.0, nn = 0.0;
    for (int i = threadIdx.x; i < n; i += CM_THREADS) {
        const double d = dx[i];
        g[(size_t)i * KB] = d;
        acc -= x[i] * d;
        nn += d * d;
    }
    for (int i = threadIdx.x; i < m; i += CM_THREADS) g[(size_t)(n + i) * KB] = 0.0;
    const double last = cm_block_sum(acc, red);
    nn = cm_block_sum(nn, red);
    if (threadIdx.x == 0) {
        g[(size_t)(N - 1) * KB] = last;
        norm2[j] = nn + last * last;
    }
}

// Outputs of direction blockIdx.y from its solution z (interleaved): forward dx = -(du - x dw) (:403-412) and dz; reverse
// g, dc = g[1:n] - g[N] x (:396-401), db = g[n+I] - g[N] vp (:414-428); the statistics.  Any output may be null.
__global__ void __launch_bounds__(CM_THREADS) conic_multi_out_kernel(int n, int m, int KB, const double* __restrict__ X,
                                                                     const double* __restrict__ st, const double* __restrict__ x,
                                                                     const double* __restrict__ vp, double* z_out, double* dx_out,
                                                                     double* dc_out, double* db_out, double* stats_out) {
    const int j = blockIdx.y, N = n + m + 1;
    const double* z = X + (size_t)(j / KB) * N * KB + j % KB;
    const double zN = z[(size_t)(N - 1) * KB];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double zi = z[(size_t)i * KB];
        if (z_out) z_out[(size_t)j * N + i] = zi;
        if (i < n) {
            if (dx_out) dx_out[(size_t)j * n + i] = -(zi - x[i] * zN);
            if (dc_out) dc_out[(size_t)j * n + i] = zi - zN * x[i];
        } else if (i < n + m) {
            if (db_out) db_out[(size_t)j * m + (i - n)] = zi - zN * vp[i - n];
        }
    }
    if (stats_out && blockIdx.x == 0 && threadIdx.x < 4)
        stats_out[(size_t)j * 4 + threadIdx.x] = st[((size_t)(j / KB) * KB + j % KB) * 4 + threadIdx.x];
}

// directions per group: 4 for a few directions, else 8
int multi_kb(int64_t k) { return k <= 4 ? 4 : 8; }

// right-hand-side, solution and scalar storage for G groups of KB directions
int32_t multi_buffers(diffopt_b200_ctx* ctx, int64_t N, int KB, int64_t G, double** rhs, double** X, double** norm2,
                      double** stats) {
    LsqrWork& l = ctx->lsqr;
    const size_t len = (size_t)G * KB * (size_t)N, d8 = sizeof(double);
    DO_CUDA(ctx, l.m_rhs.reserve(d8 * len));
    DO_CUDA(ctx, l.m_x.reserve(d8 * len));
    DO_CUDA(ctx, l.m_scal.reserve(d8 * (size_t)G * KB * 5));
    *rhs = l.m_rhs.as<double>();
    *X = l.m_x.as<double>();
    *norm2 = l.m_scal.as<double>();
    *stats = *norm2 + (size_t)G * KB;
    // directions beyond k (the last group's padding) keep a zero right-hand side: they fail the zero test
    DO_CUDA(ctx, cudaMemsetAsync(*rhs, 0, d8 * len, ctx->stream));
    DO_CUDA(ctx, cudaMemsetAsync(*norm2, 0, d8 * (size_t)G * KB, ctx->stream));
    return 0;
}

int32_t multi_finish(diffopt_b200_ctx* ctx, int64_t k, int KB, const double* X, const double* stats, double* z_out,
                     double* dx_out, double* dc_out, double* db_out, double* stats_out, int32_t memspace) {
    ConicState& S = ctx->conic;
    const int n = (int)S.n, m = (int)S.m, N = n + m + 1;
    const size_t d8 = sizeof(double), K = (size_t)k;
    void *dz, *ddx, *ddc, *ddb, *dst;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], z_out, d8 * K * N, memspace, &dz));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[1], dx_out, d8 * K * n, memspace, &ddx));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[2], dc_out, d8 * K * n, memspace, &ddc));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[3], db_out, d8 * K * m, memspace, &ddb));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[4], stats_out, d8 * K * 4, memspace, &dst));
    conic_multi_out_kernel<<<dim3((unsigned)((N + CM_THREADS - 1) / CM_THREADS), (unsigned)k), CM_THREADS, 0, ctx->stream>>>(
        n, m, KB, X, stats, S.x.as<double>(), S.vp.as<double>(), (double*)dz, (double*)ddx, (double*)ddc, (double*)ddb,
        (double*)dst);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    DO_CUDA(ctx, stage_out_finish(ctx, dz, z_out, d8 * K * N, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, ddx, dx_out, d8 * K * n, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, ddc, dc_out, d8 * K * n, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, ddb, db_out, d8 * K * m, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, dst, stats_out, d8 * K * 4, memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;  // ev0 / ev1 bracket the LSQR launches (lsqr_run_conic_multi)
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}

// Host copy of `bytes` at src (host or device memory per memspace)
int32_t host_view(diffopt_b200_ctx* ctx, const void* src, size_t bytes, int32_t memspace, std::vector<char>& tmp,
                  const void** out) {
    if (memspace == DIFFOPT_B200_HOST || bytes == 0) {
        *out = src;
        return 0;
    }
    tmp.resize(bytes);
    DO_CUDA(ctx, cudaMemcpy(tmp.data(), src, bytes, cudaMemcpyDeviceToHost));
    *out = tmp.data();
    return 0;
}

}  // namespace

extern "C" {

int32_t diffopt_b200_conic_forward_multi(diffopt_b200_ctx* ctx, int64_t k, const diffopt_b200_coo_batch* dA, const double* db,
                                         const double* dc, double atol, double btol, double conlim, int64_t maxiter,
                                         double* dx_out, double* dz_out, double* out_stats, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicState& S = ctx->conic;
    if (k < 0) BAD_ARG(ctx, "conic_forward_multi: k must be >= 0");
    if (!S.valid) BAD_ARG(ctx, "conic_forward_multi: call conic_setup first");
    if (k == 0) return 0;
    if (k > (int64_t)1 << 20) BAD_ARG(ctx, "conic_forward_multi: k too large");
    const int64_t n = S.n, m = S.m, N = n + m + 1, R = n + m;
    const size_t d8 = sizeof(double);
    // gather lists of the dA part: entry (j, r) lists the triplets of direction j in column r (r < n, times vp[row]) or
    // in row r - n (times -x[col]), each in triplet order (a stable counting sort: the sums have a fixed order)
    std::vector<long long> gptr;
    std::vector<int> gidx;
    std::vector<double> gval;
    if (dA && dA->ptr) {
        std::vector<char> t0, t1, t2, t3;
        const void *hp, *hi, *hj, *hv;
        if (int32_t rc = host_view(ctx, dA->ptr, sizeof(int64_t) * (size_t)(k + 1), memspace, t0, &hp)) return rc;
        const int64_t* ptr = (const int64_t*)hp;
        if (ptr[0] != 0) BAD_ARG(ctx, "conic_forward_multi: dA offsets must start at 0");
        for (int64_t j = 0; j < k; ++j)
            if (ptr[j + 1] < ptr[j]) BAD_ARG(ctx, "conic_forward_multi: dA offsets must be nondecreasing");
        const int64_t nnz = ptr[k];
        if (nnz > 0 && (!dA->I || !dA->J || !dA->V)) BAD_ARG(ctx, "conic_forward_multi: dA needs I, J and V");
        if (nnz > 1000000000LL) BAD_ARG(ctx, "conic_forward_multi: too many dA triplets");
        if (nnz > 0) {
            if (int32_t rc = host_view(ctx, dA->I, sizeof(int64_t) * (size_t)nnz, memspace, t1, &hi)) return rc;
            if (int32_t rc = host_view(ctx, dA->J, sizeof(int64_t) * (size_t)nnz, memspace, t2, &hj)) return rc;
            if (int32_t rc = host_view(ctx, dA->V, d8 * (size_t)nnz, memspace, t3, &hv)) return rc;
            const int64_t *I = (const int64_t*)hi, *J = (const int64_t*)hj;
            const double* V = (const double*)hv;
            for (int64_t p = 0; p < nnz; ++p)
                if (I[p] < 1 || I[p] > m || J[p] < 1 || J[p] > n)
                    BAD_ARG(ctx, "conic_forward_multi: a dA triplet lies outside the m x n matrix");
            const size_t E = (size_t)k * (size_t)R;
            gptr.assign(E + 1, 0);
            for (int64_t j = 0; j < k; ++j)
                for (int64_t p = ptr[j]; p < ptr[j + 1]; ++p) {
                    gptr[(size_t)j * R + (size_t)(J[p] - 1) + 1]++;
                    gptr[(size_t)j * R + (size_t)(n + I[p] - 1) + 1]++;
                }
            for (size_t e = 0; e < E; ++e) gptr[e + 1] += gptr[e];
            std::vector<long long> next(gptr.begin(), gptr.end() - 1);
            gidx.resize((size_t)2 * nnz);
            gval.resize((size_t)2 * nnz);
            for (int64_t j = 0; j < k; ++j)
                for (int64_t p = ptr[j]; p < ptr[j + 1]; ++p) {
                    const long long a = next[(size_t)j * R + (size_t)(J[p] - 1)]++;
                    gidx[(size_t)a] = (int)(I[p] - 1);
                    gval[(size_t)a] = V[p];
                    const long long b = next[(size_t)j * R + (size_t)(n + I[p] - 1)]++;
                    gidx[(size_t)b] = (int)(J[p] - 1);
                    gval[(size_t)b] = V[p];
                }
        }
    }
    const void *ddb, *ddc;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], db, d8 * (size_t)k * (size_t)m, memspace, &ddb));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[1], dc, d8 * (size_t)k * (size_t)n, memspace, &ddc));
    const long long* dgptr = nullptr;
    const int* dgidx = nullptr;
    const double* dgval = nullptr;
    if (!gptr.empty()) {
        const size_t bp = sizeof(long long) * gptr.size(), bv = d8 * gval.size(), bi = sizeof(int) * gidx.size();
        DO_CUDA(ctx, ctx->lsqr.m_gather.reserve(bp + bv + bi));
        char* base = ctx->lsqr.m_gather.as<char>();
        DO_CUDA(ctx, cudaMemcpyAsync(base, gptr.data(), bp, cudaMemcpyHostToDevice, ctx->stream));
        DO_CUDA(ctx, cudaMemcpyAsync(base + bp, gval.data(), bv, cudaMemcpyHostToDevice, ctx->stream));
        DO_CUDA(ctx, cudaMemcpyAsync(base + bp + bv, gidx.data(), bi, cudaMemcpyHostToDevice, ctx->stream));
        dgptr = (const long long*)base;
        dgval = (const double*)(base + bp);
        dgidx = (const int*)(base + bp + bv);
    }
    const int KB = multi_kb(k);
    const int64_t G = (k + KB - 1) / KB;
    double *rhs, *X, *norm2, *stats;
    if (int32_t rc = multi_buffers(ctx, N, KB, G, &rhs, &X, &norm2, &stats)) return rc;
    const int64_t E = k * R;
    const unsigned blocks = (unsigned)std::min<int64_t>((E + CM_THREADS - 1) / CM_THREADS, (int64_t)ctx->sm_count * 16);
    conic_fwd_rhs_multi_kernel<<<blocks, CM_THREADS, 0, ctx->stream>>>((int)n, (int)m, (int)k, KB, dgptr, dgidx, dgval,
                                                                       (const double*)ddb, (const double*)ddc, S.x.as<double>(),
                                                                       S.vp.as<double>(), rhs);
    conic_fwd_rhs_multi_finish<<<(unsigned)k, CM_THREADS, 0, ctx->stream>>>((int)n, (int)m, KB, (const double*)ddb,
                                                                            (const double*)ddc, S.x.as<double>(),
                                                                            S.vp.as<double>(), rhs, norm2);
    ctx->launches += 2;
    DO_CUDA(ctx, cudaGetLastError());
    LsqrParams prm{atol, btol, conlim, maxiter > 0 ? maxiter : N};
    // `norm(RHS) <= 1e-400` == `<= 0.0` (ConicProgram.jl:320)
    if (int32_t rc = lsqr_run_conic_multi(ctx, KB, G, rhs, norm2, 0.0, prm, X, stats)) return rc;
    // (gptr .. gval stay alive until multi_finish synchronises the stream)
    return multi_finish(ctx, k, KB, X, stats, dz_out, dx_out, nullptr, nullptr, out_stats, memspace);
}

int32_t diffopt_b200_conic_reverse_multi(diffopt_b200_ctx* ctx, int64_t k, const double* dx_seeds, double atol, double btol,
                                         double conlim, int64_t maxiter, double* g_out, double* dc_out, double* db_out,
                                         double* out_stats, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicState& S = ctx->conic;
    if (k < 0) BAD_ARG(ctx, "conic_reverse_multi: k must be >= 0");
    if (!S.valid) BAD_ARG(ctx, "conic_reverse_multi: call conic_setup first");
    if (k == 0) return 0;
    if (k > (int64_t)1 << 20) BAD_ARG(ctx, "conic_reverse_multi: k too large");
    if (!dx_seeds) BAD_ARG(ctx, "conic_reverse_multi: dx_seeds is required");
    const int64_t n = S.n, m = S.m, N = n + m + 1;
    const void* dseed;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], dx_seeds, sizeof(double) * (size_t)k * (size_t)n, memspace, &dseed));
    const int KB = multi_kb(k);
    const int64_t G = (k + KB - 1) / KB;
    double *rhs, *X, *norm2, *stats;
    if (int32_t rc = multi_buffers(ctx, N, KB, G, &rhs, &X, &norm2, &stats)) return rc;
    conic_rev_rhs_multi_kernel<<<(unsigned)k, CM_THREADS, 0, ctx->stream>>>((int)n, (int)m, KB, (const double*)dseed,
                                                                            S.x.as<double>(), rhs, norm2);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    LsqrParams prm{atol, btol, conlim, maxiter > 0 ? maxiter : N};
    if (int32_t rc = lsqr_run_conic_multi(ctx, KB, G, rhs, norm2, 1e-4 /* ConicProgram.jl:369 */, prm, X, stats)) return rc;
    return multi_finish(ctx, k, KB, X, stats, g_out, nullptr, dc_out, db_out, out_stats, memspace);
}

}  // extern "C"
