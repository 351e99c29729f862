// ConicProgram backend entry points (include/diffopt_b200.h): cone analysis (pi, Dpi data), PSD
// eigendecomposition (parallel cyclic Jacobi), forward / reverse differentiation via the persistent
// LSQR kernel on the matrix-free M, and the explicit-CSC LSQR used by the QP backend's LP branch.
#include <cmath>
#include <vector>

#include "exp_cone.cuh"
#include "pow_cone.cuh"
#include "lsqr.cuh"

ConicOpView conic_view(diffopt_b200_ctx* ctx, bool stream_blocks);

namespace {

// ---- diag rows (zero / nonneg cones): v = y - s, diag, vp ------------------------------------------
__global__ void cone_rows_kernel(int m, const double* __restrict__ y, const double* __restrict__ s,
                                 const signed char* __restrict__ kind, const signed char* __restrict__ rowtype,
                                 double* v, double* diag, double* vp) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        double vi = y[i] - s[i];
        v[i] = vi;
        if (kind[i] == 0) {
            if (rowtype[i] == DIFFOPT_CONE_ZERO) {   // dual of Zeros is the free cone: pi = id, Dpi = I
                diag[i] = 1.0;
                vp[i] = vi;
            } else {                                  // Nonnegatives: (sign(v)+1)/2, max(v,0)
                diag[i] = vi > 0.0 ? 1.0 : (vi < 0.0 ? 0.0 : 0.5);
                vp[i] = vi > 0.0 ? vi : 0.0;
            }
        } else {
            diag[i] = 0.0;
        }
    }
}

// ---- SOC cones: one warp per cone ------------------------------------------------------------------
__global__ void cone_soc_kernel(int nsoc, const int* __restrict__ off, const int* __restrict__ dim,
                                const double* __restrict__ v, int* cs, double* nxo, double* vp) {
    const int lane = threadIdx.x & 31;
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    for (int c = wid; c < nsoc; c += nw) {
        const int o = off[c], dd = dim[c];
        double acc = 0.0;
        for (int k = 1 + lane; k < dd; k += 32) acc += v[o + k] * v[o + k];
        for (int q = 16; q > 0; q >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, q);
        const double nx = sqrt(acc), t = v[o];
        int cas = nx <= t ? 0 : (nx <= -t ? 1 : 2);
        if (lane == 0) {
            cs[c] = cas;
            nxo[c] = nx;
        }
        const double scale = cas == 2 ? (nx + t) * 0.5 : 0.0;
        for (int k = lane; k < dd; k += 32) {
            double r;
            if (cas == 0) r = v[o + k];
            else if (cas == 1) r = 0.0;
            else r = (k == 0 ? 1.0 : v[o + k] / nx) * scale;
            vp[o + k] = r;
        }
    }
}

// ---- PSD cones: eigendecomposition, B and pi(v) live in psd_eig.cu ------------------------------------

__global__ void conic_fwd_rhs_kernel(int n, int m, long long nnz, const long long* __restrict__ rows,
                                     const long long* __restrict__ cols, const double* __restrict__ vals,
                                     const double* __restrict__ x, const double* __restrict__ vp, double* g) {
    // g[0:n] += dA' vp ; g[n:n+m] -= dA x     (atomic scatter; COO duplicates are summed)
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < nnz;
         k += (long long)gridDim.x * blockDim.x) {
        long long i = rows[k] - 1, j = cols[k] - 1;
        if (i < 0 || i >= m || j < 0 || j >= n) continue;
        double a = vals[k];
        atomicAdd(&g[j], a * vp[i]);
        atomicAdd(&g[n + i], -a * x[j]);
    }
}

__global__ void conic_fwd_rhs_finish(int n, int m, const double* __restrict__ db, const double* __restrict__ dc,
                                     const double* __restrict__ x, const double* __restrict__ vp, double* g,
                                     double* normsq) {
    // single CTA: add dc, db; last entry -dc'x - db'vp; ||g||^2
    __shared__ double red[32];
    __shared__ double s_last;
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double d = dc ? dc[i] : 0.0;
        g[i] += d;
        acc -= d * x[i];
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        double d = db ? db[i] : 0.0;
        g[n + i] += d;
        acc -= d * vp[i];
    }
    for (int q = 16; q > 0; q >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, q);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0;
        for (int w = 0; w < blockDim.x / 32; ++w) s += red[w];
        g[n + m] = s;
        s_last = s;
    }
    __syncthreads();
    double nn = 0.0;
    for (int i = threadIdx.x; i < n + m; i += blockDim.x) nn += g[i] * g[i];
    for (int q = 16; q > 0; q >>= 1) nn += __shfl_xor_sync(0xffffffffu, nn, q);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = nn;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = s_last * s_last;
        for (int w = 0; w < blockDim.x / 32; ++w) s += red[w];
        *normsq = s;
    }
}

__global__ void conic_rev_rhs_kernel(int n, int m, const double* __restrict__ dx, const double* __restrict__ x,
                                     double* dz, double* normsq) {
    // dz = [dx; 0; -x'dx]   (ConicProgram.jl:363-367 with dy = ds = 0)
    __shared__ double red[32], red2[32];
    double acc = 0.0, nn = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double d = dx[i];
        dz[i] = d;
        acc -= x[i] * d;
        nn += d * d;
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) dz[n + i] = 0.0;
    for (int q = 16; q > 0; q >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, q);
        nn += __shfl_xor_sync(0xffffffffu, nn, q);
    }
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = acc;
        red2[threadIdx.x >> 5] = nn;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0, t = 0;
        for (int w = 0; w < blockDim.x / 32; ++w) {
            s += red[w];
            t += red2[w];
        }
        dz[n + m] = s;
        *normsq = t + s * s;
    }
}

__global__ void conic_fwd_dx_kernel(int n, int m, const double* __restrict__ dz, const double* __restrict__ x, double* dx) {
    const double dw = dz[n + m];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        dx[i] = -(dz[i] - x[i] * dw);   // ConicProgram.jl:403-412
}

__global__ void conic_rev_getters_kernel(int n, int m, const double* __restrict__ g, const double* __restrict__ x,
                                         const double* __restrict__ vp, double* dc, double* db) {
    const double gN = g[n + m];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n + m; i += gridDim.x * blockDim.x) {
        if (i < n) {
            if (dc) dc[i] = g[i] - gN * x[i];            // :396-401
        } else if (db) {
            db[i - n] = g[i] - gN * vp[i - n];           // :414-428
        }
    }
}

// ---- lock-step batch (diffopt_b200_conic_batch_*) ----------------------------------------------------------------
// Per-problem pointers the batched right-hand-side / getter kernels need (the operator itself travels as OpArgs).
struct ConicBatchPtrs {
    const double* x;
    const double* vp;
};

// One CTA per problem: rhs_p = [dx_p; 0; -x_p'dx_p]  (ConicProgram.jl:363-367 with dy = ds = 0) at the head of the
// problem's work region; the norm test of :369 is made by the LSQR kernel itself (zero_below).
__global__ void conic_rev_rhs_batch_kernel(int n, int m, const double* __restrict__ seeds, const ConicBatchPtrs* __restrict__ pp,
                                           double* work, size_t stride) {
    __shared__ double red[32];
    const int p = blockIdx.x;
    const double* dx = seeds + (size_t)p * n;
    const double* x = pp[p].x;
    double* dz = work + (size_t)p * stride;
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double d = dx[i];
        dz[i] = d;
        acc -= x[i] * d;
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) dz[n + i] = 0.0;
    for (int q = 16; q > 0; q >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, q);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0;
        for (int w = 0; w < blockDim.x / 32; ++w) s += red[w];
        dz[n + m] = s;
    }
}

// g_p (the problem's x region), getters dc_p = g[1:n] - g[N] x, db_p = g[n+I] - g[N] vp (:396-428) and the LSQR
// statistics, gathered into the caller's instance-major arrays.
__global__ void conic_rev_out_batch_kernel(int n, int m, const ConicBatchPtrs* __restrict__ pp, const double* __restrict__ work,
                                           LsqrBatchLayout L, double* g_out, double* dc, double* db, double* stats) {
    const int p = blockIdx.y;
    const int N = n + m + 1;
    const double* g = work + (size_t)p * L.stride + L.x;
    const double gN = g[n + m];
    const double* x = pp[p].x;
    const double* vp = pp[p].vp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double gi = g[i];
        if (g_out) g_out[(size_t)p * N + i] = gi;
        if (i < n) {
            if (dc) dc[(size_t)p * n + i] = gi - gN * x[i];
        } else if (i < n + m) {
            if (db) db[(size_t)p * m + (i - n)] = gi - gN * vp[i - n];
        }
    }
    if (stats && blockIdx.x == 0 && threadIdx.x < 4)
        stats[(size_t)p * 4 + threadIdx.x] = work[(size_t)p * L.stride + L.stats + threadIdx.x];
}

int32_t to_host_copy(diffopt_b200_ctx* ctx, const void* src, size_t bytes, int memspace, std::vector<char>& tmp,
                     const void** host) {
    if (memspace == DIFFOPT_B200_HOST) {
        *host = src;
        return 0;
    }
    tmp.resize(bytes);
    DO_CUDA(ctx, cudaMemcpy(tmp.data(), src, bytes, cudaMemcpyDeviceToHost));
    *host = tmp.data();
    return 0;
}

}  // namespace

extern "C" {

int32_t diffopt_b200_lsqr_csc(diffopt_b200_ctx* ctx, int64_t nrows, int64_t ncols, const int64_t* colptr,
                              const int64_t* rowval, const double* nzval, int32_t trans, const double* rhs,
                              double atol, double btol, double conlim, int64_t maxiter, double* x_out,
                              double* out_stats, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!colptr || !rowval || !nzval || !rhs || !x_out) BAD_ARG(ctx, "lsqr_csc: null argument");
    std::vector<char> t0, t1, t2;
    const void *hc, *hr, *hv;
    if (int32_t rc = to_host_copy(ctx, colptr, sizeof(int64_t) * (size_t)(ncols + 1), memspace, t0, &hc)) return rc;
    const int64_t nnz = ((const int64_t*)hc)[ncols] - 1;
    if (int32_t rc = to_host_copy(ctx, rowval, sizeof(int64_t) * (size_t)nnz, memspace, t1, &hr)) return rc;
    if (int32_t rc = to_host_copy(ctx, nzval, sizeof(double) * (size_t)nnz, memspace, t2, &hv)) return rc;
    if (int32_t rc = csr_from_csc_host(ctx, nrows, ncols, (const int64_t*)hc, (const int64_t*)hr, (const double*)hv,
                                       ctx->lsqr_mat))
        return rc;
    const int64_t rlen = trans ? ncols : nrows, xlen = trans ? nrows : ncols;
    const void* drhs;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], rhs, sizeof(double) * (size_t)rlen, memspace, &drhs));
    void* dx;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], x_out, sizeof(double) * (size_t)xlen, memspace, &dx));
    LsqrParams prm{atol, btol, conlim, maxiter > 0 ? maxiter : (nrows > ncols ? nrows : ncols)};
    double st[7];
    if (int32_t rc = lsqr_run_csr(ctx, ctx->lsqr_mat, trans != 0, (const double*)drhs, prm, (double*)dx, st)) return rc;
    DO_CUDA(ctx, stage_out_finish(ctx, dx, x_out, sizeof(double) * (size_t)xlen, memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (out_stats) {
        if (memspace == DIFFOPT_B200_HOST) memcpy(out_stats, st, sizeof(double) * 4);
        else DO_CUDA(ctx, cudaMemcpy(out_stats, st, sizeof(double) * 4, cudaMemcpyHostToDevice));
    }
    return 0;
}

}  // extern "C"

namespace {

// conic_setup and conic_setup_ex: cone_param (one exponent per cone, read for power cones) may be NULL when the list
// has no power cone.
int32_t conic_setup_impl(diffopt_b200_ctx* ctx, int64_t n, int64_t m, const int64_t* A_colptr, const int64_t* A_rowval,
                         const double* A_nzval, const double* b, const double* c, const double* x, const double* s,
                         const double* y, int64_t ncones, const int32_t* cone_type, const int64_t* cone_dim,
                         const double* cone_param, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicState& S = ctx->conic;
    S.valid = false;
    if (n <= 0 || m < 0 || ncones < 0) BAD_ARG(ctx, "conic_setup: bad sizes");
    if (!A_colptr || !b || !c || !x || !s || !y || (ncones > 0 && (!cone_type || !cone_dim)))
        BAD_ARG(ctx, "conic_setup: null argument");
    std::vector<char> t0, t1, t2, t3, t4, t5;
    const void *hc, *hr, *hv, *hct, *hcd, *hcp = nullptr;
    if (int32_t rc = to_host_copy(ctx, A_colptr, sizeof(int64_t) * (size_t)(n + 1), memspace, t0, &hc)) return rc;
    const int64_t nnz = ((const int64_t*)hc)[n] - 1;
    if (int32_t rc = to_host_copy(ctx, A_rowval, sizeof(int64_t) * (size_t)nnz, memspace, t1, &hr)) return rc;
    if (int32_t rc = to_host_copy(ctx, A_nzval, sizeof(double) * (size_t)nnz, memspace, t2, &hv)) return rc;
    if (int32_t rc = to_host_copy(ctx, cone_type, sizeof(int32_t) * (size_t)ncones, memspace, t3, &hct)) return rc;
    if (int32_t rc = to_host_copy(ctx, cone_dim, sizeof(int64_t) * (size_t)ncones, memspace, t4, &hcd)) return rc;
    if (cone_param && ncones > 0)
        if (int32_t rc = to_host_copy(ctx, cone_param, sizeof(double) * (size_t)ncones, memspace, t5, &hcp)) return rc;
    const int32_t* ct = (const int32_t*)hct;
    const int64_t* cd = (const int64_t*)hcd;
    const double* cp = (const double*)hcp;
    // cone bookkeeping (host): row kinds and per-cone index lists
    std::vector<signed char> kind((size_t)m, 0), rowtype((size_t)m, 0);
    std::vector<int> soc_off, soc_dim, psd_off, psd_d, exp_off, pow_off;
    std::vector<signed char> exp_neg, pow_neg;
    std::vector<double> pow_alpha;
    std::vector<long long> psd_uoff;
    int64_t row = 0, sumd2 = 0, maxd = 0;
    for (int64_t k = 0; k < ncones; ++k) {
        const int64_t dim = cd[k];
        if (dim < 0 || row + dim > m) BAD_ARG(ctx, "conic_setup: cone dimensions exceed the number of rows");
        switch (ct[k]) {
            case DIFFOPT_CONE_ZERO:
            case DIFFOPT_CONE_NONNEG:
                for (int64_t i = 0; i < dim; ++i) rowtype[(size_t)(row + i)] = (signed char)ct[k];
                break;
            case DIFFOPT_CONE_SOC:
                if (dim < 1) BAD_ARG(ctx, "conic_setup: SOC dimension must be >= 1");
                for (int64_t i = 0; i < dim; ++i) kind[(size_t)(row + i)] = 2;
                soc_off.push_back((int)row);
                soc_dim.push_back((int)dim);
                break;
            case DIFFOPT_CONE_PSD: {
                int64_t d = (int64_t)((std::sqrt(8.0 * (double)dim + 1.0) - 1.0) / 2.0 + 0.5);
                if (d * (d + 1) / 2 != dim) BAD_ARG(ctx, "conic_setup: PSD triangle length must be d(d+1)/2");
                if (d > 1024) BAD_ARG(ctx, "conic_setup: PSD side > 1024 not supported");
                for (int64_t i = 0; i < dim; ++i) kind[(size_t)(row + i)] = 3;
                psd_off.push_back((int)row);
                psd_d.push_back((int)d);
                psd_uoff.push_back(sumd2);
                sumd2 += d * d;
                maxd = d > maxd ? d : maxd;
            } break;
            case DIFFOPT_CONE_EXP:
            case DIFFOPT_CONE_DUAL_EXP:
                if (dim != 3) BAD_ARG(ctx, "conic_setup: exponential cone dimension must be 3");
                for (int64_t i = 0; i < 3; ++i) kind[(size_t)(row + i)] = (signed char)(4 + i);
                exp_off.push_back((int)row);
                exp_neg.push_back(ct[k] == DIFFOPT_CONE_EXP ? 1 : 0);
                break;
            case DIFFOPT_CONE_POW:
            case DIFFOPT_CONE_DUAL_POW: {
                if (dim != 3) BAD_ARG(ctx, "conic_setup: power cone dimension must be 3");
                if (!cp) BAD_ARG(ctx, "conic_setup: power cones need their exponents: call conic_setup_ex with cone_param");
                const double a = cp[k];
                if (!(std::isfinite(a) && a > 0.0 && a < 1.0))
                    BAD_ARG(ctx, "conic_setup: power cone exponent must be finite and in (0, 1)");
                for (int64_t i = 0; i < 3; ++i) kind[(size_t)(row + i)] = (signed char)(4 + i);
                pow_off.push_back((int)row);
                pow_neg.push_back(ct[k] == DIFFOPT_CONE_POW ? 1 : 0);
                pow_alpha.push_back(a);
            } break;
            default:
                BAD_ARG(ctx, "conic_setup: unknown cone type");
        }
        row += dim;
    }
    if (row != m) BAD_ARG(ctx, "conic_setup: cone dimensions do not add up to m");
    S.n = n; S.m = m; S.ncones = ncones;
    S.nsoc = (int64_t)soc_off.size();
    S.npsd = (int64_t)psd_off.size();
    S.nexp = (int64_t)exp_off.size();
    S.npow = (int64_t)pow_off.size();
    S.psd_sumd2 = sumd2;
    S.psd_maxd = maxd;
    if (int32_t rc = csr_from_csc_host(ctx, m, n, (const int64_t*)hc, (const int64_t*)hr, (const double*)hv, S.A))
        return rc;
    const size_t d8 = sizeof(double);
    cudaMemcpyKind kd = memspace == DIFFOPT_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    auto keep = [&](DevBuf& buf, const void* src, size_t bytes, cudaMemcpyKind k) -> cudaError_t {
        cudaError_t e = buf.reserve(bytes ? bytes : 8);
        if (e != cudaSuccess || bytes == 0) return e;
        return cudaMemcpyAsync(buf.ptr, src, bytes, k, ctx->stream);
    };
    DO_CUDA(ctx, keep(S.b, b, d8 * m, kd));
    DO_CUDA(ctx, keep(S.c, c, d8 * n, kd));
    DO_CUDA(ctx, keep(S.x, x, d8 * n, kd));
    DO_CUDA(ctx, keep(S.s, s, d8 * m, kd));
    DO_CUDA(ctx, keep(S.y, y, d8 * m, kd));
    DO_CUDA(ctx, keep(S.row_kind, kind.data(), (size_t)m, cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(ctx->in[15], rowtype.data(), (size_t)m, cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.soc_off, soc_off.data(), sizeof(int) * soc_off.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.soc_dim, soc_dim.data(), sizeof(int) * soc_dim.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.psd_off, psd_off.data(), sizeof(int) * psd_off.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.psd_d, psd_d.data(), sizeof(int) * psd_d.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.psd_uoff, psd_uoff.data(), sizeof(long long) * psd_uoff.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.exp_off, exp_off.data(), sizeof(int) * exp_off.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.exp_neg, exp_neg.data(), exp_neg.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.pow_off, pow_off.data(), sizeof(int) * pow_off.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.pow_neg, pow_neg.data(), pow_neg.size(), cudaMemcpyHostToDevice));
    DO_CUDA(ctx, keep(S.pow_alpha, pow_alpha.data(), d8 * pow_alpha.size(), cudaMemcpyHostToDevice));
    // (blk3 holds 3 coefficients for every row when any cone has a 3 x 3 block: exponential or power)
    DO_CUDA(ctx, S.blk3.reserve(exp_off.empty() && pow_off.empty() ? 8 : d8 * 3 * (size_t)m));
    {   // flattened list of 32 x 32 output tiles of the PSD apply
        std::vector<int> toff(psd_d.size() + 1, 0);
        for (size_t k = 0; k < psd_d.size(); ++k) {
            const int nt = (psd_d[k] + 31) / 32;
            toff[k + 1] = toff[k] + nt * nt;
        }
        S.psd_ntiles = toff.back();
        DO_CUDA(ctx, keep(S.psd_toff, toff.data(), sizeof(int) * toff.size(), cudaMemcpyHostToDevice));
    }
    DO_CUDA(ctx, S.v.reserve(d8 * (m ? m : 1)));
    DO_CUDA(ctx, S.vp.reserve(d8 * (m ? m : 1)));
    DO_CUDA(ctx, S.nn_scale.reserve(d8 * (m ? m : 1)));
    DO_CUDA(ctx, S.soc_case.reserve(sizeof(int) * (soc_off.size() + 1)));
    DO_CUDA(ctx, S.soc_nx.reserve(d8 * (soc_off.size() + 1)));
    DO_CUDA(ctx, S.psd_U.reserve(d8 * (size_t)(sumd2 + 1)));
    DO_CUDA(ctx, S.psd_Bm.reserve(d8 * (size_t)(sumd2 + 1)));
    DO_CUDA(ctx, S.psd_ident.reserve(sizeof(int) * (psd_off.size() + 1)));
    DO_CUDA(ctx, S.psd_work.reserve(d8 * (size_t)(3 * sumd2 + 1)));
    DO_CUDA(ctx, S.w1.reserve(d8 * (size_t)(2 * m + 2)));
    DO_CUDA(ctx, S.w2.reserve(d8 * (size_t)(n + m + 2)));
    DO_CUDA(ctx, S.w3.reserve(d8 * (size_t)(n + m + 2)));
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (m > 0) {
        int blocks = (int)((m + 255) / 256);
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        cone_rows_kernel<<<blocks, 256, 0, ctx->stream>>>((int)m, S.y.as<double>(), S.s.as<double>(),
                                                           S.row_kind.as<signed char>(), ctx->in[15].as<signed char>(),
                                                           S.v.as<double>(), S.nn_scale.as<double>(), S.vp.as<double>());
        ctx->launches++;
    }
    if (S.nsoc > 0) {
        int blocks = (int)((S.nsoc * 32 + 255) / 256);
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        cone_soc_kernel<<<blocks, 256, 0, ctx->stream>>>((int)S.nsoc, S.soc_off.as<int>(), S.soc_dim.as<int>(),
                                                          S.v.as<double>(), S.soc_case.as<int>(), S.soc_nx.as<double>(),
                                                          S.vp.as<double>());
        ctx->launches++;
    }
    if (S.nexp > 0) {
        int blocks = (int)((S.nexp + 127) / 128);
        if (blocks > ctx->sm_count * 16) blocks = ctx->sm_count * 16;
        cone_exp_kernel<<<blocks, 128, 0, ctx->stream>>>((int)S.nexp, S.exp_off.as<int>(), S.exp_neg.as<signed char>(),
                                                          S.v.as<double>(), S.vp.as<double>(), S.blk3.as<double>(), nullptr);
        ctx->launches++;
    }
    if (S.npow > 0) {
        int blocks = (int)((S.npow + 127) / 128);
        if (blocks > ctx->sm_count * 16) blocks = ctx->sm_count * 16;
        cone_pow_kernel<<<blocks, 128, 0, ctx->stream>>>((int)S.npow, S.pow_off.as<int>(), S.pow_neg.as<signed char>(),
                                                          S.pow_alpha.as<double>(), S.v.as<double>(), S.vp.as<double>(),
                                                          S.blk3.as<double>(), nullptr);
        ctx->launches++;
    }
    if (S.npsd > 0)
        if (int32_t rc = psd_eig_launch(ctx, psd_d, psd_uoff, psd_off)) return rc;
    DO_CUDA(ctx, cudaGetLastError());
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    S.valid = true;
    return 0;
}

}  // namespace

extern "C" {

int32_t diffopt_b200_conic_setup(diffopt_b200_ctx* ctx, int64_t n, int64_t m, const int64_t* A_colptr,
                                 const int64_t* A_rowval, const double* A_nzval, const double* b, const double* c,
                                 const double* x, const double* s, const double* y, int64_t ncones,
                                 const int32_t* cone_type, const int64_t* cone_dim, int32_t memspace) {
    return conic_setup_impl(ctx, n, m, A_colptr, A_rowval, A_nzval, b, c, x, s, y, ncones, cone_type, cone_dim, nullptr,
                            memspace);
}

int32_t diffopt_b200_conic_setup_ex(diffopt_b200_ctx* ctx, int64_t n, int64_t m, const int64_t* A_colptr,
                                    const int64_t* A_rowval, const double* A_nzval, const double* b, const double* c,
                                    const double* x, const double* s, const double* y, int64_t ncones,
                                    const int32_t* cone_type, const int64_t* cone_dim, const double* cone_param,
                                    int32_t memspace) {
    return conic_setup_impl(ctx, n, m, A_colptr, A_rowval, A_nzval, b, c, x, s, y, ncones, cone_type, cone_dim,
                            cone_param, memspace);
}

int32_t diffopt_b200_conic_get_vp(diffopt_b200_ctx* ctx, double* vp_out, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!ctx->conic.valid) BAD_ARG(ctx, "conic_get_vp: call conic_setup first");
    if (!vp_out) BAD_ARG(ctx, "conic_get_vp: null output");
    DO_CUDA(ctx, cudaMemcpyAsync(vp_out, ctx->conic.vp.ptr, sizeof(double) * (size_t)ctx->conic.m,
                                 memspace == DIFFOPT_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                                 ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int32_t conic_op_call(diffopt_b200_ctx* ctx, const double* t, int32_t transpose, double* out, int32_t memspace,
                             bool full_M) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicState& S = ctx->conic;
    if (!S.valid) BAD_ARG(ctx, "conic operator: call conic_setup first");
    if (!t || !out) BAD_ARG(ctx, "conic operator: null argument");
    const size_t len = (size_t)(full_M ? S.n + S.m + 1 : S.m);
    const void* dt;
    void* dout;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], t, sizeof(double) * len, memspace, &dt));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], out, sizeof(double) * len, memspace, &dout));
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int32_t rc = full_M ? conic_apply_M(ctx, (const double*)dt, transpose != 0, (double*)dout)
                        : conic_apply_dpi(ctx, (const double*)dt, transpose != 0, (double*)dout);
    if (rc) return rc;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, stage_out_finish(ctx, dout, out, sizeof(double) * len, memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}

int32_t diffopt_b200_conic_dpi_apply(diffopt_b200_ctx* ctx, const double* t, int32_t transpose, double* out,
                                     int32_t memspace) {
    return conic_op_call(ctx, t, transpose, out, memspace, false);
}

int32_t diffopt_b200_conic_M_apply(diffopt_b200_ctx* ctx, const double* t, int32_t transpose, double* out,
                                   int32_t memspace) {
    return conic_op_call(ctx, t, transpose, out, memspace, true);
}

int32_t diffopt_b200_conic_forward(diffopt_b200_ctx* ctx, int64_t dA_nnz, const int64_t* dA_row, const int64_t* dA_col,
                                   const double* dA_val, const double* db, const double* dc, double atol, double btol,
                                   double conlim, int64_t maxiter, double* dx_out, double* dz_out, double* out_stats,
                                   int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicState& S = ctx->conic;
    if (!S.valid) BAD_ARG(ctx, "conic_forward: call conic_setup first");
    if (dA_nnz < 0 || (dA_nnz > 0 && (!dA_row || !dA_col || !dA_val))) BAD_ARG(ctx, "conic_forward: bad dA triplets");
    const int n = (int)S.n, m = (int)S.m, N = n + m + 1;
    const size_t d8 = sizeof(double);
    const void *drow, *dcol, *dval, *ddb, *ddc;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], dA_row, sizeof(int64_t) * (size_t)dA_nnz, memspace, &drow));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[1], dA_col, sizeof(int64_t) * (size_t)dA_nnz, memspace, &dcol));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[2], dA_val, d8 * (size_t)dA_nnz, memspace, &dval));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[3], db, d8 * (size_t)m, memspace, &ddb));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[4], dc, d8 * (size_t)n, memspace, &ddc));
    double* g = S.w2.as<double>();
    double* dz = S.w3.as<double>();
    DO_CUDA(ctx, cudaMemsetAsync(g, 0, d8 * (size_t)(N + 1), ctx->stream));
    if (dA_nnz > 0) {
        int blocks = (int)((dA_nnz + 255) / 256);
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        conic_fwd_rhs_kernel<<<blocks, 256, 0, ctx->stream>>>(n, m, (long long)dA_nnz, (const long long*)drow,
                                                               (const long long*)dcol, (const double*)dval,
                                                               S.x.as<double>(), S.vp.as<double>(), g);
        ctx->launches++;
    }
    conic_fwd_rhs_finish<<<1, 1024, 0, ctx->stream>>>(n, m, (const double*)ddb, (const double*)ddc, S.x.as<double>(),
                                                      S.vp.as<double>(), g, g + N);
    ctx->launches++;
    double normsq = 0.0;
    DO_CUDA(ctx, cudaMemcpyAsync(&normsq, g + N, d8, cudaMemcpyDeviceToHost, ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    double st[7] = {0, 0, 0, 0, 0, 0, 0};
    if (std::sqrt(normsq) <= 0.0) {                       // `norm(RHS) <= 1e-400` == `<= 0.0` (ConicProgram.jl:320)
        DO_CUDA(ctx, cudaMemsetAsync(dz, 0, d8 * (size_t)N, ctx->stream));
    } else {
        LsqrParams prm{atol, btol, conlim, maxiter > 0 ? maxiter : (int64_t)N};
        if (int32_t rc = lsqr_run_conic(ctx, g, prm, dz, st)) return rc;
    }
    if (dx_out) {
        void* ddx;
        DO_CUDA(ctx, stage_out_prepare(ctx->out[0], dx_out, d8 * (size_t)n, memspace, &ddx));
        conic_fwd_dx_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n, m, dz, S.x.as<double>(), (double*)ddx);
        ctx->launches++;
        DO_CUDA(ctx, stage_out_finish(ctx, ddx, dx_out, d8 * (size_t)n, memspace));
    }
    if (dz_out)
        DO_CUDA(ctx, cudaMemcpyAsync(dz_out, dz, d8 * (size_t)N,
                                     memspace == DIFFOPT_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                                     ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (out_stats) {
        if (memspace == DIFFOPT_B200_HOST) memcpy(out_stats, st, d8 * 4);
        else DO_CUDA(ctx, cudaMemcpy(out_stats, st, d8 * 4, cudaMemcpyHostToDevice));
    }
    return 0;
}

int32_t diffopt_b200_conic_reverse(diffopt_b200_ctx* ctx, const double* dx_seed, double atol, double btol,
                                   double conlim, int64_t maxiter, double* g_out, double* dc_out, double* db_out,
                                   double* out_stats, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicState& S = ctx->conic;
    if (!S.valid) BAD_ARG(ctx, "conic_reverse: call conic_setup first");
    if (!dx_seed) BAD_ARG(ctx, "conic_reverse: dx_seed is required");
    const int n = (int)S.n, m = (int)S.m, N = n + m + 1;
    const size_t d8 = sizeof(double);
    const void* dseed;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], dx_seed, d8 * (size_t)n, memspace, &dseed));
    double* dz = S.w2.as<double>();
    double* g = S.w3.as<double>();
    conic_rev_rhs_kernel<<<1, 1024, 0, ctx->stream>>>(n, m, (const double*)dseed, S.x.as<double>(), dz, dz + N);
    ctx->launches++;
    double normsq = 0.0;
    DO_CUDA(ctx, cudaMemcpyAsync(&normsq, dz + N, d8, cudaMemcpyDeviceToHost, ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    double st[7] = {0, 0, 0, 0, 0, 0, 0};
    if (std::sqrt(normsq) <= 1e-4) {                       // ConicProgram.jl:369
        DO_CUDA(ctx, cudaMemsetAsync(g, 0, d8 * (size_t)N, ctx->stream));
    } else {
        LsqrParams prm{atol, btol, conlim, maxiter > 0 ? maxiter : (int64_t)N};
        if (int32_t rc = lsqr_run_conic(ctx, dz, prm, g, st)) return rc;
    }
    void *ddc, *ddb;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], dc_out, d8 * (size_t)n, memspace, &ddc));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[1], db_out, d8 * (size_t)m, memspace, &ddb));
    if (dc_out || db_out) {
        int blocks = (N + 255) / 256;
        conic_rev_getters_kernel<<<blocks, 256, 0, ctx->stream>>>(n, m, g, S.x.as<double>(), S.vp.as<double>(),
                                                                   (double*)ddc, (double*)ddb);
        ctx->launches++;
    }
    DO_CUDA(ctx, stage_out_finish(ctx, ddc, dc_out, d8 * (size_t)n, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, ddb, db_out, d8 * (size_t)m, memspace));
    if (g_out)
        DO_CUDA(ctx, cudaMemcpyAsync(g_out, g, d8 * (size_t)N,
                                     memspace == DIFFOPT_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                                     ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (out_stats) {
        if (memspace == DIFFOPT_B200_HOST) memcpy(out_stats, st, d8 * 4);
        else DO_CUDA(ctx, cudaMemcpy(out_stats, st, d8 * 4, cudaMemcpyHostToDevice));
    }
    return 0;
}

}  // extern "C"

// Problems of a lock-step batch (every one a full conic_setup state) and the launch's work area.
struct ConicBatchImpl {
    std::vector<ConicState> states;
    int64_t B = 0, n = 0, m = 0;
    int C = 1;
    DevBuf work, ops, vecs, rhs, ptrs;
};

void conic_batch_release(diffopt_b200_ctx* ctx) {
    ConicBatchImpl* b = ctx->conic_batch;
    if (!b) return;
    for (ConicState& s : b->states) conic_state_release(s);
    for (DevBuf* d : {&b->work, &b->ops, &b->vecs, &b->rhs, &b->ptrs}) d->release();
    delete b;
    ctx->conic_batch = nullptr;
}

extern "C" {

int32_t diffopt_b200_conic_batch_begin(diffopt_b200_ctx* ctx, int64_t B, int32_t ctas_per_problem) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (B <= 0) BAD_ARG(ctx, "conic_batch_begin: the batch must hold at least one problem");
    if (ctas_per_problem < 0 || ctas_per_problem > 16) BAD_ARG(ctx, "conic_batch_begin: ctas_per_problem must be 0 (default) .. 16");
    conic_batch_release(ctx);
    ctx->conic_batch = new ConicBatchImpl();
    ctx->conic_batch->B = B;
    ctx->conic_batch->C = ctas_per_problem > 0 ? ctas_per_problem : 1;
    ctx->conic_batch->states.reserve((size_t)B);
    return 0;
}

}  // extern "C"

namespace {

int32_t conic_batch_add_impl(diffopt_b200_ctx* ctx, int64_t n, int64_t m, const int64_t* A_colptr,
                             const int64_t* A_rowval, const double* A_nzval, const double* b, const double* c,
                             const double* x, const double* s, const double* y, int64_t ncones,
                             const int32_t* cone_type, const int64_t* cone_dim, const double* cone_param,
                             int32_t memspace) {
    if (!ctx) return -1;
    ConicBatchImpl* bt = ctx->conic_batch;
    if (!bt) BAD_ARG(ctx, "conic_batch_add: call conic_batch_begin first");
    if ((int64_t)bt->states.size() >= bt->B) BAD_ARG(ctx, "conic_batch_add: the batch is full");
    if (!bt->states.empty() && (n != bt->n || m != bt->m))
        BAD_ARG(ctx, "conic_batch_add: every problem of a batch must have the same n and m");
    // the single-problem state is parked while this problem is analysed by the ordinary setup, with the row blocks of
    // its CSR copies cut for the CTAs one problem gets in the batched kernel
    ConicState parked = ctx->conic;
    ctx->conic = ConicState{};
    const int prev_ctas = ctx->csr_cluster_ctas;
    ctx->csr_cluster_ctas = bt->C;
    int32_t rc = conic_setup_impl(ctx, n, m, A_colptr, A_rowval, A_nzval, b, c, x, s, y, ncones, cone_type, cone_dim,
                                  cone_param, memspace);
    ctx->csr_cluster_ctas = prev_ctas;
    ConicState fresh = ctx->conic;
    ctx->conic = parked;
    if (rc == 0 && fresh.npsd > 0) {
        ctx->err = "conic_batch_add: problems with PSD cones are not batched (use conic_setup / conic_reverse)";
        rc = -1;
    }
    if (rc) {
        conic_state_release(fresh);
        return rc;
    }
    bt->n = n;
    bt->m = m;
    bt->states.push_back(fresh);
    return 0;
}

}  // namespace

extern "C" {

int32_t diffopt_b200_conic_batch_add(diffopt_b200_ctx* ctx, int64_t n, int64_t m, const int64_t* A_colptr,
                                     const int64_t* A_rowval, const double* A_nzval, const double* b, const double* c,
                                     const double* x, const double* s, const double* y, int64_t ncones,
                                     const int32_t* cone_type, const int64_t* cone_dim, int32_t memspace) {
    return conic_batch_add_impl(ctx, n, m, A_colptr, A_rowval, A_nzval, b, c, x, s, y, ncones, cone_type, cone_dim,
                                nullptr, memspace);
}

int32_t diffopt_b200_conic_batch_add_ex(diffopt_b200_ctx* ctx, int64_t n, int64_t m, const int64_t* A_colptr,
                                        const int64_t* A_rowval, const double* A_nzval, const double* b, const double* c,
                                        const double* x, const double* s, const double* y, int64_t ncones,
                                        const int32_t* cone_type, const int64_t* cone_dim, const double* cone_param,
                                        int32_t memspace) {
    return conic_batch_add_impl(ctx, n, m, A_colptr, A_rowval, A_nzval, b, c, x, s, y, ncones, cone_type, cone_dim,
                                cone_param, memspace);
}

int32_t diffopt_b200_conic_batch_reverse(diffopt_b200_ctx* ctx, const double* dx_seeds, double atol, double btol,
                                         double conlim, int64_t maxiter, double* g_out, double* dc_out, double* db_out,
                                         double* out_stats, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    ConicBatchImpl* bt = ctx->conic_batch;
    if (!bt || (int64_t)bt->states.size() != bt->B) BAD_ARG(ctx, "conic_batch_reverse: the batch is not complete (conic_batch_add)");
    if (!dx_seeds) BAD_ARG(ctx, "conic_batch_reverse: dx_seeds is required");
    const int n = (int)bt->n, m = (int)bt->m, N = n + m + 1, C = bt->C;
    const int64_t B = bt->B;
    const size_t d8 = sizeof(double);
    const LsqrBatchLayout L(N, C);
    DO_CUDA(ctx, bt->work.reserve(d8 * L.stride * (size_t)B));
    if (!bt->ptrs.ptr) {
        std::vector<ConicBatchPtrs> hp((size_t)B);
        for (int64_t p = 0; p < B; ++p) hp[(size_t)p] = ConicBatchPtrs{bt->states[(size_t)p].x.as<double>(), bt->states[(size_t)p].vp.as<double>()};
        DO_CUDA(ctx, bt->ptrs.reserve(sizeof(ConicBatchPtrs) * (size_t)B));
        DO_CUDA(ctx, cudaMemcpy(bt->ptrs.ptr, hp.data(), sizeof(ConicBatchPtrs) * (size_t)B, cudaMemcpyHostToDevice));
    }
    const void* dseed;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[0], dx_seeds, d8 * (size_t)n * (size_t)B, memspace, &dseed));
    conic_rev_rhs_batch_kernel<<<(unsigned)B, 512, 0, ctx->stream>>>(n, m, (const double*)dseed, bt->ptrs.as<ConicBatchPtrs>(),
                                                                    bt->work.as<double>(), L.stride);
    ctx->launches++;
    LsqrParams prm{atol, btol, conlim, maxiter > 0 ? maxiter : (int64_t)N};
    const char* env = getenv("DIFFOPT_B200_CONIC_BATCH_STAGE");
    const bool stage = !(env && env[0] == '0');
    if (int32_t rc = lsqr_run_conic_batch(ctx, bt->states, C, stage, bt->work.as<double>(), L, prm, 1e-4 /* :369 */,
                                          bt->ops, bt->vecs, bt->rhs))
        return rc;
    void *dg, *ddc, *ddb, *dst;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], g_out, d8 * (size_t)N * (size_t)B, memspace, &dg));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[1], dc_out, d8 * (size_t)n * (size_t)B, memspace, &ddc));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[2], db_out, d8 * (size_t)m * (size_t)B, memspace, &ddb));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[3], out_stats, d8 * 4 * (size_t)B, memspace, &dst));
    conic_rev_out_batch_kernel<<<dim3((unsigned)((N + 255) / 256), (unsigned)B), 256, 0, ctx->stream>>>(
        n, m, bt->ptrs.as<ConicBatchPtrs>(), bt->work.as<double>(), L, (double*)dg, (double*)ddc, (double*)ddb, (double*)dst);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    DO_CUDA(ctx, stage_out_finish(ctx, dg, g_out, d8 * (size_t)N * (size_t)B, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, ddc, dc_out, d8 * (size_t)n * (size_t)B, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, ddb, db_out, d8 * (size_t)m * (size_t)B, memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, dst, out_stats, d8 * 4 * (size_t)B, memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;   // ev0 / ev1 bracket the LSQR kernel (lsqr_run_conic_batch)
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}

}  // extern "C"
