// The LSQR branch of solve_system for a batch of LPs (Q = 0, QuadraticProgram.jl:333-335, :436-438, :486-488):
// diffopt_b200_qp_batch_solve_lsqr.  One CTA per instance runs the reverse solve (LHS) and the forward solve (LHS') in
// lock-step against the matrix-free KKT operator
//   LHS  = [0 G'diag(lam) A'; G diag(d) 0; A 0 0],   d = G z - h   (create_LHS_matrix with Q = 0),
// with the arithmetic of every other LSQR driver (LsqrScalars in lsqr.cuh, the deferred x / w update) and every sum in a
// fixed order inside the CTA: an instance's result is bitwise reproducible and independent of the rest of the batch.
// Solve 0 is the forward solve, solve 1 the reverse one; a solve that has stopped is frozen while the other goes on.
#include <algorithm>

#include "lsqr.cuh"

namespace {

constexpr int LP_THREADS = 256;
constexpr int LP_WARPS = LP_THREADS / 32;
constexpr int LP_RPL = 4;              // rows of W a lane holds in one chunk of the W pass
constexpr int LP_CHUNK = 32 * LP_RPL;  // rows of W per chunk

struct LpArgs {
    int n, m, p;
    int shared;  // G, A are one instance for the batch
    int staged;  // W = [G; A] is copied into shared memory
    int chunk;   // rows per chunk of the W pass: min(LP_CHUNK, max(m, p, 1))
    const double *G, *A, *h, *z, *lam, *nu;
    const double *dQ, *dq, *dG, *dh, *dA, *db, *seed;
    double *fwd, *rev, *stats;
    LsqrParams prm;
};

// doubles of dynamic shared memory: u, v, w, x of both solves | lam, d | y [2][m+p] | W'b [2][n] | W a partials
// [LP_WARPS][2][chunk] | W (staged route)
size_t lp_smem_doubles(int n, int m, int p, int chunk, bool staged) {
    const size_t N = (size_t)n + m + p, M = (size_t)m + p;
    return 8 * N + 2 * (size_t)m + 2 * M + 2 * (size_t)n + (size_t)LP_WARPS * 2 * chunk + (staged ? M * n : 0);
}

struct Seg {  // rows [off, off + rows) of W, column-major with leading dimension ld
    const double* p;
    int ld, rows, off;
};

__device__ __forceinline__ double lp_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// fixed-order sums over the CTA of one value per solve (result in every thread)
__device__ __forceinline__ void block_sum2(double& s0, double& s1, double* red) {
    s0 = lp_warp_sum(s0);
    s1 = lp_warp_sum(s1);
    __syncthreads();  // red is still read by the previous call
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = s0;
        red[LP_WARPS + (threadIdx.x >> 5)] = s1;
    }
    __syncthreads();
    s0 = s1 = 0.0;
    for (int w = 0; w < LP_WARPS; ++w) {
        s0 += red[w];
        s1 += red[LP_WARPS + w];
    }
}

// One pass over W = [G; A] serves the products of both solves: y_k = W a_k and wt_k = W' b_k (k = 0, 1), with
// a_k = src_k[0, n) and b_k = src_k[n, N), its first m entries scaled by lam when lam_k.  Lane l of a warp holds rows
// r0 + l + 32 q of a chunk and the warp sweeps the columns j = warp, warp + LP_WARPS, ...: every element read feeds four
// FMAs, and the lanes of a warp read consecutive addresses of one column for both products (no bank conflicts in shared
// memory at any leading dimension, coalesced loads on the global route).  W' b is summed over the lanes by a butterfly
// and over the chunks in order; W a over the warps in order.
__device__ void w_pass(const Seg (&seg)[2], int n, int m, int M, int chunk, const double* src0, const double* src1,
                       bool lam0, bool lam1, const double* lam, double* y, double* wt, double* part) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j = threadIdx.x; j < 2 * n; j += LP_THREADS) wt[j] = 0.0;
    __syncthreads();
#pragma unroll
    for (int sg = 0; sg < 2; ++sg) {
        const Seg s = seg[sg];
        for (int r0 = 0; r0 < s.rows; r0 += chunk) {
            const int rows = min(chunk, s.rows - r0), nq = (rows + 31) >> 5;
            double acc0[LP_RPL], acc1[LP_RPL], b0[LP_RPL], b1[LP_RPL];
#pragma unroll
            for (int q = 0; q < LP_RPL; ++q) {
                const int r = lane + 32 * q, i = s.off + r0 + r;
                const bool ok = r < rows;
                const double l = ok && i < m ? lam[i] : 1.0;
                acc0[q] = acc1[q] = 0.0;
                b0[q] = ok ? (lam0 ? l * src0[n + i] : src0[n + i]) : 0.0;
                b1[q] = ok ? (lam1 ? l * src1[n + i] : src1[n + i]) : 0.0;
            }
            for (int j = warp; j < n; j += LP_WARPS) {
                const double* col = s.p + (size_t)j * s.ld + r0 + lane;
                const double a0 = src0[j], a1 = src1[j];
                double t0 = 0.0, t1 = 0.0;
#pragma unroll
                for (int q = 0; q < LP_RPL; ++q) {
                    if (q < nq) {
                        const double g = lane + 32 * q < rows ? col[32 * q] : 0.0;
                        acc0[q] = fma(g, a0, acc0[q]);
                        acc1[q] = fma(g, a1, acc1[q]);
                        t0 = fma(g, b0[q], t0);
                        t1 = fma(g, b1[q], t1);
                    }
                }
                t0 = lp_warp_sum(t0);
                t1 = lp_warp_sum(t1);
                if (lane == 0) {
                    wt[j] += t0;
                    wt[n + j] += t1;
                }
            }
#pragma unroll
            for (int q = 0; q < LP_RPL; ++q) {
                const int r = lane + 32 * q;
                if (r < rows) {
                    part[(warp * 2) * chunk + r] = acc0[q];
                    part[(warp * 2 + 1) * chunk + r] = acc1[q];
                }
            }
            __syncthreads();
            for (int t = threadIdx.x; t < 2 * rows; t += LP_THREADS) {
                const int k = t >= rows ? 1 : 0, r = t - k * rows;
                double sum = 0.0;
                for (int w = 0; w < LP_WARPS; ++w) sum += part[(w * 2 + k) * chunk + r];
                y[k * M + s.off + r0 + r] = sum;
            }
            __syncthreads();
        }
    }
}

// dst_k = s_src_k OP_k(src_k) + s_dst_k dst_k for the solves with act_k; returns ||dst_k||^2 in nrm_k.  tr0: solve 0
// applies LHS' (solve 1 then applies LHS), else the other way round.
//   LHS  src = [G'(lam o s2) + A's3;       G s1 + d o s2; A s1]
//   LHS' src = [G's2 + A's3;         lam o (G s1) + d o s2; A s1]
struct LpView {
    Seg seg[2];
    int n, m, M, N, chunk;
    const double *lam, *d;
    double *y, *wt, *part, *red;
};

__device__ __forceinline__ void apply2(const LpView& o, bool tr0, const double* src0, const double* src1, double* dst0,
                                       double* dst1, double ss0, double sd0, double ss1, double sd1, bool act0, bool act1,
                                       double& nrm0, double& nrm1) {
    const int n = o.n, m = o.m, M = o.M;
    w_pass(o.seg, n, m, M, o.chunk, src0, src1, !tr0, tr0, o.lam, o.y, o.wt, o.part);
    double acc0 = 0.0, acc1 = 0.0;
    for (int i = threadIdx.x; i < o.N; i += LP_THREADS) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (!(k == 0 ? act0 : act1)) continue;
            const bool tr = (k == 0) == tr0;
            const double* src = k == 0 ? src0 : src1;
            double* dst = k == 0 ? dst0 : dst1;
            double out;
            if (i < n) {
                out = o.wt[k * n + i];
            } else if (i < n + m) {
                const int r = i - n;
                const double g = o.y[k * M + r];
                out = (tr ? o.lam[r] * g : g) + o.d[r] * src[i];
            } else {
                out = o.y[k * M + i - n];
            }
            const double v = (k == 0 ? ss0 : ss1) * out + (k == 0 ? sd0 : sd1) * dst[i];
            dst[i] = v;
            if (k == 0) acc0 += v * v;
            else acc1 += v * v;
        }
    }
    block_sum2(acc0, acc1, o.red);
    nrm0 = acc0;
    nrm1 = acc1;
}

__global__ void __launch_bounds__(LP_THREADS, 2) qp_lp_lsqr_kernel(LpArgs a) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double red[2 * LP_WARPS];
    __shared__ LsqrScalars sc[2];
    __shared__ int active[2], op1[2];
    const size_t b = blockIdx.x;
    const int n = a.n, m = a.m, p = a.p, M = m + p, N = n + M;
    const int tid = threadIdx.x;
    double* const vec = smem;  // solve k: u, v, w, x at vec + (4 k + 0 .. 3) N
    LpView o;
    o.n = n; o.m = m; o.M = M; o.N = N; o.chunk = a.chunk;
    double* lam = vec + (size_t)8 * N;
    double* d = lam + m;
    o.lam = lam; o.d = d;
    o.y = d + m;
    o.wt = o.y + 2 * M;
    o.part = o.wt + 2 * n;
    o.red = red;
    double* const W = o.part + (size_t)LP_WARPS * 2 * a.chunk;
    const double* G = a.G ? a.G + (a.shared ? 0 : b * m * n) : nullptr;
    const double* A = a.A ? a.A + (a.shared ? 0 : b * p * n) : nullptr;
    if (a.staged) {
        for (int e = tid; e < M * n; e += LP_THREADS) {
            const int j = e / M, i = e - j * M;
            W[e] = i < m ? G[i + (size_t)j * m] : A[(i - m) + (size_t)j * p];
        }
        o.seg[0] = Seg{W, M, m, 0};
        o.seg[1] = Seg{W + m, M, p, m};
    } else {
        o.seg[0] = Seg{G, m, m, 0};
        o.seg[1] = Seg{A, p, p, m};
    }
    const double* z = a.z + b * n;
    const double* lam_g = m ? a.lam + b * m : nullptr;
    const double* nu = p ? a.nu + b * p : nullptr;
    const double* h = m ? a.h + b * m : nullptr;
    for (int i = tid; i < m; i += LP_THREADS) lam[i] = lam_g[i];
    __syncthreads();
    for (int i = tid; i < m; i += LP_THREADS) {  // d = G z - h
        const double* g = o.seg[0].p + i;
        double s = 0.0;
        for (int j = 0; j < n; ++j) s += g[(size_t)j * o.seg[0].ld] * z[j];
        d[i] = s - h[i];
    }

    // right-hand sides: forward [dQ z + dq + dG'lam + dA'nu; lam o (dG z) - lam o dh; dA z - db] (:429-433), reverse
    // [dl_dz; 0; 0]; u = rhs, v = w = x = 0
    const double* dQ = a.dQ ? a.dQ + b * n * n : nullptr;
    const double* dq = a.dq ? a.dq + b * n : nullptr;
    const double* dG = a.dG && m ? a.dG + b * m * n : nullptr;
    const double* dh = a.dh && m ? a.dh + b * m : nullptr;
    const double* dA = a.dA && p ? a.dA + b * p * n : nullptr;
    const double* db = a.db && p ? a.db + b * p : nullptr;
    const double* seed = a.seed ? a.seed + b * n : nullptr;
    double b0 = 0.0, b1 = 0.0;
    for (int i = tid; i < N; i += LP_THREADS) {
        double r = 0.0;
        if (a.fwd) {
            if (i < n) {
                if (dQ) for (int c = 0; c < n; ++c) r += dQ[i + (size_t)c * n] * z[c];
                if (dq) r += dq[i];
                if (dG) for (int k = 0; k < m; ++k) r += dG[k + (size_t)i * m] * lam_g[k];
                if (dA) for (int k = 0; k < p; ++k) r += dA[k + (size_t)i * p] * nu[k];
            } else if (i < n + m) {
                const int k = i - n;
                double gz = 0.0;
                if (dG) for (int c = 0; c < n; ++c) gz += dG[k + (size_t)c * m] * z[c];
                r = lam_g[k] * gz - lam_g[k] * (dh ? dh[k] : 0.0);
            } else {
                const int k = i - n - m;
                double az = 0.0;
                if (dA) for (int c = 0; c < n; ++c) az += dA[k + (size_t)c * p] * z[c];
                r = az - (db ? db[k] : 0.0);
            }
        }
        const double s = a.rev && seed && i < n ? seed[i] : 0.0;
        vec[i] = r;
        vec[(size_t)4 * N + i] = s;
        b0 += r * r;
        b1 += s * s;
#pragma unroll
        for (int k = 0; k < 2; ++k)
            for (int q = 1; q < 4; ++q) vec[(size_t)(4 * k + q) * N + i] = 0.0;
    }
    block_sum2(b0, b1, red);
    if (tid < 2) op1[tid] = sc[tid].start(tid == 0 ? b0 : b1, -1.0);
    __syncthreads();
    double* const u0 = vec;
    double* const v0 = vec + N;
    double* const u1 = vec + (size_t)4 * N;
    double* const v1 = vec + (size_t)5 * N;
    double n0, n1;
    // v_mem = M' u_true: the forward solve's M' is LHS
    apply2(o, false, u0, u1, v0, v1, sc[0].su, 0.0, sc[1].su, 0.0, op1[0] != 0, op1[1] != 0, n0, n1);
    if (tid < 2) {
        sc[tid].first_alpha(op1[tid] ? (tid == 0 ? n0 : n1) : 0.0);
        active[tid] = sc[tid].arnorm != 0.0;
    }
    bool first = true;
    while (true) {
        __syncthreads();
        const bool act0 = active[0] != 0, act1 = active[1] != 0;
        if (!act0 && !act1) break;
        double dd0 = 0.0, dd1 = 0.0;
#pragma unroll
        for (int k = 0; k < 2; ++k) {  // deferred update: w = sv v at start, later x += t1 w, w = sv v + t2 w
            if (!(k == 0 ? act0 : act1)) continue;
            const double *v = vec + (size_t)(4 * k + 1) * N;
            double *w = vec + (size_t)(4 * k + 2) * N, *x = vec + (size_t)(4 * k + 3) * N;
            const double sv = sc[k].sv, t1 = sc[k].t1, t2 = sc[k].t2, irho = 1.0 / sc[k].rho;
            double dd = 0.0;
            for (int i = tid; i < N; i += LP_THREADS) {
                if (first) {
                    w[i] = sv * v[i];
                } else {
                    const double wi = w[i];
                    const double dk = wi * irho;
                    dd += dk * dk;
                    x[i] += t1 * wi;
                    w[i] = sv * v[i] + t2 * wi;
                }
            }
            if (k == 0) dd0 = dd;
            else dd1 = dd;
        }
        block_sum2(dd0, dd1, red);
        const bool more0 = sc[0].itn < a.prm.maxiter, more1 = sc[1].itn < a.prm.maxiter;
        // u_mem = M v_true - alpha u_true: the forward solve's M is LHS'
        apply2(o, true, v0, v1, u0, u1, sc[0].sv, -sc[0].alpha * sc[0].su, sc[1].sv, -sc[1].alpha * sc[1].su,
               act0 && more0, act1 && more1, n0, n1);
        if (tid < 2 && active[tid]) {
            const int k = tid;
            if (!first) sc[k].stop_tests(k == 0 ? dd0 : dd1, a.prm);
            if (sc[k].istop > 0 || !(k == 0 ? more0 : more1)) active[k] = 0;
            else op1[k] = sc[k].next_beta(k == 0 ? n0 : n1);
        }
        first = false;
        __syncthreads();
        const bool go0 = active[0] != 0, go1 = active[1] != 0;
        if (!go0 && !go1) break;
        // v_mem = M' u_true - beta v_true
        apply2(o, false, u0, u1, v0, v1, sc[0].su, -sc[0].beta * sc[0].sv, sc[1].su, -sc[1].beta * sc[1].sv,
               go0 && op1[0], go1 && op1[1], n0, n1);
        if (tid < 2 && active[tid]) {
            const int k = tid;
            if (op1[k]) sc[k].next_alpha(k == 0 ? n0 : n1);
            sc[k].rotate();
        }
    }
    const double* x0 = vec + (size_t)3 * N;
    const double* x1 = vec + (size_t)7 * N;
    for (int i = tid; i < N; i += LP_THREADS) {
        if (a.fwd) a.fwd[b * N + i] = -x0[i];
        if (a.rev) a.rev[b * N + i] = -x1[i];
    }
    if (a.stats && tid < 2) {
        double* st = a.stats + b * 8 + tid * 4;
        st[0] = (double)sc[tid].istop;
        st[1] = (double)sc[tid].itn;
        st[2] = sc[tid].rnorm;
        st[3] = sc[tid].arnorm;
    }
}

}  // namespace

extern "C" int32_t diffopt_b200_qp_batch_solve_lsqr(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p, const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu, const double* dQ, const double* dq, const double* dG,
    const double* dh, const double* dA, const double* db, const double* dl_dz, double atol, double btol, double conlim,
    int64_t maxiter, double* fwd_out, double* rev_out, double* stats_out, int32_t memspace, int32_t flags) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (B < 0 || n <= 0 || m < 0 || p < 0) BAD_ARG(ctx, "qp_batch_solve_lsqr: need B >= 0, n > 0, m >= 0, p >= 0");
    if (flags & ~DIFFOPT_QP_SHARED_MATRICES) BAD_ARG(ctx, "qp_batch_solve_lsqr: flags may hold DIFFOPT_QP_SHARED_MATRICES only");
    if (memspace != DIFFOPT_B200_HOST && memspace != DIFFOPT_B200_DEVICE) BAD_ARG(ctx, "qp_batch_solve_lsqr: bad memspace");
    if (maxiter < 0) BAD_ARG(ctx, "qp_batch_solve_lsqr: need maxiter >= 0");
    if (!z || (m > 0 && (!G || !h || !lam)) || (p > 0 && (!A || !nu)))
        BAD_ARG(ctx, "qp_batch_solve_lsqr: z (and G, h, lam when m > 0; A, nu when p > 0) are required");
    if (B == 0) return 0;
    const int64_t N = (int64_t)n + m + p;
    const int chunk = std::min(LP_CHUNK, std::max(std::max(m, p), 1));
    cudaFuncAttributes fa;
    DO_CUDA(ctx, cudaFuncGetAttributes(&fa, qp_lp_lsqr_kernel));
    const size_t limit = ctx->smem_optin - fa.sharedSizeBytes;
    const size_t base = sizeof(double) * lp_smem_doubles(n, m, p, chunk, false);
    const size_t full = sizeof(double) * lp_smem_doubles(n, m, p, chunk, true);
    if (B > 0x7fffffff) BAD_ARG(ctx, "qp_batch_solve_lsqr: B exceeds the grid limit (2^31 - 1 instances per call)");
    if (base > limit) {
        ctx->err = "qp_batch_solve_lsqr: the LSQR vectors of one instance do not fit one CTA's shared memory "
                   "(use diffopt_b200_lsqr_csc for this size)";
        return -3;
    }
    const bool staged = full <= limit;
    const size_t smem = staged ? full : base;

    LpArgs a{};
    a.n = n; a.m = m; a.p = p;
    a.shared = (flags & DIFFOPT_QP_SHARED_MATRICES) != 0;
    a.staged = staged;
    a.chunk = chunk;
    a.prm = LsqrParams{atol, btol, conlim, maxiter > 0 ? (long long)maxiter : (long long)N};
    const size_t d = sizeof(double);
    const int64_t Bm = a.shared ? 1 : B;
    const void* ptr;
#define STAGE_LP(slot, field, src, count)                                                           \
    DO_CUDA(ctx, stage_in(ctx, ctx->in[slot], src, d * (size_t)(count), memspace, &ptr)); \
    a.field = (const double*)ptr;
    STAGE_LP(1, G, G, Bm * m * n)
    STAGE_LP(2, A, A, Bm * p * n)
    STAGE_LP(3, h, h, B * m)
    STAGE_LP(4, z, z, B * n)
    STAGE_LP(5, lam, lam, B * m)
    STAGE_LP(6, nu, nu, B * p)
    if (fwd_out) {
        STAGE_LP(7, dQ, dQ, B * n * n)
        STAGE_LP(8, dq, dq, B * n)
        STAGE_LP(9, dG, dG, B * m * n)
        STAGE_LP(10, dh, dh, B * m)
        STAGE_LP(11, dA, dA, B * p * n)
        STAGE_LP(12, db, db, B * p)
    }
    if (rev_out) { STAGE_LP(13, seed, dl_dz, B * n) }
#undef STAGE_LP
    void* dptr;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[0], fwd_out, d * (size_t)(B * N), memspace, &dptr));
    a.fwd = (double*)dptr;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[1], rev_out, d * (size_t)(B * N), memspace, &dptr));
    a.rev = (double*)dptr;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[2], stats_out, d * (size_t)(B * 8), memspace, &dptr));
    a.stats = (double*)dptr;
    DO_CUDA(ctx, kernel_config((const void*)qp_lp_lsqr_kernel, ctx->device, LP_THREADS, smem, nullptr));
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (fwd_out || rev_out || stats_out) {
        qp_lp_lsqr_kernel<<<(unsigned)B, LP_THREADS, smem, ctx->stream>>>(a);
        ctx->launches++;
        DO_CUDA(ctx, cudaGetLastError());
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, stage_out_finish(ctx, a.fwd, fwd_out, d * (size_t)(B * N), memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, a.rev, rev_out, d * (size_t)(B * N), memspace));
    DO_CUDA(ctx, stage_out_finish(ctx, a.stats, stats_out, d * (size_t)(B * 8), memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}
