// Batched QP sensitivities against STORED factors: qp_batch_factorize runs the pivot-free LDL' of the shape-generic kernel
// (qp_batch_sqd_any.cu, store mode) once per setup and keeps every instance's factor on the device; qp_batch_reverse_multi /
// qp_batch_forward_multi then solve k right-hand sides per instance with two triangular sweeps over it, instead of k full
// assemblies and factorisations (the reference refactorises per call, QuadraticProgram.jl:335, :438).
//
// qp_factored_solve_kernel: persistent, one 128-thread CTA per instance at a time.  The instance's tiles and 1/d are staged
// into shared memory once (16-byte cp.async, already in DMMA fragment order); warp w owns a block of 8 right-hand sides and
// runs both sweeps on it alone (the warps share the read-only factor, no barrier between warps during the sweeps):
//   forward   V_j = D_j^-1 L_jj^-1 R_j,  R_I -= W(I, j) V_j  for I > j       (W(I, j) = L(I, j) D_j, the DMMA A operand)
//   backward  X_j = L_jj^-T (V_j - D_j^-1 sum_{I > j} W(I, j)' X_I)
// -- the arithmetic of factor<>()'s riding-along rows and of backward() in qp_sqd_dev.cuh, in block form.  Every sum runs
// in a fixed order: results are bitwise reproducible from run to run.  The mapping to the reduced order and back is the one
// of qp_kkt_sqd_any_kernel: forward mode takes the right-hand side of qp_coo_rhs_kernel (active rows unscaled: the symmetric
// form's 1/lam cancels the reference's lam) and returns -x with 0 for the inactive lam; reverse mode takes [seed; 0; 0] and
// returns -x, -x/lam for the active rows and (G x_z)_i / D_i for the inactive ones.
// Instances the factorisation rejected (pivot test failed, active set beyond shared memory) are solved by the pivoted-LU
// kernel over the stored list, one launch per direction (it refactorises: correct and slow, for rare instances).
#include <algorithm>
#include <numeric>
#include <vector>

#include "qp_sqd_dev.cuh"

int32_t qp_generic_launch_list(diffopt_b200_ctx* ctx, const QpSolveArgs& a, const int* list, const int* count);
int32_t qp_sqd_any_store_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a, int nt_cap, double* store, int64_t stride, int* fb_list,
                                int* fb_count);
int32_t qp_max_active_any_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a, int* dmax);
bool qp_sqd_any_supported(diffopt_b200_ctx* ctx, const QpSolveArgs& a);
int qp_sqd_any_nt(const QpSolveArgs& a, int active);
int qp_sqd_any_nt_limit(diffopt_b200_ctx* ctx, const QpSolveArgs& a);
int32_t finish_info(diffopt_b200_ctx* ctx, int64_t B, int* dinfo, int32_t* info_user, int memspace, std::vector<int>& hinfo);
void fill_from_state(const QpBatchState& s, QpSolveArgs& a);

namespace {

using namespace sqd;

// shared memory of qp_factored_solve_kernel (doubles): 1/d and the tiles at the same relative offsets as in the store (one
// contiguous copy), nb right-hand-side blocks of 8 nt_cap rows x 8 columns (row-major), a 64-double scratch per block,
// D, and the ints apos[m], ainv[m] (reduced row -> inequality)
struct SolveLayout {
    int rd, tiles, rhs, part, dvec, ints, total;
    __host__ __device__ SolveLayout(int m, int nt_cap, int nb) {
        rd = 0;
        tiles = 8 * nt_cap;
        rhs = tiles + (nt_cap * (nt_cap + 1) / 2) * 64;
        part = rhs + nb * 64 * nt_cap;
        dvec = part + nb * 64;
        ints = dvec + ((m + 1) & ~1);
        total = ints + m;
    }
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}

// Both sweeps for the 8 right-hand sides of one warp: R (np x 8, row-major) holds the right-hand sides on entry and the
// solutions on exit; S is the warp's 8 x 8 scratch.  Lane (g, t) owns column g in the triangular solves (the four lanes of a
// column compute it redundantly) and the DMMA fragments of row g / columns 2t, 2t+1.
__device__ void sweep(double* const R, double* const S, const double* const T, const double* const rd, const int nt, const int g,
                      const int t) {
    for (int j = 0; j < nt; ++j) {
        const int c0 = j << 3;
        const double* Ld = T + tix(j, j) * 64;
        double x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = R[(c0 + i) * 8 + g];
#pragma unroll
        for (int c = 1; c < 8; ++c) {
            double acc = x[c];
#pragma unroll
            for (int k = 0; k < c; ++k) acc = fma(-x[k], Ld[el(c, k)], acc);
            x[c] = acc;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] *= rd[c0 + i];
        __syncwarp();
        if (t == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) R[(c0 + i) * 8 + g] = x[i];
        }
        double b0 = x[0], b1 = x[1];  // B fragment: rows 2t, 2t+1 of V_j, column g
#pragma unroll
        for (int q = 1; q < 4; ++q)
            if (t == q) {
                b0 = x[2 * q];
                b1 = x[2 * q + 1];
            }
        for (int I = j + 1; I < nt; ++I) {
            const double2 w = *reinterpret_cast<const double2*>(T + tix(I, j) * 64 + el(g, 2 * t));
            double2* cp = reinterpret_cast<double2*>(R + (8 * I + g) * 8 + 2 * t);
            double2 c = *cp;
            dmma(c.x, c.y, -w.x, b0);
            dmma(c.x, c.y, -w.y, b1);
            *cp = c;
        }
        __syncwarp();
    }
    for (int j = nt - 1; j >= 0; --j) {
        const int c0 = j << 3;
        double2 s = make_double2(0.0, 0.0);  // rows g, columns 2t, 2t+1 of sum_{I > j} W(I, j)' X_I
        for (int I = nt - 1; I > j; --I) {
            const double* W = T + tix(I, j) * 64;
            const double* X = R + 64 * I;
            dmma(s.x, s.y, W[el(2 * t, g)], X[(2 * t) * 8 + g]);
            dmma(s.x, s.y, W[el(2 * t + 1, g)], X[(2 * t + 1) * 8 + g]);
        }
        *reinterpret_cast<double2*>(S + g * 8 + 2 * t) = s;
        __syncwarp();
        const double* Dt = T + tix(j, j) * 64;
        double x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = fma(-rd[c0 + i], S[i * 8 + g], R[(c0 + i) * 8 + g]);
#pragma unroll
        for (int k = 7; k >= 1; --k) {
#pragma unroll
            for (int c = 0; c < k; ++c) x[c] = fma(-Dt[el(k, c)], x[k], x[c]);
        }
        __syncwarp();
        if (t == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) R[(c0 + i) * 8 + g] = x[i];
        }
        __syncwarp();
    }
}

// FWD: in = right-hand sides [B k][N] (qp_coo_rhs_kernel, slot b k + j), out = fwd [B][k][N]
// else: in = seeds [B][k][n], out = rev [B][k][N]; G, lam: the setup's (reverse mode reads them for the inequality rows)
template <bool FWD>
__global__ void __launch_bounds__(THREADS) qp_factored_solve_kernel(const double* __restrict__ F, const int64_t stride, const int nt_cap,
                                                                    const int64_t B, const int n, const int m, const int p,
                                                                    const int64_t k, const int nb, const double* __restrict__ in,
                                                                    double* __restrict__ out, const double* __restrict__ G,
                                                                    const double* __restrict__ lam) {
    extern __shared__ __align__(16) double sm[];
    const SolveLayout L(m, nt_cap, nb);
    const FactorLayout fl(m, nt_cap);
    const double* const rd = sm + L.rd;
    const double* const T = sm + L.tiles;
    double* const Rall = sm + L.rhs;
    double* const dvec = sm + L.dvec;
    int* const apos = reinterpret_cast<int*>(sm + L.ints);
    int* const ainv = apos + m;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int N = n + m + p, n8 = (n + 7) & ~7, npc = 8 * nt_cap, ncol = 8 * nb;
    for (int64_t inst = blockIdx.x; inst < B; inst += gridDim.x) {
        const double* Fb = F + inst * stride;
        const int* Fi = reinterpret_cast<const int*>(Fb);
        const int ma = Fi[0];
        if (ma < 0) continue;  // the pivoted-LU kernel serves it
        const int nt = (n8 + ma + p + 7) >> 3, np = nt << 3, nred = n8 + ma + p;
        {
            const int chunks = (8 * nt_cap + ((nt * (nt + 1)) >> 1) * 64) >> 1;
            for (int i = tid; i < chunks; i += THREADS) cp_async16(sm + L.rd + 2 * i, Fb + fl.rd + 2 * i);
            asm volatile("cp.async.commit_group;" ::: "memory");
            for (int i = tid; i < m; i += THREADS) {
                const int ar = Fi[1 + i];
                apos[i] = ar;
                if (ar >= 0) ainv[ar] = i;
                dvec[i] = Fb[fl.dvec + i];
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        for (int64_t c0 = 0; c0 < k; c0 += ncol) {
            // ---- right-hand sides in the reduced order (qp_batch_sqd_any.cu: z rows, active rows, equalities, zero padding)
            for (int idx = tid; idx < ncol * np; idx += THREADS) {
                const int c = idx / np, r = idx - c * np;
                const int64_t col = c0 + c;
                double v = 0.0;
                if (col < k) {
                    const int64_t slot = inst * k + col;
                    if (FWD) {
                        const double* src = in + slot * N;
                        if (r < n) v = src[r];
                        else if (r >= n8 && r < n8 + ma) v = src[n + ainv[r - n8]];
                        else if (r >= n8 + ma && r < nred) v = src[n + m + (r - n8 - ma)];
                    } else if (r < n) {
                        v = in[slot * n + r];
                    }
                }
                Rall[(c >> 3) * npc * 8 + r * 8 + (c & 7)] = v;
            }
            __syncthreads();
            if (warp < nb && c0 + 8 * warp < k) sweep(Rall + warp * npc * 8, sm + L.part + warp * 64, T, rd, nt, g, t);
            __syncthreads();
            // ---- outputs (dz, dlam, dnu) = -x
            for (int idx = tid; idx < ncol * N; idx += THREADS) {
                const int c = idx / N, i = idx - c * N;
                const int64_t col = c0 + c;
                if (col >= k) continue;
                const double* X = Rall + (c >> 3) * npc * 8 + (c & 7);
                double v;
                if (i < n) {
                    v = -X[i * 8];
                } else if (i < n + m) {
                    const int ar = apos[i - n];
                    if (ar >= 0) v = FWD ? -X[(n8 + ar) * 8] : -X[(n8 + ar) * 8] * fast_rcp(lam[inst * m + (i - n)]);
                    else if (FWD) v = 0.0;
                    else continue;  // below
                } else {
                    v = -X[(n8 + ma + (i - n - m)) * 8];
                }
                out[(inst * k + col) * N + i] = v;
            }
            if (!FWD && m) {  // inactive inequalities: (G x_z)_i / D_i, one product for the block's columns
                const double* Gb = G + inst * m * n;
                for (int idx = tid; idx < ncol * m; idx += THREADS) {
                    const int c = idx / m, i = idx - c * m;
                    const int64_t col = c0 + c;
                    if (col >= k || apos[i] >= 0) continue;
                    const double* X = Rall + (c >> 3) * npc * 8 + (c & 7);
                    double s0 = 0.0, s1 = 0.0;
                    int j = 0;
                    for (; j + 1 < n; j += 2) {
                        s0 = fma(__ldg(Gb + i + (size_t)j * m), X[j * 8], s0);
                        s1 = fma(__ldg(Gb + i + (size_t)(j + 1) * m), X[(j + 1) * 8], s1);
                    }
                    if (j < n) s0 = fma(__ldg(Gb + i + (size_t)j * m), X[j * 8], s0);
                    out[(inst * k + col) * N + n + i] = (s0 + s1) * fast_rcp(dvec[i]);
                }
            }
            __syncthreads();
        }
    }
}

// dst[b dstride + i] = src[b sstride + i], i < len, for the listed instances b (one direction in and out of the [B][...]
// layout of the pivoted-LU kernel)
__global__ void list_copy_kernel(const int* __restrict__ list, const int* __restrict__ count, const double* __restrict__ src,
                                 const int64_t sstride, double* __restrict__ dst, const int64_t dstride, const int len) {
    const int cnt = *count;
    for (int it = blockIdx.x; it < cnt; it += gridDim.x) {
        const int64_t b = list[it];
        for (int i = threadIdx.x; i < len; i += blockDim.x) dst[b * dstride + i] = src[b * sstride + i];
    }
}

}  // namespace

// k right-hand sides per instance against the stored factors: in (device) as qp_factored_solve_kernel reads it, out_user
// [B][k][N] in memspace.  Returns 0, first singular instance + 1, or < 0.
int32_t qp_factored_run(diffopt_b200_ctx* ctx, int64_t k, const double* in, double* out_user, int memspace, bool fwd) {
    QpFactorState& f = ctx->qpf;
    const QpBatchState& s = ctx->qp;
    const int64_t B = s.B;
    const int n = s.n, m = s.m, p = s.p, N = n + m + p;
    const size_t d = sizeof(double);
    void* dout = nullptr;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[fwd ? 0 : 1], out_user, d * (size_t)B * (size_t)k * N, memspace, &dout));
    double* out = (double*)dout;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (f.nt_cap > 0) {
        // RHS blocks per CTA: up to 4 (one per warp), fewer when the staged factor leaves no room for them
        int nb = (int)std::min<int64_t>(4, (k + 7) / 8);
        while (nb > 1 && (size_t)SolveLayout(m, f.nt_cap, nb).total * d > ctx->smem_optin) nb >>= 1;
        const size_t smem = (size_t)SolveLayout(m, f.nt_cap, nb).total * d;
        if (smem > ctx->smem_optin) {
            ctx->err = "qp_batch_*_multi: the stored factor does not fit shared memory";
            return -3;
        }
        const void* kern = fwd ? (const void*)qp_factored_solve_kernel<true> : (const void*)qp_factored_solve_kernel<false>;
        int per_sm = 1;
        DO_CUDA(ctx, kernel_config(kern, ctx->device, THREADS, smem, &per_sm));
        int64_t grid = (int64_t)ctx->sm_count * std::max(per_sm, 1);
        grid = std::max<int64_t>(1, std::min(grid, B));
        const double* G = m ? s.G.as<double>() : nullptr;
        if (fwd)
            qp_factored_solve_kernel<true><<<(unsigned)grid, THREADS, smem, ctx->stream>>>(f.f.as<double>(), f.stride, f.nt_cap, B, n, m, p,
                                                                                           k, nb, in, out, G, s.lam.as<double>());
        else
            qp_factored_solve_kernel<false><<<(unsigned)grid, THREADS, smem, ctx->stream>>>(f.f.as<double>(), f.stride, f.nt_cap, B, n, m,
                                                                                            p, k, nb, in, out, G, s.lam.as<double>());
        ctx->launches++;
        DO_CUDA(ctx, cudaGetLastError());
    }
    int* dinfo = nullptr;
    if (f.nrej > 0) {
        DO_CUDA(ctx, ctx->info.reserve(sizeof(int) * (size_t)B));
        dinfo = ctx->info.as<int>();
        DO_CUDA(ctx, cudaMemsetAsync(dinfo, 0, sizeof(int) * (size_t)B, ctx->stream));
        const int len_in = fwd ? N : n;
        DO_CUDA(ctx, f.gin.reserve(d * (size_t)B * len_in));
        DO_CUDA(ctx, f.gout.reserve(d * (size_t)B * N));
        QpSolveArgs a{};
        fill_from_state(s, a);
        a.info = dinfo;
        if (fwd) {
            a.rhs_pre = f.gin.as<double>();
            a.fwd = f.gout.as<double>();
        } else {
            a.seed = f.gin.as<double>();
            a.rev = f.gout.as<double>();
        }
        const int* count = f.fb.as<int>();
        const int* list = count + 1;
        const unsigned cgrid = (unsigned)std::min<int64_t>(f.nrej, (int64_t)ctx->sm_count * 4);
        for (int64_t j = 0; j < k; ++j) {
            list_copy_kernel<<<cgrid, 128, 0, ctx->stream>>>(list, count, in + j * len_in, k * len_in, f.gin.as<double>(), len_in, len_in);
            if (int32_t rc = qp_generic_launch_list(ctx, a, list, count)) return rc;
            list_copy_kernel<<<cgrid, 128, 0, ctx->stream>>>(list, count, f.gout.as<double>(), N, out + j * N, k * N, N);
            ctx->launches += 2;
        }
        DO_CUDA(ctx, cudaGetLastError());
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, stage_out_finish(ctx, dout, out_user, d * (size_t)B * (size_t)k * N, memspace));
    int32_t rc = 0;
    if (dinfo) {
        std::vector<int> hinfo;
        rc = finish_info(ctx, B, dinfo, nullptr, memspace, hinfo);
        if (rc < 0) return rc;
    } else {
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            ctx->err = std::string("kernel failed: ") + cudaGetErrorString(e);
            return -100 - (int32_t)e;
        }
    }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return rc;
}

extern "C" {

int32_t diffopt_b200_qp_batch_factorize(diffopt_b200_ctx* ctx, int32_t* info, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!ctx->qp.valid) BAD_ARG(ctx, "qp_batch_factorize: call qp_batch_setup first");
    QpFactorState& f = ctx->qpf;
    const QpBatchState& s = ctx->qp;
    const int64_t B = s.B;
    f.valid = false;
    f.nt_cap = 0;
    f.stride = 0;
    f.nrej = 0;
    ctx->qp_last_kernel = 3;
    ctx->qp_last_hint = 0;
    if (B == 0) {
        f.valid = true;
        return 0;
    }
    QpSolveArgs a{};
    fill_from_state(s, a);
    DO_CUDA(ctx, f.fb.reserve(sizeof(int) * ((size_t)B + 2)));  // [count, list (B), largest active set]
    int* fb_count = f.fb.as<int>();
    int* fb_list = fb_count + 1;
    int* dmax = fb_list + B;
    int* dinfo;
    if (info && memspace == DIFFOPT_B200_DEVICE) {
        dinfo = info;
    } else {
        DO_CUDA(ctx, ctx->info.reserve(sizeof(int) * (size_t)B));
        dinfo = ctx->info.as<int>();
    }
    DO_CUDA(ctx, cudaMemsetAsync(dinfo, 0, sizeof(int) * (size_t)B, ctx->stream));
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    // the factor storage is sized for the batch's true largest active set (one host read per setup)
    int nt_cap = 0;
    if (qp_sqd_any_supported(ctx, a)) {
        DO_CUDA(ctx, cudaMemsetAsync(dmax, 0, sizeof(int), ctx->stream));
        if (int32_t rc = qp_max_active_any_launch(ctx, a, dmax)) return rc;
        int hmax = 0;
        DO_CUDA(ctx, cudaMemcpyAsync(&hmax, dmax, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        nt_cap = std::min(qp_sqd_any_nt(a, hmax), qp_sqd_any_nt_limit(ctx, a));
    }
    int nrej = (int)B;
    if (nt_cap > 0) {
        const int64_t stride = FactorLayout(s.m, nt_cap).stride;
        const size_t bytes = sizeof(double) * (size_t)B * (size_t)stride;
        if (f.f.reserve(bytes) != cudaSuccess) {
            cudaGetLastError();
            char msg[160];
            snprintf(msg, sizeof msg, "qp_batch_factorize: cannot allocate %zu bytes of factor storage", bytes);
            ctx->err = msg;
            return -3;
        }
        a.info = dinfo;
        if (int32_t rc = qp_sqd_any_store_launch(ctx, a, nt_cap, f.f.as<double>(), stride, fb_list, fb_count)) return rc;
        DO_CUDA(ctx, cudaMemcpyAsync(&nrej, fb_count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        f.stride = stride;
    } else {  // no instance fits the fast path: the pivoted LU serves the whole batch
        std::vector<int> all((size_t)B + 1);
        all[0] = (int)B;
        std::iota(all.begin() + 1, all.end(), 0);
        DO_CUDA(ctx, cudaMemcpyAsync(fb_count, all.data(), sizeof(int) * all.size(), cudaMemcpyHostToDevice, ctx->stream));
        DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    f.nt_cap = nt_cap;
    f.nrej = nrej;
    ctx->qp_last_hint = nt_cap;
    if (nrej > 0) {  // the listed instances are factorised here once as well: a singular one is reported now
        QpSolveArgs b = a;
        b.info = dinfo;
        if (int32_t rc = qp_generic_launch_list(ctx, b, fb_list, fb_count)) return rc;
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    std::vector<int> hinfo;
    int32_t rc = finish_info(ctx, B, dinfo, info, memspace, hinfo);
    if (rc < 0) return rc;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    f.valid = true;
    return rc;
}

int32_t diffopt_b200_qp_batch_reverse_multi(diffopt_b200_ctx* ctx, int64_t k, const double* dl_dz, double* rev_out, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!ctx->qpf.valid) BAD_ARG(ctx, "qp_batch_reverse_multi: call qp_batch_factorize first (qp_batch_setup drops the stored factor)");
    if (k < 0) BAD_ARG(ctx, "qp_batch_reverse_multi: need k >= 0");
    const QpBatchState& s = ctx->qp;
    if (k == 0 || s.B == 0) return 0;
    if (!dl_dz || !rev_out) BAD_ARG(ctx, "qp_batch_reverse_multi: dl_dz and rev_out are required");
    const void* ptr;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[13], dl_dz, sizeof(double) * (size_t)s.B * (size_t)k * s.n, memspace, &ptr));
    return qp_factored_run(ctx, k, (const double*)ptr, rev_out, memspace, false);
}

}  // extern "C"
