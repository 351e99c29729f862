// Extended batched-QP entry points (include/diffopt_b200.h):
//   * diffopt_b200_qp_batch_solve_ex  -- flags for batch-invariant Q, G, A (OptNet layers: the weights are ONE instance,
//     read once and kept in L2 instead of 75 KB per solve over PCIe / HBM), batch-invariant directions, and Q / dQ as
//     packed lower triangles (they are symmetric: utils.jl:46-69 symmetrises them on the reference's side too);
//   * diffopt_b200_qp_batch_shared_grads -- reverse-mode gradients of the SHARED parameters: the getters of
//     QuadraticProgram.jl:307-314, :448-473 summed over the batch on the device (deterministic two-stage sum), then ONE
//     device-resident fp64 ncclAllReduce over the ranks that each own a shard of the batch (SURVEY.md 8e) -- the `+=`
//     over samples of docs/src/examples/polyhedral_project.jl:95-104 / src/parameters.jl:355-360;
//   * diffopt_b200_nccl_*  -- the communicator lives in the ctx; NCCL itself is bound at run time (dlopen of
//     libnccl.so.2, the copy the host process already carries), so the library loads and runs without it.
#include <dlfcn.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

int32_t qp_solve_common(diffopt_b200_ctx* ctx, QpSolveArgs a, double* fwd_user, double* rev_user, int32_t* info_user, int memspace,
                        bool async);
int32_t qp_factored_run(diffopt_b200_ctx* ctx, int64_t k, const double* in, double* out_user, int memspace, bool fwd);

namespace {

// packed lower triangle (column-major: column j holds rows j .. n-1) -> full symmetric n x n, one instance per blockIdx.y
__global__ void unpack_lower_kernel(const double* __restrict__ packed, double* __restrict__ full, const int n, const int64_t B) {
    const int64_t per = (int64_t)n * (n + 1) / 2;
    for (int64_t b = blockIdx.y; b < B; b += gridDim.y) {
        const double* src = packed + b * per;
        double* dst = full + b * (int64_t)n * n;
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n * n; e += gridDim.x * blockDim.x) {
            const int i = e % n, j = e / n;
            const int r = i >= j ? i : j, c = i >= j ? j : i;
            dst[e] = src[(int64_t)c * n - (int64_t)c * (c - 1) / 2 + (r - c)];
        }
    }
}

// Forward right-hand side [dQ z + dq + dG'lam + dA'nu; dG z - dh; dA z - db] (QuadraticProgram.jl:429-433, the middle block
// before its scaling by lam) from the direction's sparse triplets -- what the reference holds after diff_opt.jl:594-656 and
// SparseArrays.sparse (duplicates add up).  One thread per slot walks its triplets in storage order (a fixed summation
// order); an index outside its matrix raises *err and is skipped.  k directions per instance: slot s = b k + j is direction j
// of instance b (triplets, dq, dh, db and rhs are per slot; z, lam, nu per instance).
struct CooDev {
    const int64_t *ptr, *I, *J;
    const double* V;
};

__global__ void qp_coo_rhs_kernel(const int64_t B, const int64_t k, const int n, const int m, const int p, const double* __restrict__ z,
                                  const double* __restrict__ lam, const double* __restrict__ nu, const CooDev cq, const CooDev cg,
                                  const CooDev ca, const double* __restrict__ dq, const double* __restrict__ dh,
                                  const double* __restrict__ db, const int shared_dir, double* __restrict__ rhs, int* err) {
    const int N = n + m + p;
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < B * k; s += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = s / k;
        double* r = rhs + s * N;
        const double* zb = z + b * n;
        const int64_t bt = shared_dir ? 0 : s;
        for (int i = 0; i < n; ++i) r[i] = dq ? dq[s * n + i] : 0.0;
        for (int i = 0; i < m; ++i) r[n + i] = dh ? -dh[s * m + i] : 0.0;
        for (int i = 0; i < p; ++i) r[n + m + i] = db ? -db[s * p + i] : 0.0;
        if (cq.ptr)
            for (int64_t k = cq.ptr[bt]; k < cq.ptr[bt + 1]; ++k) {
                const int64_t i = cq.I[k] - 1, j = cq.J[k] - 1;
                if (i < 0 || i >= n || j < 0 || j >= n) { *err = 1; continue; }
                r[i] += cq.V[k] * zb[j];
            }
        if (cg.ptr && m)
            for (int64_t k = cg.ptr[bt]; k < cg.ptr[bt + 1]; ++k) {
                const int64_t i = cg.I[k] - 1, j = cg.J[k] - 1;
                if (i < 0 || i >= m || j < 0 || j >= n) { *err = 1; continue; }
                const double v = cg.V[k];
                r[n + i] += v * zb[j];
                r[j] += v * lam[b * m + i];
            }
        if (ca.ptr && p)
            for (int64_t k = ca.ptr[bt]; k < ca.ptr[bt + 1]; ++k) {
                const int64_t i = ca.I[k] - 1, j = ca.J[k] - 1;
                if (i < 0 || i >= p || j < 0 || j >= n) { *err = 1; continue; }
                const double v = ca.V[k];
                r[n + m + i] += v * zb[j];
                r[j] += v * nu[b * p + i];
            }
    }
}

// The triplets of dQ, dG, dA on the device: used in place (device memspace) or, after their offsets were checked, staged into
// ctx->qp_coo[0..2] as ptr | I | J | V back to back (host memspace).  `slots` = entries of ptr minus one.
int32_t stage_triplets(diffopt_b200_ctx* ctx, const char* who, const diffopt_b200_coo_batch* const src[3], const int lim_rows[3],
                       const int64_t slots, const int memspace, CooDev dev[3]) {
    for (int q = 0; q < 3; ++q) {
        const diffopt_b200_coo_batch* c = src[q];
        dev[q] = CooDev{};
        if (!c || !c->ptr || lim_rows[q] == 0) continue;
        if (memspace == DIFFOPT_B200_DEVICE) {
            dev[q] = CooDev{c->ptr, c->I, c->J, c->V};
            continue;
        }
        const int64_t nnz = c->ptr[slots];
        if (c->ptr[0] != 0 || nnz < 0 || (nnz > 0 && (!c->I || !c->J || !c->V)))
            BAD_ARG(ctx, std::string(who) + ": triplet offsets must start at 0 and I, J, V must be given");
        for (int64_t b = 0; b < slots; ++b)
            if (c->ptr[b + 1] < c->ptr[b]) BAD_ARG(ctx, std::string(who) + ": triplet offsets must be nondecreasing");
        const size_t np8 = sizeof(int64_t) * (size_t)(slots + 1), nz8 = sizeof(int64_t) * (size_t)nnz;
        DevBuf& buf = ctx->qp_coo[q];
        DO_CUDA(ctx, buf.reserve(np8 + 3 * nz8 + 8));
        char* base = buf.as<char>();
        DO_CUDA(ctx, cudaMemcpyAsync(base, c->ptr, np8, cudaMemcpyHostToDevice, ctx->stream));
        if (nnz > 0) {
            DO_CUDA(ctx, cudaMemcpyAsync(base + np8, c->I, nz8, cudaMemcpyHostToDevice, ctx->stream));
            DO_CUDA(ctx, cudaMemcpyAsync(base + np8 + nz8, c->J, nz8, cudaMemcpyHostToDevice, ctx->stream));
            DO_CUDA(ctx, cudaMemcpyAsync(base + np8 + 2 * nz8, c->V, nz8, cudaMemcpyHostToDevice, ctx->stream));
        }
        dev[q] = CooDev{(const int64_t*)base, (const int64_t*)(base + np8), (const int64_t*)(base + np8 + nz8),
                        (const double*)(base + np8 + 2 * nz8)};
    }
    return 0;
}

constexpr int GR_THREADS = 256;
constexpr int GR_STAGE = 16;  // instances whose vectors one CTA keeps in shared memory at a time

// one output element of the getters for one instance (vectors of the instance in shared memory)
__device__ __forceinline__ double grad_term(const int kind, const int i, const int j, const int n, const int m, const double* z,
                                            const double* lam, const double* nu, const double* r) {
    switch (kind) {
        case 0: return 0.5 * (r[i] * z[j] + z[i] * r[j]);                     // dQ = (dz z' + z dz')/2
        case 1: return r[i];                                                  // dq = dz
        case 2: { const double l = lam[i]; return l * r[n + i] * z[j] + l * r[j]; }  // dG_i = lam_i dlam_i z + lam_i dz
        case 3: return -lam[i] * r[n + i];                                    // dh = -lam . dlam
        case 4: return r[n + m + i] * z[j] + nu[i] * r[j];                    // dA_i = dnu_i z + nu_i dz
        default: return -r[n + m + i];                                        // db = -dnu
    }
}

// stage 1: CTA c sums the instances b = c, c + G, c + 2G, ... in that order -> partial[c][per]
__global__ void __launch_bounds__(GR_THREADS) shared_grads_partial_kernel(const int64_t B, const int n, const int m, const int p,
                                                                          const double* __restrict__ z, const double* __restrict__ lam,
                                                                          const double* __restrict__ nu, const double* __restrict__ rev,
                                                                          double* __restrict__ partial) {
    extern __shared__ __align__(16) double gr_smem[];
    const int N = n + m + p, V = 2 * N;  // per instance: z, lam, nu, rev
    const int64_t per = (int64_t)n * n + n + (int64_t)m * n + m + (int64_t)p * n + p;
    const int tid = threadIdx.x;
    double* out = partial + (int64_t)blockIdx.x * per;
    bool first = true;
    for (int64_t b0 = blockIdx.x; b0 < B; b0 += (int64_t)gridDim.x * GR_STAGE) {
        int cnt = 0;
        for (int q = 0; q < GR_STAGE; ++q) {
            const int64_t b = b0 + (int64_t)q * gridDim.x;
            if (b >= B) break;
            ++cnt;
            double* s = gr_smem + q * V;
            for (int i = tid; i < V; i += GR_THREADS) {
                double v;
                if (i < n) v = z[b * n + i];
                else if (i < n + m) v = lam[b * m + (i - n)];
                else if (i < N) v = nu[b * p + (i - n - m)];
                else v = rev[b * N + (i - N)];
                s[i] = v;
            }
        }
        __syncthreads();
        for (int64_t e0 = tid; e0 < per; e0 += GR_THREADS) {
            int64_t e = e0;
            int kind, i = 0, j = 0;
            if (e < (int64_t)n * n) { kind = 0; i = (int)(e % n); j = (int)(e / n); }
            else if ((e -= (int64_t)n * n) < n) { kind = 1; i = (int)e; }
            else if ((e -= n) < (int64_t)m * n) { kind = 2; i = (int)(e % m); j = (int)(e / m); }
            else if ((e -= (int64_t)m * n) < m) { kind = 3; i = (int)e; }
            else if ((e -= m) < (int64_t)p * n) { kind = 4; i = (int)(e % p); j = (int)(e / p); }
            else { e -= (int64_t)p * n; kind = 5; i = (int)e; }
            double acc = first ? 0.0 : out[e0];
            for (int q = 0; q < cnt; ++q) {
                const double* s = gr_smem + q * V;
                acc += grad_term(kind, i, j, n, m, s, s + n, s + n + m, s + N);
            }
            out[e0] = acc;
        }
        first = false;
        __syncthreads();
    }
    if (first)  // a CTA without instances still owns a row of partial[]
        for (int64_t e0 = tid; e0 < per; e0 += GR_THREADS) out[e0] = 0.0;
}

// stage 2: fixed-order sum over the CTAs of stage 1
__global__ void shared_grads_final_kernel(const int64_t per, const int G, const double* __restrict__ partial, double* __restrict__ out) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < per; e += (int64_t)gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int c = 0; c < G; ++c) acc += partial[(int64_t)c * per + e];
        out[e] = acc;
    }
}

// ---- NCCL, bound at run time -------------------------------------------------------------------------------------
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, NcclUniqueIdBytes, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string why;
};

NcclApi& nccl_api() {
    static NcclApi api;
    if (api.lib || !api.why.empty()) return api;
    const char* names[3] = {getenv("DIFFOPT_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        if (!nm || !*nm) continue;
        api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) break;
    }
    if (!api.lib) {
        api.why = "NCCL is not available: dlopen(libnccl.so.2) failed (set DIFFOPT_B200_NCCL_LIB to its path)";
        return api;
    }
    api.GetUniqueId = (int (*)(void*))dlsym(api.lib, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void**, int, NcclUniqueIdBytes, int))dlsym(api.lib, "ncclCommInitRank");
    api.CommDestroy = (int (*)(void*))dlsym(api.lib, "ncclCommDestroy");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(api.lib, "ncclAllReduce");
    api.GetErrorString = (const char* (*)(int))dlsym(api.lib, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce) {
        api.why = "NCCL library found but a required symbol is missing";
        dlclose(api.lib);
        api.lib = nullptr;
    }
    return api;
}

constexpr int NCCL_DOUBLE = 8, NCCL_SUM = 0;  // ncclFloat64, ncclSum (nccl.h)

int32_t nccl_fail(diffopt_b200_ctx* ctx, const char* what, int rc) {
    NcclApi& api = nccl_api();
    char buf[256];
    snprintf(buf, sizeof buf, "%s failed: %s", what, api.GetErrorString ? api.GetErrorString(rc) : "NCCL error");
    if (ctx) ctx->err = buf;
    return -50 - rc;
}

}  // namespace

void nccl_release(diffopt_b200_ctx* ctx) {
    if (ctx->nccl_comm) {
        NcclApi& api = nccl_api();
        if (api.CommDestroy) api.CommDestroy(ctx->nccl_comm);
        ctx->nccl_comm = nullptr;
        ctx->nccl_ranks = 0;
    }
}

extern "C" {

int32_t diffopt_b200_nccl_unique_id(void* id128) {
    if (!id128) return -1;
    NcclApi& api = nccl_api();
    if (!api.lib) return -6;
    const int rc = api.GetUniqueId(id128);
    return rc == 0 ? 0 : -50 - rc;
}

int32_t diffopt_b200_nccl_init(diffopt_b200_ctx* ctx, int32_t nranks, int32_t rank, const void* id128) {
    if (!ctx || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return -1;
    NcclApi& api = nccl_api();
    if (!api.lib) {
        ctx->err = api.why;
        return -6;
    }
    DeviceGuard guard_(ctx->device);
    nccl_release(ctx);
    NcclUniqueIdBytes id;
    memcpy(id.internal, id128, sizeof id.internal);
    const int rc = api.CommInitRank(&ctx->nccl_comm, nranks, id, rank);
    if (rc != 0) {
        ctx->nccl_comm = nullptr;
        return nccl_fail(ctx, "ncclCommInitRank", rc);
    }
    ctx->nccl_ranks = nranks;
    ctx->nccl_rank = rank;
    return 0;
}

int32_t diffopt_b200_nccl_destroy(diffopt_b200_ctx* ctx) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    nccl_release(ctx);
    return 0;
}

int32_t diffopt_b200_qp_batch_shared_grads(diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p, const double* z,
                                           const double* lam, const double* nu, const double* rev, double* out_flat, int32_t memspace,
                                           int32_t flags) {
    if (!ctx) return -1;
    if (B < 0 || n <= 0 || m < 0 || p < 0) BAD_ARG(ctx, "qp_batch_shared_grads: need B >= 0, n > 0, m >= 0, p >= 0");
    if (!out_flat || (B > 0 && (!z || !rev || (m > 0 && !lam) || (p > 0 && !nu)))) BAD_ARG(ctx, "qp_batch_shared_grads: missing argument");
    const bool allreduce = (flags & DIFFOPT_QP_ALLREDUCE) != 0, async = (flags & DIFFOPT_QP_ASYNC) != 0;
    if (async && memspace != DIFFOPT_B200_DEVICE) BAD_ARG(ctx, "qp_batch_shared_grads: DIFFOPT_QP_ASYNC needs device memory");
    if (allreduce && !ctx->nccl_comm) BAD_ARG(ctx, "qp_batch_shared_grads: DIFFOPT_QP_ALLREDUCE without diffopt_b200_nccl_init");
    DeviceGuard guard_(ctx->device);
    const int N = n + m + p;
    const int64_t per = (int64_t)n * n + n + (int64_t)m * n + m + (int64_t)p * n + p;
    const size_t d = sizeof(double);
    const void *dz = nullptr, *dl = nullptr, *dn = nullptr, *dr = nullptr;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[4], z, d * B * n, memspace, &dz));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[5], lam, d * B * m, memspace, &dl));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[6], nu, d * B * p, memspace, &dn));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[14], rev, d * B * N, memspace, &dr));
    void* dout = nullptr;
    DO_CUDA(ctx, stage_out_prepare(ctx->out[2], out_flat, d * per, memspace, &dout));
    int G = (int)std::min<int64_t>(ctx->sm_count, std::max<int64_t>(1, (B + 3) / 4));
    DO_CUDA(ctx, ctx->out[3].reserve(d * (size_t)G * (size_t)per));
    const size_t smem = d * (size_t)GR_STAGE * 2 * (size_t)N;
    if (smem > ctx->smem_optin) BAD_ARG(ctx, "qp_batch_shared_grads: n + m + p too large for the staging buffer");
    DO_CUDA(ctx, cudaFuncSetAttribute(shared_grads_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    shared_grads_partial_kernel<<<G, GR_THREADS, smem, ctx->stream>>>(B, n, m, p, (const double*)dz, (const double*)dl, (const double*)dn,
                                                                    (const double*)dr, ctx->out[3].as<double>());
    shared_grads_final_kernel<<<(unsigned)std::min<int64_t>((per + 255) / 256, ctx->sm_count * 4), 256, 0, ctx->stream>>>(
        per, G, ctx->out[3].as<double>(), (double*)dout);
    ctx->launches += 2;
    DO_CUDA(ctx, cudaGetLastError());
    if (allreduce) {  // also with a single rank: the collective path is the same code at any communicator size
        const int rc = nccl_api().AllReduce(dout, dout, (size_t)per, NCCL_DOUBLE, NCCL_SUM, ctx->nccl_comm, ctx->stream);
        if (rc != 0) return nccl_fail(ctx, "ncclAllReduce", rc);
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, stage_out_finish(ctx, dout, out_flat, d * per, memspace));
    if (async) return 0;
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}

int32_t diffopt_b200_qp_batch_solve_ex(diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p, const double* Q,
                                       const double* G, const double* A, const double* h, const double* z, const double* lam,
                                       const double* nu, const double* dQ, const double* dq, const double* dG, const double* dh,
                                       const double* dA, const double* db, const double* dl_dz, double* fwd_out, double* rev_out,
                                       int32_t* info, int32_t memspace, int32_t flags) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (B < 0 || n <= 0 || m < 0 || p < 0) BAD_ARG(ctx, "qp_batch_solve_ex: need B >= 0, n > 0, m >= 0, p >= 0");
    if (B == 0) return 0;
    if (!Q || !z || (m > 0 && (!G || !h || !lam)) || (p > 0 && (!A || !nu)))
        BAD_ARG(ctx, "qp_batch_solve_ex: Q, z (and G, h, lam when m > 0; A, nu when p > 0) are required");
    if (rev_out && !dl_dz) BAD_ARG(ctx, "qp_batch_solve_ex: rev_out requested without dl_dz");
    if (!fwd_out && !rev_out) BAD_ARG(ctx, "qp_batch_solve_ex: nothing to compute (fwd_out and rev_out are NULL)");
    const bool async = (flags & DIFFOPT_QP_ASYNC) != 0;
    if (async && memspace != DIFFOPT_B200_DEVICE) BAD_ARG(ctx, "qp_batch_solve_ex: DIFFOPT_QP_ASYNC needs device memory");
    const bool shm = (flags & DIFFOPT_QP_SHARED_MATRICES) != 0, shd = (flags & DIFFOPT_QP_SHARED_DIRECTION) != 0;
    const bool packed = (flags & DIFFOPT_QP_PACKED_Q) != 0;
    QpSolveArgs a{};
    a.B = B; a.n = n; a.m = m; a.p = p;
    a.shared = (shm ? 1 : 0) | (shd ? 2 : 0);
    const size_t d = sizeof(double);
    const int64_t Bm = shm ? 1 : B, Bd = shd ? 1 : B;
    const size_t qcount = packed ? (size_t)n * (n + 1) / 2 : (size_t)n * n;
    const void* ptr;
#define STAGE_EX(slot, field, src, batch, count)                                                                    \
    DO_CUDA(ctx, stage_in(ctx, ctx->in[slot], src, d * (size_t)(batch) * (size_t)(count), memspace, &ptr)); \
    a.field = (const double*)ptr;
    STAGE_EX(0, Q, Q, Bm, qcount)
    STAGE_EX(1, G, G, Bm, (size_t)m * n)
    STAGE_EX(2, A, A, Bm, (size_t)p * n)
    STAGE_EX(3, h, h, B, m)
    STAGE_EX(4, z, z, B, n)
    STAGE_EX(5, lam, lam, B, m)
    STAGE_EX(6, nu, nu, B, p)
    if (fwd_out) {
        STAGE_EX(7, dQ, dQ, Bd, qcount)
        STAGE_EX(8, dq, dq, B, n)
        STAGE_EX(9, dG, dG, Bd, (size_t)m * n)
        STAGE_EX(10, dh, dh, B, m)
        STAGE_EX(11, dA, dA, Bd, (size_t)p * n)
        STAGE_EX(12, db, db, B, p)
    }
    if (rev_out) { STAGE_EX(13, seed, dl_dz, B, n) }
#undef STAGE_EX
    if (packed) {  // symmetric matrices arrive as lower triangles: expand on the device (HBM traffic, not PCIe)
        const dim3 grid((unsigned)std::min<int>((n * n + 255) / 256, 64), (unsigned)std::min<int64_t>(Bm, 32768));
        DO_CUDA(ctx, ctx->qp_unpacked[0].reserve(d * (size_t)Bm * n * n));
        unpack_lower_kernel<<<grid, 256, 0, ctx->stream>>>(a.Q, ctx->qp_unpacked[0].as<double>(), n, Bm);
        a.Q = ctx->qp_unpacked[0].as<double>();
        ctx->launches++;
        if (fwd_out && a.dQ) {
            const dim3 gridd((unsigned)std::min<int>((n * n + 255) / 256, 64), (unsigned)std::min<int64_t>(Bd, 32768));
            DO_CUDA(ctx, ctx->qp_unpacked[1].reserve(d * (size_t)Bd * n * n));
            unpack_lower_kernel<<<gridd, 256, 0, ctx->stream>>>(a.dQ, ctx->qp_unpacked[1].as<double>(), n, Bd);
            a.dQ = ctx->qp_unpacked[1].as<double>();
            ctx->launches++;
        }
        DO_CUDA(ctx, cudaGetLastError());
    }
    return qp_solve_common(ctx, a, fwd_out, rev_out, info, memspace, async);
}

int32_t diffopt_b200_qp_batch_solve_coo(diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p, const double* Q,
                                        const double* G, const double* A, const double* h, const double* z, const double* lam,
                                        const double* nu, const diffopt_b200_coo_batch* dQ, const double* dq,
                                        const diffopt_b200_coo_batch* dG, const double* dh, const diffopt_b200_coo_batch* dA,
                                        const double* db, const double* dl_dz, double* fwd_out, double* rev_out, int32_t* info,
                                        int32_t memspace, int32_t flags) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (B < 0 || n <= 0 || m < 0 || p < 0) BAD_ARG(ctx, "qp_batch_solve_coo: need B >= 0, n > 0, m >= 0, p >= 0");
    if (B == 0) return 0;
    if (!Q || !z || (m > 0 && (!G || !h || !lam)) || (p > 0 && (!A || !nu)))
        BAD_ARG(ctx, "qp_batch_solve_coo: Q, z (and G, h, lam when m > 0; A, nu when p > 0) are required");
    if (!fwd_out) BAD_ARG(ctx, "qp_batch_solve_coo: fwd_out is required (use qp_batch_solve for reverse mode alone)");
    if (rev_out && !dl_dz) BAD_ARG(ctx, "qp_batch_solve_coo: rev_out requested without dl_dz");
    if (flags & ~(DIFFOPT_QP_SHARED_MATRICES | DIFFOPT_QP_SHARED_DIRECTION | DIFFOPT_QP_ASYNC))
        BAD_ARG(ctx, "qp_batch_solve_coo: flags may hold SHARED_MATRICES, SHARED_DIRECTION, ASYNC");
    const bool async = (flags & DIFFOPT_QP_ASYNC) != 0;
    if (async && memspace != DIFFOPT_B200_DEVICE) BAD_ARG(ctx, "qp_batch_solve_coo: DIFFOPT_QP_ASYNC needs device memory");
    const bool shm = (flags & DIFFOPT_QP_SHARED_MATRICES) != 0, shd = (flags & DIFFOPT_QP_SHARED_DIRECTION) != 0;
    QpSolveArgs a{};
    a.B = B; a.n = n; a.m = m; a.p = p;
    a.shared = shm ? 1 : 0;
    const size_t d = sizeof(double);
    const int64_t Bm = shm ? 1 : B, Bd = shd ? 1 : B;
    const void* ptr;
    const double *ddq = nullptr, *ddh = nullptr, *ddb = nullptr;
#define STAGE_COO(slot, dst, src, count)                                                             \
    DO_CUDA(ctx, stage_in(ctx, ctx->in[slot], src, d * (size_t)(count), memspace, &ptr)); \
    dst = (const double*)ptr;
    STAGE_COO(0, a.Q, Q, (size_t)Bm * n * n)
    STAGE_COO(1, a.G, G, (size_t)Bm * m * n)
    STAGE_COO(2, a.A, A, (size_t)Bm * p * n)
    STAGE_COO(3, a.h, h, (size_t)B * m)
    STAGE_COO(4, a.z, z, (size_t)B * n)
    STAGE_COO(5, a.lam, lam, (size_t)B * m)
    STAGE_COO(6, a.nu, nu, (size_t)B * p)
    STAGE_COO(8, ddq, dq, (size_t)B * n)
    STAGE_COO(10, ddh, dh, (size_t)B * m)
    STAGE_COO(12, ddb, db, (size_t)B * p)
    if (rev_out) { STAGE_COO(13, a.seed, dl_dz, (size_t)B * n) }
#undef STAGE_COO
    CooDev dev[3];
    const diffopt_b200_coo_batch* src[3] = {dQ, dG, dA};
    const int lim_rows[3] = {n, m, p};
    if (int32_t rc = stage_triplets(ctx, "qp_batch_solve_coo", src, lim_rows, Bd, memspace, dev)) return rc;
    const int N = n + m + p;
    DO_CUDA(ctx, ctx->qp_coo[3].reserve(d * (size_t)B * N + sizeof(int)));
    double* rhs = ctx->qp_coo[3].as<double>();
    int* derr = reinterpret_cast<int*>(rhs + (size_t)B * N);
    DO_CUDA(ctx, cudaMemsetAsync(derr, 0, sizeof(int), ctx->stream));
    const int64_t blocks = std::min<int64_t>((B + 63) / 64, (int64_t)ctx->sm_count * 8);
    qp_coo_rhs_kernel<<<(unsigned)blocks, 64, 0, ctx->stream>>>(B, 1, n, m, p, a.z, a.lam, a.nu, dev[0], dev[1], dev[2], ddq, ddh, ddb,
                                                              shd ? 1 : 0, rhs, derr);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    a.rhs_pre = rhs;
    int32_t rc = qp_solve_common(ctx, a, fwd_out, rev_out, info, memspace, async);
    if (rc < 0 || async) return rc;
    int herr = 0;  // the blocking call has synchronised: out-of-range triplet indices are an argument error
    DO_CUDA(ctx, cudaMemcpy(&herr, derr, sizeof(int), cudaMemcpyDeviceToHost));
    if (herr) BAD_ARG(ctx, "qp_batch_solve_coo: a triplet index lies outside its matrix (1-based I, J expected)");
    return rc;
}

int32_t diffopt_b200_qp_batch_forward_multi(diffopt_b200_ctx* ctx, int64_t k, const diffopt_b200_coo_batch* dQ, const double* dq,
                                            const diffopt_b200_coo_batch* dG, const double* dh, const diffopt_b200_coo_batch* dA,
                                            const double* db, double* fwd_out, int32_t memspace) {
    if (!ctx) return -1;
    DeviceGuard guard_(ctx->device);
    if (!ctx->qpf.valid) BAD_ARG(ctx, "qp_batch_forward_multi: call qp_batch_factorize first (qp_batch_setup drops the stored factor)");
    if (k < 0) BAD_ARG(ctx, "qp_batch_forward_multi: need k >= 0");
    const QpBatchState& s = ctx->qp;
    const int64_t B = s.B;
    const int n = s.n, m = s.m, p = s.p, N = n + m + p;
    if (k == 0 || B == 0) return 0;
    if (!fwd_out) BAD_ARG(ctx, "qp_batch_forward_multi: fwd_out is required");
    const int64_t S = B * k;  // direction j of instance b is slot b k + j
    const size_t d = sizeof(double);
    const void *ddq, *ddh, *ddb;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[8], dq, d * (size_t)S * n, memspace, &ddq));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[10], dh, d * (size_t)S * m, memspace, &ddh));
    DO_CUDA(ctx, stage_in(ctx, ctx->in[12], db, d * (size_t)S * p, memspace, &ddb));
    CooDev dev[3];
    const diffopt_b200_coo_batch* src[3] = {dQ, dG, dA};
    const int lim_rows[3] = {n, m, p};
    if (int32_t rc = stage_triplets(ctx, "qp_batch_forward_multi", src, lim_rows, S, memspace, dev)) return rc;
    DO_CUDA(ctx, ctx->qp_coo[3].reserve(d * (size_t)S * N + sizeof(int)));
    double* rhs = ctx->qp_coo[3].as<double>();
    int* derr = reinterpret_cast<int*>(rhs + (size_t)S * N);
    DO_CUDA(ctx, cudaMemsetAsync(derr, 0, sizeof(int), ctx->stream));
    const int64_t blocks = std::max<int64_t>(1, std::min<int64_t>((S + 63) / 64, (int64_t)ctx->sm_count * 8));
    qp_coo_rhs_kernel<<<(unsigned)blocks, 64, 0, ctx->stream>>>(B, k, n, m, p, s.z.as<double>(), s.lam.as<double>(), s.nu.as<double>(),
                                                              dev[0], dev[1], dev[2], (const double*)ddq, (const double*)ddh,
                                                              (const double*)ddb, 0, rhs, derr);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    const int32_t rc = qp_factored_run(ctx, k, rhs, fwd_out, memspace, true);
    if (rc < 0) return rc;
    int herr = 0;  // qp_factored_run has synchronised: out-of-range triplet indices are an argument error
    DO_CUDA(ctx, cudaMemcpy(&herr, derr, sizeof(int), cudaMemcpyDeviceToHost));
    if (herr) BAD_ARG(ctx, "qp_batch_forward_multi: a triplet index lies outside its matrix (1-based I, J expected)");
    return rc;
}

}  // extern "C"
