// Shared host-side plumbing of libdiffopt_b200: the opaque ctx, error handling and
// grow-only device buffers.  No torch types anywhere in this library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/diffopt_b200.h"

struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(ptr); }
};

// Resident state of a qp_batch_setup.
struct QpBatchState {
    int64_t B = 0;
    int n = 0, m = 0, p = 0;
    bool valid = false;
    DevBuf Q, G, A, h, z, lam, nu;  // device copies (or nothing when borrowed)
    const double *dQ_ = nullptr, *dG_ = nullptr, *dA_ = nullptr, *dh_ = nullptr, *dz_ = nullptr,
                 *dlam_ = nullptr, *dnu_ = nullptr;  // device pointers actually used
};

// LDL' factors of the setup's instances kept by qp_batch_factorize (FactorLayout in qp_sqd_dev.cuh); a new setup drops them.
struct QpFactorState {
    bool valid = false;
    int nt_cap = 0;      // tile order the factors were stored for (0: no instance fits, the pivoted LU serves the batch)
    int64_t stride = 0;  // doubles per instance
    int nrej = 0;        // instances served by the pivoted LU (listed in fb)
    DevBuf f;            // [B][stride] factors
    DevBuf fb;           // [count, list...] of those instances
    DevBuf gin, gout;    // one direction of the listed instances in the [B][...] layout the pivoted-LU kernel reads and writes
};

struct CsrDev {  // device CSR (0-based, int32 indices) of a sparse matrix and of its transpose
    int64_t nrows = 0, ncols = 0, nnz = 0;
    DevBuf rowptr, colind, val;     // A   (nrows x ncols)
    DevBuf t_rowptr, t_colind, t_val;  // A'  (ncols x nrows)
    // row blocks for the streaming SpMV (lsqr.cu): block k = rows [blk[k], blk[k+1]) holding <= ST_CHUNK nonzeros
    DevBuf blk, t_blk;
    int64_t nblk = 0, t_nblk = 0;
    bool sorted = false;  // column-ordered copies of the streaming blocks exist
    DevBuf sval, scol, spos, t_sval, t_scol, t_spos;
    DevBuf cblk, t_cblk;  // coarser blocks for the cluster-synchronised persistent kernel (16 CTAs)
    int64_t ncblk = 0, t_ncblk = 0;
    DevBuf gblk, t_gblk;  // ... and for the one-CTA-per-SM persistent kernel
    int64_t ngblk = 0, t_ngblk = 0;
};

struct ConicState {
    bool valid = false;
    int64_t n = 0, m = 0, ncones = 0;
    CsrDev A;
    DevBuf b, c, x, s, y, v, vp;
    // per-row cone metadata and per-cone data
    DevBuf row_kind;     // int8 per row: 0 zero / nonneg (diagonal), 2 soc, 3 psd, 4 + j row j of a 3 x 3 block cone
    DevBuf nn_scale;     // double per row: (sign(v)+1)/2 for nonneg rows, 1 for zero rows
    DevBuf soc_off, soc_dim, soc_case, soc_nx;  // per SOC cone
    int64_t nsoc = 0;
    // cones with a symmetric 3 x 3 Dpi block (exponential, dual exponential): first row, v negated (DIFFOPT_CONE_EXP:
    // pi onto K* = -(pi onto K°)(-v)); blk3: 3 coefficients per row of such a cone (row i: blk3[3 i .. 3 i + 2])
    DevBuf exp_off, exp_neg, blk3;
    int64_t nexp = 0;
    // power cones (same blk3 rows): first row, v negated (DIFFOPT_CONE_POW: pi onto K*), exponent
    DevBuf pow_off, pow_neg, pow_alpha;
    int64_t npow = 0;
    // PSD cones
    DevBuf psd_off, psd_d, psd_uoff;  // per PSD cone: row offset, side d, offset into U/B storage
    DevBuf psd_U, psd_Bm, psd_ident;  // eigenvectors (col-major d x d), B matrix, identity flag
    DevBuf psd_work;                  // scratch 3 * sum d^2
    DevBuf psd_toff;                  // tile offsets of the PSD apply (lsqr.cu)
    int64_t psd_ntiles = 0;
    DevBuf psd_lam, psd_loff;         // eigenvalues (+ shifts) and per-cone offsets into them (+ small-cone list)
    DevBuf psd_tri;                   // tau, diagonal, off-diagonal, scale, cluster flags of the tridiagonal route (psd_tridiag.cu)
    int64_t npsd = 0, psd_maxd = 0, psd_sumd2 = 0;
    std::vector<int64_t> h_psd_off, h_psd_d, h_psd_uoff;
    // work vectors for M apply / LSQR
    DevBuf w1, w2, w3;
};

struct NcclUniqueIdBytes { char internal[128]; };  // ncclUniqueId (nccl.h), passed by value to ncclCommInitRank
void nccl_release(struct diffopt_b200_ctx* ctx);

void conic_state_release(struct ConicState& c);
struct ConicBatchImpl;  // lock-step batch of conic problems (conic.cu)
void conic_batch_release(struct diffopt_b200_ctx* ctx);

struct SparseMfImpl;  // multifrontal factorisation kept by diffopt_b200_sparse_setup (sparse_mf.cu)
void sparse_mf_release(struct diffopt_b200_ctx* ctx);

struct LsqrWork {
    DevBuf u, v, w, x, tmp, scal;  // vectors and a small block of device scalars
};

struct diffopt_b200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    int64_t launches = 0;
    double last_ms = 0.0;
    int sm_count = 0;
    size_t smem_optin = 0;
    // generic staging buffers for HOST-memspace calls
    DevBuf in[16];
    DevBuf out[8];
    DevBuf info;
    DevBuf qp_fb;   // [count, list...] of instances the LDL' fast path hands to the pivoted LU kernel
    DevBuf qp_max;  // device scalar: largest active-set size of the batch
    // pinned ring of D2H copies of that word (slot = call number & 3), each followed by an event: a later call only
    // trusts a slot whose event has completed (stream-ordered calls do not end synchronised), newest call wins
    int* qp_hmax_host = nullptr;
    cudaEvent_t qp_hmax_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int64_t qp_hmax_call[4] = {-1, -1, -1, -1};  // host-side call counter of the copy in flight in each slot (-1: none)
    int64_t qp_calls = 0;
    int qp_last_kernel = -1;      // kernel of the last qp_batch call: 0 generic pivoted LU, 1 tuned pivoted LU, 2 LDL' fast path,
                                  // 3 stored LDL' (qp_batch_factorize)
    int qp_last_hint = -1;        // active-set size that launch was configured for
    int qp_seq = 0;               // call number, tags the active-set word written by the LDL' kernel
    int qp_hint = -1;             // active-set size the next launch of the LDL' fast path is configured for (-1: unknown)
    int64_t qp_hint_shape = -1;   // (n, m, p) that hint belongs to
    // stream-ordered calls: every kernel that finds a singular instance lowers this device word with atomicMin to
    // (call number << 32 | instance + 1); diffopt_b200_synchronize reads it, so a failure in ANY queued call surfaces
    DevBuf qp_sticky;
    unsigned async_calls = 0;     // calls enqueued since the last synchronize
    bool async_pending = false;
    QpBatchState qp;
    QpFactorState qpf;
    ConicState conic;
    LsqrWork lsqr;
    CsrDev lsqr_mat;
    void* nccl_comm = nullptr;    // ncclComm_t of diffopt_b200_nccl_init (one rank per ctx)
    int nccl_ranks = 0, nccl_rank = 0;
    DevBuf qp_unpacked[2];        // Q / dQ expanded from packed lower triangles (qp_batch_solve_ex)
    DevBuf qp_scratch;            // KKT matrices of the generic pivoted-LU kernel when they exceed shared memory
    DevBuf qp_coo[4];             // staged triplets of dQ, dG, dA and the assembled right-hand side (qp_batch_solve_coo)
    ConicBatchImpl* conic_batch = nullptr;
    int csr_cluster_ctas = 0;     // CTAs the cluster-kernel row blocks of csr_from_csc_host are cut for (0: default 16)
    SparseMfImpl* sparse_mf = nullptr;
    int sparse_method = 0;        // factorisation currently held: 0 none, 2 multifrontal LU
    int64_t sparse_N = 0;
};

// Launch configuration of a kernel at one dynamic shared-memory size: the attribute call is made only when the size differs
// from the last one set for this (kernel, device), the occupancy answer is cached.  Both runtime calls cost host
// microseconds per call, which a stream of small batches (512 instances per rank at 8 GPUs: 50 us of device time per
// call) cannot hide.
inline cudaError_t kernel_config(const void* kernel, int device, int threads, size_t smem, int* per_sm) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> last_smem;
    static std::map<std::tuple<const void*, int, int, size_t>, int> occupancy;
    std::lock_guard<std::mutex> lock(mu);
    auto ls = last_smem.find({kernel, device});
    if (ls == last_smem.end() || ls->second != smem) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        last_smem[{kernel, device}] = smem;
    }
    if (per_sm) {
        auto key = std::make_tuple(kernel, device, threads, smem);
        auto oc = occupancy.find(key);
        if (oc == occupancy.end()) {
            int n = 1;
            cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem);
            if (e != cudaSuccess) return e;
            oc = occupancy.emplace(key, n).first;
        }
        *per_sm = oc->second;
    }
    return cudaSuccess;
}

// Entry points make the ctx's device current for their duration and restore the caller's device on exit (a host
// process that drives several GPUs, e.g. through torch or CUDA.jl, keeps its own current device).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

#define DO_CUDA(ctx, expr)                                                              \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) {                                                        \
            char _b[512];                                                               \
            snprintf(_b, sizeof _b, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,       \
                     cudaGetErrorString(_e));                                           \
            (ctx)->err = _b;                                                            \
            return -100 - (int32_t)_e;                                                  \
        }                                                                               \
    } while (0)

#define BAD_ARG(ctx, msg)   \
    do {                    \
        (ctx)->err = (msg); \
        return -1;          \
    } while (0)

// Copies `bytes` from src (host or device per memspace) into buf (device) unless src is
// already a device pointer, in which case it is used in place.  Returns the device pointer.
static inline cudaError_t stage_in(diffopt_b200_ctx* ctx, DevBuf& buf, const void* src, size_t bytes,
                                   int memspace, const void** dev_out) {
    if (src == nullptr || bytes == 0) {
        *dev_out = nullptr;
        return cudaSuccess;
    }
    if (memspace == DIFFOPT_B200_DEVICE) {
        *dev_out = src;
        return cudaSuccess;
    }
    cudaError_t e = buf.reserve(bytes);
    if (e != cudaSuccess) return e;
    *dev_out = buf.ptr;
    return cudaMemcpyAsync(buf.ptr, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
}

static inline cudaError_t stage_out_prepare(DevBuf& buf, void* dst, size_t bytes, int memspace, void** dev_out) {
    if (dst == nullptr || bytes == 0) {
        *dev_out = nullptr;
        return cudaSuccess;
    }
    if (memspace == DIFFOPT_B200_DEVICE) {
        *dev_out = dst;
        return cudaSuccess;
    }
    cudaError_t e = buf.reserve(bytes);
    if (e != cudaSuccess) return e;
    *dev_out = buf.ptr;
    return cudaSuccess;
}

static inline cudaError_t stage_out_finish(diffopt_b200_ctx* ctx, void* dev, void* dst, size_t bytes, int memspace) {
    if (dst == nullptr || bytes == 0 || memspace == DIFFOPT_B200_DEVICE) return cudaSuccess;
    return cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream);
}

// kernel-side launchers implemented in the .cu files -------------------------------------
struct QpSolveArgs {
    int64_t B;
    int n, m, p;
    const double *Q, *G, *A, *h, *z, *lam, *nu;
    const double *dQ, *dq, *dG, *dh, *dA, *db, *seed;
    double *fwd, *rev;
    int* info;
    long long* prof;  // optional per-phase clock counters of CTA 0 (DIFFOPT_B200_PROFILE=1)
    unsigned long long* sticky;  // optional: first failing (call, instance) of a stream-ordered sequence of calls
    unsigned call_seq;
    int shared;  // bit 0: Q, G, A are ONE instance shared by the whole batch; bit 1: dQ, dG, dA likewise
    // optional: forward right-hand side already assembled on the device from sparse triplets (qp_batch_solve_coo),
    // [B][n+m+p] = [dQ z + dq + dG'lam + dA'nu; dG z - dh; dA z - db]; dQ .. db are then unused
    const double* rhs_pre;
};

// what a kernel does when instance `inst` turned out singular in a stream-ordered call
__device__ __forceinline__ void qp_report_sticky(const QpSolveArgs& a, long long inst) {
    if (a.sticky) atomicMin(a.sticky, ((unsigned long long)a.call_seq << 32) | (unsigned)(inst + 1));
}
int32_t psd_eig_launch(diffopt_b200_ctx* ctx, const std::vector<int>& h_d, const std::vector<long long>& h_uoff,
                       const std::vector<int>& h_off);
int32_t qp_batch_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a);
int32_t qp_param_grads_launch(diffopt_b200_ctx* ctx, int64_t B, int n, int m, int p, const double* z,
                              const double* lam, const double* nu, const double* rev, int reduce,
                              double* dQ, double* dq, double* dG, double* dh, double* dA, double* db);
