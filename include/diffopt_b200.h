/*
 * diffopt_b200.h -- C ABI of the B200-native DiffOpt.jl sensitivity hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain C, opaque handle, plain
 * pointers and sizes.  It is what a Julia `ccall` (see INTEGRATION.md and
 * julia/DiffOptB200.jl) or any other FFI binds.  All references below are to the
 * reference tree andrewrosemberg/DiffOpt.jl v0.5.0.
 *
 * Conventions
 *  - every entry point returns int32 status: 0 ok; >0 LAPACK-style info (first
 *    instance/pivot that failed, 1-based); <0 bad argument / unsupported shape /
 *    CUDA error (text via diffopt_b200_last_error).  Nothing throws or aborts.
 *  - all floating point data is IEEE fp64.  Dense matrices are COLUMN-MAJOR (Julia
 *    layout) per instance, batches are instance-major (instance b starts at
 *    b * rows * cols).
 *  - `memspace` says where EVERY data pointer of that call lives:
 *    DIFFOPT_B200_HOST (pageable or pinned host memory; copies happen inside the
 *    call) or DIFFOPT_B200_DEVICE (device memory of the ctx's GPU; no copies).
 *  - calls are blocking (the ctx stream is synchronised before return), so the
 *    reference's `diff_time = @elapsed ...` (QuadraticProgram.jl:317,358;
 *    ConicProgram.jl:258,337) stays truthful.  One ctx per GPU; a ctx is not
 *    thread-safe.
 *  - lam / nu are the reference's stored duals, i.e. the NEGATED MOI duals
 *    (QuadraticProgram.jl:156-180).
 */
#ifndef DIFFOPT_B200_H
#define DIFFOPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct diffopt_b200_ctx diffopt_b200_ctx;

#define DIFFOPT_B200_HOST 0
#define DIFFOPT_B200_DEVICE 1

/* cone type codes for the conic entry points (dual cone is taken internally,
 * diff_opt.jl:496,515) */
#define DIFFOPT_CONE_ZERO 0   /* MOI.Zeros           */
#define DIFFOPT_CONE_NONNEG 1 /* MOI.Nonnegatives    */
#define DIFFOPT_CONE_SOC 2    /* MOI.SecondOrderCone */
#define DIFFOPT_CONE_PSD 3    /* MOI.PositiveSemidefiniteConeTriangle (unscaled, column-wise upper) */
/* MOI.ExponentialCone K = cl{(x, y, z) : y > 0, y e^(x/y) <= z}, dimension 3; pi onto K* (Moreau:
 * Pi_K*(v) = v + Pi_K(-v), DPi_K*(v) = I - DPi_K(-v)) */
#define DIFFOPT_CONE_EXP 4
/* MOI.DualExponentialCone K* = cl{(u, v, w) : u < 0, -u e^(v/u) <= e w}, dimension 3; pi onto K.
 * Pi_K(v), v = (r, s, t), cases in this order (the order decides ties): v in K -> v, I;
 * v in -K* -> 0, 0; r <= 0 and s <= 0 -> (r, 0, max(t, 0)), diag(1, 0, [t > 0]);
 * else the curved boundary (root of Friberg's univariate h), symmetric 3 x 3 Jacobian. */
#define DIFFOPT_CONE_DUAL_EXP 5
/* MOI.PowerCone(a) K_a = {(x, y, z) : x >= 0, y >= 0, x^a y^(1-a) >= |z|}, dimension 3, 0 < a < 1 (the exponent of
 * each power cone is passed in cone_param of conic_setup_ex); pi onto K_a* (Moreau: Pi_K*(v) = v + Pi_K(-v),
 * DPi_K*(v) = I - DPi_K(-v)) */
#define DIFFOPT_CONE_POW 6
/* MOI.DualPowerCone(a) K_a* = {(u, v, w) : u >= 0, v >= 0, (u/a)^a (v/(1-a))^(1-a) >= |w|}, dimension 3; pi onto K_a.
 * Pi_K(v), v = (x0, y0, z0), cases in this order (the order decides ties): v in K -> v, I; v in -K* -> 0, 0;
 * z0 = 0 -> (max(x0, 0), max(y0, 0), 0), diag([x0 > 0], [y0 > 0], 0); else the curved boundary (root of Hien's
 * univariate psi), symmetric 3 x 3 Jacobian. */
#define DIFFOPT_CONE_DUAL_POW 7

/* ---- lifetime ------------------------------------------------------------------- */
int32_t diffopt_b200_version(void);
/* Fails (<0) when no CUDA device / wrong architecture: there is no CPU fallback. */
int32_t diffopt_b200_create(int32_t device, diffopt_b200_ctx** out);
int32_t diffopt_b200_destroy(diffopt_b200_ctx* ctx);
const char* diffopt_b200_last_error(diffopt_b200_ctx* ctx);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
int64_t diffopt_b200_launch_count(diffopt_b200_ctx* ctx);
/* the ctx's cudaStream_t (as void*), so a caller that owns device buffers can order work */
void* diffopt_b200_stream(diffopt_b200_ctx* ctx);
/* pinned host buffers for callers that want full-speed PCIe copies */
int32_t diffopt_b200_host_alloc(void** ptr, int64_t bytes);
int32_t diffopt_b200_host_free(void* ptr);
/* device time (ms, CUDA events on the ctx stream) of the kernels of the last call */
double diffopt_b200_last_kernel_ms(diffopt_b200_ctx* ctx);

/* ---- QuadraticProgram backend: batched dense KKT sensitivities --------------------
 *
 * Replaces, for a batch of B independent QPs with n variables, m inequality rows
 * (G z <= h) and p equality rows (A z = b):
 *   create_LHS_matrix        QuadraticProgram.jl:256-282
 *   reverse_differentiate!   QuadraticProgram.jl:316-351   (RHS = [dl_dz; 0; 0], solve with LHS)
 *   forward_differentiate!   QuadraticProgram.jl:357-446   (RHS :429-433, solve with LHS')
 *   solve_system (direct)    QuadraticProgram.jl:486-492   (`LHS \ RHS`)
 * Outputs are the reference's (dz, dlam, dnu) = -solve(...), concatenated per
 * instance as N = n+m+p doubles.
 *
 * Q[B][n*n], G[B][m*n], A[B][p*n] column-major; h[B][m], z[B][n], lam[B][m], nu[B][p].
 * Forward direction (any of these may be NULL = zero): dQ[B][n*n] (symmetric, as
 * sparse_array_representation gives it), dq[B][n], dG[B][m*n], dh[B][m], dA[B][p*n],
 * db[B][p] in the reference's packed sign convention (db,dh = -constant,
 * QuadraticProgram.jl:374-395).  dl_dz[B][n] is the reverse seed.
 * fwd_out / rev_out [B][N] may be NULL to skip that mode.  info[B] (may be NULL):
 * 0, or nonzero when the factorisation met an exactly zero pivot (the reference throws
 * SingularException there).  The nonzero value is a 1-based position in the elimination order
 * of the kernel that served the instance (the tuned kernels eliminate a reduced, reordered
 * system), so it identifies "singular", not a row of LHS.
 * Return: 0, or (first failing instance + 1) if any info != 0.
 * Any shape is accepted.  Regular instances (Q positive definite, strict complementarity, independent active rows) run the
 * pivot-free LDL' fast path when their reduced system -- n variables + active inequalities + p equalities, at most about
 * 216 unknowns -- fits one CTA's shared memory; every other instance is solved by a partially pivoted LU of the full
 * KKT matrix (in shared memory up to n+m+p = 165, in global memory beyond: correct, slow).  -3: the KKT matrix of one
 * instance exceeds the 1 GiB scratch buffer (use diffopt_b200_sparse_setup / kkt_solve_csc for one large system).
 */
int32_t diffopt_b200_qp_batch_solve(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* Q, const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu,
    const double* dQ, const double* dq, const double* dG, const double* dh,
    const double* dA, const double* db, const double* dl_dz,
    double* fwd_out, double* rev_out, int32_t* info, int32_t memspace);

/* Stream-ordered form for device-resident pipelines (memspace must be DIFFOPT_B200_DEVICE, e.g. CUDA.jl arrays):
 * the same work is enqueued on the ctx stream and the call returns without waiting, so consecutive batches run back
 * to back with no host round trip in between.  `diffopt_b200_synchronize` waits for the stream and returns 0, or
 * (first failing instance + 1) of the EARLIEST call enqueued since the previous synchronize that met a singular
 * instance (every queued call is covered: the kernels record failures in a device word; the message of
 * diffopt_b200_last_error names the call) -- the blocking form above is this pair in one call, which is what the
 * reference's `@elapsed` timing (QuadraticProgram.jl:317,358) needs.  `info`, when given, must be a distinct device
 * array per queued call. */
int32_t diffopt_b200_qp_batch_solve_async(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* Q, const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu,
    const double* dQ, const double* dq, const double* dG, const double* dh,
    const double* dA, const double* db, const double* dl_dz,
    double* fwd_out, double* rev_out, int32_t* info);
int32_t diffopt_b200_synchronize(diffopt_b200_ctx* ctx);
/* Diagnostics of the last qp_batch call on this ctx (waits for the stream): out3[0] = instances the pivot-free LDL'
 * fast path handed to the partially pivoted LU kernel (semidefinite Q, rank-deficient active set, ... -- results are
 * the same, throughput is not), out3[1] = active-set size the launch was configured for, out3[2] = kernel that served
 * the call (0 generic pivoted LU, 1 tuned pivoted LU, 2 LDL' fast path, 3 stored LDL' of qp_batch_factorize -- then out3[0]
 * counts the instances the multi calls serve with the pivoted LU and out3[1] is the tile order the factors were stored for). */
int32_t diffopt_b200_qp_batch_last_stats(diffopt_b200_ctx* ctx, int64_t* out3);

/* Extended form of qp_batch_solve.  flags (OR of):
 *   DIFFOPT_QP_SHARED_MATRICES  Q, G, A are ONE instance ([n*n], [m*n], [p*n]) shared by all B problems -- an OptNet-style
 *                               layer whose weights do not depend on the sample (docs/src/examples/polyhedral_project.jl,
 *                               custom-relu.jl); h, z, lam, nu and the seeds stay per instance;
 *   DIFFOPT_QP_SHARED_DIRECTION dQ, dG, dA are one instance shared by the batch (a perturbation of the shared weights);
 *   DIFFOPT_QP_PACKED_Q         Q and dQ hold only their lower triangles, packed column by column (n(n+1)/2 doubles per
 *                               instance: column j = rows j..n-1) -- both are symmetric (utils.jl:46-69), so half of their
 *                               bytes over PCIe are redundant;
 *   DIFFOPT_QP_ASYNC            stream-ordered like qp_batch_solve_async (memspace must be DIFFOPT_B200_DEVICE). */
#define DIFFOPT_QP_SHARED_MATRICES 1
#define DIFFOPT_QP_SHARED_DIRECTION 2
#define DIFFOPT_QP_PACKED_Q 4
#define DIFFOPT_QP_ASYNC 8
#define DIFFOPT_QP_ALLREDUCE 16
int32_t diffopt_b200_qp_batch_solve_ex(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* Q, const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu,
    const double* dQ, const double* dq, const double* dG, const double* dh,
    const double* dA, const double* db, const double* dl_dz,
    double* fwd_out, double* rev_out, int32_t* info, int32_t memspace, int32_t flags);

/* Forward direction given as SPARSE TRIPLETS, the way the reference holds it: src/diff_opt.jl:594-656 collects (I, J, V)
 * per matrix from the perturbed constraint / objective functions and QuadraticProgram.jl:396-424 turns them into
 * SparseArrays.sparse(I, J, V, rows, n) (duplicates add up) before forming the right-hand side (:429-433).  The dense form
 * above moves n*n + m*n + p*n doubles per instance for a direction that usually has a handful of entries; here the
 * right-hand side is assembled on the device from the triplets and the dense matrices never exist.
 *   ptr[b] .. ptr[b+1]-1 (0-based offsets, ptr[0] = 0, B+1 entries; 2 entries with DIFFOPT_QP_SHARED_DIRECTION) are the
 *   triplets of instance b; I, J are 1-based (Julia's); dQ triplets name the full symmetric matrix (both triangles), as the
 *   reference's sparse dQ does.  A NULL struct pointer or NULL ptr means the matrix is zero.  The struct lives in host
 *   memory; the arrays it points to live in `memspace`.
 * flags: DIFFOPT_QP_SHARED_MATRICES, DIFFOPT_QP_SHARED_DIRECTION, DIFFOPT_QP_ASYNC.  fwd_out is required; rev_out / dl_dz
 * optional as in qp_batch_solve.  Returns as qp_batch_solve; -1 when a triplet index lies outside its matrix. */
typedef struct diffopt_b200_coo_batch {
    const int64_t* ptr;
    const int64_t* I;
    const int64_t* J;
    const double* V;
} diffopt_b200_coo_batch;
int32_t diffopt_b200_qp_batch_solve_coo(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* Q, const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu,
    const diffopt_b200_coo_batch* dQ, const double* dq, const diffopt_b200_coo_batch* dG, const double* dh,
    const diffopt_b200_coo_batch* dA, const double* db, const double* dl_dz,
    double* fwd_out, double* rev_out, int32_t* info, int32_t memspace, int32_t flags);

/* Reverse-mode gradients of parameters SHARED by the B instances (the getters of QuadraticProgram.jl:307-314, :448-473
 * accumulated over the samples as docs/src/examples/polyhedral_project.jl:95-104 and src/parameters.jl:355-360 do):
 * out_flat = [dQ (n*n, column-major) | dq (n) | dG (m*n) | dh (m) | dA (p*n) | db (p)], each the SUM over the batch of
 *   dQ = (dz z' + z dz')/2, dq = dz, dG_i = lam_i dlam_i z + lam_i dz, dh = -lam.dlam, dA_i = dnu_i z + nu_i dz, db = -dnu
 * from rev[B][n+m+p] = (dz, dlam, dnu) (the rev_out of a qp_batch call) and z, lam, nu of the same instances.  The sum is
 * formed on the device in a fixed order (bitwise reproducible).  flags: DIFFOPT_QP_ALLREDUCE adds ONE fp64 ncclAllReduce
 * (sum) of out_flat over the ranks of diffopt_b200_nccl_init -- every rank owns a shard of the batch, the buffer never
 * leaves the GPUs; DIFFOPT_QP_ASYNC enqueues on the ctx stream without waiting (device memory only). */
int32_t diffopt_b200_qp_batch_shared_grads(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* z, const double* lam, const double* nu, const double* rev,
    double* out_flat, int32_t memspace, int32_t flags);

/* NCCL communicator owned by the ctx (one rank per ctx / GPU).  Rank 0 obtains a 128-byte ncclUniqueId with
 * nccl_unique_id and hands it to the other ranks by whatever means the host program has (MPI, torch.distributed,
 * a file); every rank then calls nccl_init.  NCCL is bound at run time (libnccl.so.2 of the host process, or
 * DIFFOPT_B200_NCCL_LIB); -6 = not available. */
int32_t diffopt_b200_nccl_unique_id(void* id128);
int32_t diffopt_b200_nccl_init(diffopt_b200_ctx* ctx, int32_t nranks, int32_t rank, const void* id128);
int32_t diffopt_b200_nccl_destroy(diffopt_b200_ctx* ctx);

/* Two-phase form mirroring the reference's cache (`_gradient_cache` builds LHS once,
 * QuadraticProgram.jl:182-213; seeds may then change): setup keeps the problem data
 * resident on the device, forward/reverse solve against it. */
int32_t diffopt_b200_qp_batch_setup(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* Q, const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu, int32_t memspace);
int32_t diffopt_b200_qp_batch_reverse(
    diffopt_b200_ctx* ctx, const double* dl_dz, double* rev_out, int32_t* info, int32_t memspace);
int32_t diffopt_b200_qp_batch_forward(
    diffopt_b200_ctx* ctx, const double* dQ, const double* dq, const double* dG,
    const double* dh, const double* dA, const double* db,
    double* fwd_out, int32_t* info, int32_t memspace);

/* Factorise once, solve many directions.  qp_batch_factorize (after qp_batch_setup) computes the LDL' factor of every
 * instance's reduced KKT system and keeps it on the device (about 40 KB per instance at n=64, m=64, p=16 with 16 active
 * rows); a new qp_batch_setup drops it, destroy frees it.  The multi calls then take k directions per instance and cost two
 * triangular sweeps over the stored factor per direction instead of a full assembly and factorisation.  Instances the
 * pivot-free factorisation rejects (semidefinite Q, rank-deficient active set, wrong-sign duals, an active set beyond shared
 * memory) are listed at factorize time and solved by the pivoted LU, one launch per direction.
 *   factorize: info[B] (may be NULL) as in qp_batch_solve.  Returns 0, first singular instance + 1, -3 when the factor
 *     storage cannot be allocated.
 *   reverse_multi: dl_dz[B][k][n] (instance-major, then direction: Julia's Array{Float64,3} of size (n, k, B)) ->
 *     rev_out[B][k][N], direction j of instance b = what qp_batch_reverse returns for that seed (to rounding: the sums run
 *     in another order).
 *   forward_multi: dq[B][k][n], dh[B][k][m], db[B][k][p] (any may be NULL = zero); dQ, dG, dA as in qp_batch_solve_coo
 *     with B*k+1 offsets (direction j of instance b is slot b*k + j) -> fwd_out[B][k][N], direction j of instance b = what
 *     qp_batch_forward returns for that direction.  -1 when a triplet index lies outside its matrix.
 *   Both return 0, first singular instance + 1, or < 0 (a call before factorize, or after a new setup, is -1 and
 *   diffopt_b200_last_error names the missing step); k = 0 returns 0. */
int32_t diffopt_b200_qp_batch_factorize(diffopt_b200_ctx* ctx, int32_t* info, int32_t memspace);
int32_t diffopt_b200_qp_batch_reverse_multi(
    diffopt_b200_ctx* ctx, int64_t k, const double* dl_dz, double* rev_out, int32_t memspace);
int32_t diffopt_b200_qp_batch_forward_multi(
    diffopt_b200_ctx* ctx, int64_t k,
    const diffopt_b200_coo_batch* dQ, const double* dq, const diffopt_b200_coo_batch* dG, const double* dh,
    const diffopt_b200_coo_batch* dA, const double* db, double* fwd_out, int32_t memspace);

/* The LSQR branch of solve_system for a batch of B LPs (Q = 0, QuadraticProgram.jl:333-335, :436-438, :486-488):
 * per instance, LHS = [0 G'diag(lam) A'; G diag(Gz-h) 0; A 0 0] (create_LHS_matrix with Q = 0);
 * rev_out = -lsqr(LHS, [dl_dz; 0; 0]), fwd_out = -lsqr(LHS', RHS of :429-433), from x0 = 0 with (atol, btol, conlim,
 * maxiter) -- maxiter = 0 means N = n+m+p, IterativeSolvers' max(size(LHS)).  Arguments as qp_batch_solve without Q
 * (dQ still enters the forward right-hand side through dQ z); any direction array may be NULL (zero); fwd_out / rev_out
 * may be NULL to skip that mode.  stats_out[B][2][4] (may be NULL) = (istop, itn, rnorm, arnorm) of the forward, then
 * the reverse solve (zeros for a skipped mode).  flags: DIFFOPT_QP_SHARED_MATRICES (G, A one instance for the batch).
 * An LP's KKT matrix is singular whenever the solution is not a nondegenerate vertex; LSQR then returns the minimum-norm
 * least-squares answer, as the reference does, where the direct entries above report the instance singular.
 * Each instance is solved by one CTA, bitwise reproducibly and independently of the rest of the batch.
 * Never reports singular: returns 0, < 0 for bad arguments / unknown flags / CUDA errors, -3 for an instance whose
 * LSQR vectors do not fit one CTA (use the single-instance lsqr_csc route).  Blocking; last_kernel_ms is its device time. */
int32_t diffopt_b200_qp_batch_solve_lsqr(
    diffopt_b200_ctx* ctx, int64_t B, int32_t n, int32_t m, int32_t p,
    const double* G, const double* A, const double* h,
    const double* z, const double* lam, const double* nu,
    const double* dQ, const double* dq, const double* dG, const double* dh,
    const double* dA, const double* db, const double* dl_dz,
    double atol, double btol, double conlim, int64_t maxiter,
    double* fwd_out, double* rev_out, double* stats_out, int32_t memspace, int32_t flags);

/* Reverse-mode gradients w.r.t. the problem data from rev = (dz, dlam, dnu)
 * (getters QuadraticProgram.jl:307-314, :448-473; signs as the reference's tests read
 * them, test/utils.jl:178-233):
 *   dQ = (dz z' + z dz')/2, dq = dz, dG_i = lam_i dlam_i z + lam_i dz, dh = -lam.dlam,
 *   dA_i = dnu_i z + nu_i dz, db = -dnu.
 * reduce_over_batch = 0: outputs are per instance ([B][...]); 1: summed over the
 * batch into single-instance sized outputs (parameters shared across instances --
 * the local half of the multi-GPU all-reduce, SURVEY.md 8e).  Needs a prior
 * qp_batch_setup (z, lam, nu resident).  Any output may be NULL. */
int32_t diffopt_b200_qp_batch_param_grads(
    diffopt_b200_ctx* ctx, const double* rev, int32_t reduce_over_batch,
    double* dQ, double* dq, double* dG, double* dh, double* dA, double* db, int32_t memspace);

/* ---- direct branch of solve_system for one KKT system (QuadraticProgram.jl:486-492: `LHS \ RHS`) --------------
 *
 * LHS is Julia's SparseMatrixCSC{Float64,Int} (colptr/rowval 1-based int64, N x N); trans = 1 solves with LHS'
 * (the `Adjoint` forward_differentiate! passes, QuadraticProgram.jl:438).  rhs / x_out are N x nrhs column-major:
 * all right-hand sides share ONE partially pivoted LU factorisation (the reference refactorises per call).
 * Returns 0, or > 0 when the matrix is singular (an exactly zero pivot; reference: SingularException).
 * Small systems (N <= 1024) are densified and factorised by one CTA; larger ones go through the sparse
 * factorisation below (setup + solve in one call), as the reference's sparse `\` does at any size. */
int32_t diffopt_b200_kkt_solve_csc(
    diffopt_b200_ctx* ctx, int64_t N, const int64_t* colptr, const int64_t* rowval, const double* nzval,
    int32_t trans, int64_t nrhs, const double* rhs, double* x_out, int32_t memspace);

/* ---- sparse direct path: one large KKT system, many right-hand sides (BASELINE config 3) ----------------------
 *
 * sparse_setup factorises LHS (SparseMatrixCSC{Float64,Int} in HOST memory, 1-based; trans = 1: LHS') once and keeps
 * the factorisation in the ctx: `LHS \ RHS` of QuadraticProgram.jl:490 (UMFPACK in the reference) without the
 * reference's refactorisation per direction (:438).  Method: multifrontal LU for general patterns -- nested-dissection
 * ordering and symbolic factorisation on the host, fronts factorised level by level on the device with partial
 * pivoting inside each front (a front that needs a delayed pivot is merged into its parent and the factorisation
 * repeated until no front delays a pivot).
 * sparse_solve then solves for nrhs columns (rhs / x_out are N x nrhs column-major, host or device per memspace).
 * Returns 0; > 0: the matrix is singular (SingularException in the reference); -3: the factorisation cannot be held
 * (a front or the factor structure is too large).
 * bandwidth_out (may be NULL) receives -1. */
int32_t diffopt_b200_sparse_setup(
    diffopt_b200_ctx* ctx, int64_t N, const int64_t* colptr, const int64_t* rowval, const double* nzval,
    int32_t trans, int64_t* bandwidth_out);
int32_t diffopt_b200_sparse_solve(
    diffopt_b200_ctx* ctx, int64_t nrhs, const double* rhs, double* x_out, int32_t memspace);
/* out8 = {method (0 none, 2 multifrontal), fronts, tree levels, largest front order, nnz(L+U) stored,
 * factorisation flop, host analysis ms, delayed-pivot repetitions} of the factorisation held by the ctx. */
int32_t diffopt_b200_sparse_stats(diffopt_b200_ctx* ctx, double* out8);
/* Host-only analysis (ordering + symbolic factorisation, no GPU involved): out8 as above with out8[7] = number of
 * kernel launches one factorisation takes.  nzval may be NULL (no pairing of weak diagonals with a partner row). */
int32_t diffopt_b200_sparse_analyze(
    int64_t N, const int64_t* colptr, const int64_t* rowval, const double* nzval, int32_t trans, double* out8);

/* ---- LSQR (IterativeSolvers.lsqr call sites QuadraticProgram.jl:488, ConicProgram.jl:323,372)
 *
 * min ||M x - rhs|| from x0 = 0 on an explicit sparse matrix in Julia's
 * SparseMatrixCSC{Float64,Int} layout (colptr/rowval 1-based int64).  trans = 1 solves
 * with M' (the `Adjoint` the forward QP mode passes, QuadraticProgram.jl:438).
 * This is the iterative branch of `solve_system` (LP case, Q == 0).
 * out_stats[4] (may be NULL) = {istop, iterations, ||r|| estimate, ||M'r|| estimate}. */
int32_t diffopt_b200_lsqr_csc(
    diffopt_b200_ctx* ctx, int64_t nrows, int64_t ncols,
    const int64_t* colptr, const int64_t* rowval, const double* nzval, int32_t trans,
    const double* rhs, double atol, double btol, double conlim, int64_t maxiter,
    double* x_out, double* out_stats, int32_t memspace);

/* ---- ConicProgram backend ---------------------------------------------------------
 *
 * conic_setup replaces `_gradient_cache` (ConicProgram.jl:172-255): keeps A (m x n CSC,
 * already the reference's A = -coefficients), b, c, the solution (x, s, y) and the cone
 * list resident, computes v = y - s, vp = pi(v) (diff_opt.jl:491-499) and the
 * operator-form data of Dpi(v) (diff_opt.jl:509-519) -- dense blocks are never formed.
 * Cones are listed in row order: cone_type[i] in DIFFOPT_CONE_*, cone_dim[i] rows.
 */
int32_t diffopt_b200_conic_setup(
    diffopt_b200_ctx* ctx, int64_t n, int64_t m,
    const int64_t* A_colptr, const int64_t* A_rowval, const double* A_nzval,
    const double* b, const double* c, const double* x, const double* s, const double* y,
    int64_t ncones, const int32_t* cone_type, const int64_t* cone_dim, int32_t memspace);
/* conic_setup with one parameter per cone: cone_param[i] (in memspace, like cone_type) is the exponent a of cone i,
 * read only for DIFFOPT_CONE_POW / DIFFOPT_CONE_DUAL_POW, which need it (finite, 0 < a < 1; the end points are not
 * supported).  cone_param may be NULL when the list has no power cone; conic_setup is conic_setup_ex with NULL. */
int32_t diffopt_b200_conic_setup_ex(
    diffopt_b200_ctx* ctx, int64_t n, int64_t m,
    const int64_t* A_colptr, const int64_t* A_rowval, const double* A_nzval,
    const double* b, const double* c, const double* x, const double* s, const double* y,
    int64_t ncones, const int32_t* cone_type, const int64_t* cone_dim, const double* cone_param, int32_t memspace);
/* vp = pi(y - s) of the current setup (length m) */
int32_t diffopt_b200_conic_get_vp(diffopt_b200_ctx* ctx, double* vp_out, int32_t memspace);
/* out = Dpi(v) * t or Dpi(v)' * t (length m): the `Dπ` operator on its own */
int32_t diffopt_b200_conic_dpi_apply(
    diffopt_b200_ctx* ctx, const double* t, int32_t transpose, double* out, int32_t memspace);
/* out = M t or M' t, M as in ConicProgram.jl:243-247 (length n+m+1) */
int32_t diffopt_b200_conic_M_apply(
    diffopt_b200_ctx* ctx, const double* t, int32_t transpose, double* out, int32_t memspace);
/* forward_differentiate! (ConicProgram.jl:257-334): dA as COO triplets (1-based rows/cols,
 * duplicates summed, values as packed by the reference i.e. un-negated), db[m], dc[n];
 * dz_out[n+m+1] = lsqr(M, g) (zeros if ||g|| == 0); dx_out[n] = -(du - x dw) (:403-412).
 * Any of dA (nnz = 0), db, dc may be NULL. */
int32_t diffopt_b200_conic_forward(
    diffopt_b200_ctx* ctx, int64_t dA_nnz, const int64_t* dA_row, const int64_t* dA_col,
    const double* dA_val, const double* db, const double* dc,
    double atol, double btol, double conlim, int64_t maxiter,
    double* dx_out, double* dz_out, double* out_stats, int32_t memspace);
/* reverse_differentiate! (ConicProgram.jl:336-394): g_out[n+m+1] = lsqr(M, [dx; 0; -x'dx])
 * (zeros if the norm of that vector is <= 1e-4, :369).  Optional getters
 * (:396-428): dc_out[n] = g[1:n] - g[N] x ; db_out[m] = g[n+I] - g[N] vp. */
int32_t diffopt_b200_conic_reverse(
    diffopt_b200_ctx* ctx, const double* dx_seed,
    double atol, double btol, double conlim, int64_t maxiter,
    double* g_out, double* dc_out, double* db_out, double* out_stats, int32_t memspace);
/* Many directions against the current conic_setup (any cone kind), one LSQR launch for all of them; direction j gets
 * the single-direction semantics of conic_forward / conic_reverse, and its result does not depend on the other
 * directions of the call (bitwise).  Layout is direction-major: Julia's Matrix{Float64} of size (n, k) passes as is.
 * k forward directions of forward_differentiate! (ConicProgram.jl:257-334) against the current conic_setup.
 * dA: triplets with k+1 offsets (direction j = ptr[j] .. ptr[j+1]-1; 1-based rows / cols, duplicates summed,
 * un-negated as conic_forward takes them); NULL struct or NULL ptr = zero.  db[k][m], dc[k][n] (NULL = zero).
 * dx_out[k][n] = -(du - x dw), dz_out[k][n+m+1] (may be NULL), out_stats[k][4] = (istop, itn, rnorm, arnorm).
 * A direction with ||g_j|| = 0 (:320) returns zeros and stats (0, 0, 0, 0); maxiter = 0 means n+m+1.
 * Returns 0 for k = 0; -1 for k < 0, before conic_setup, or for a triplet outside the m x n matrix (conic_forward
 * skips such triplets). */
int32_t diffopt_b200_conic_forward_multi(
    diffopt_b200_ctx* ctx, int64_t k, const diffopt_b200_coo_batch* dA, const double* db, const double* dc,
    double atol, double btol, double conlim, int64_t maxiter,
    double* dx_out, double* dz_out, double* out_stats, int32_t memspace);
/* k reverse seeds of reverse_differentiate! (ConicProgram.jl:336-394): dx_seeds[k][n] ->
 * g_out[k][n+m+1], dc_out[k][n], db_out[k][m], out_stats[k][4]; any output may be NULL.  A seed whose right-hand side
 * has norm <= 1e-4 (:369) returns zeros. */
int32_t diffopt_b200_conic_reverse_multi(
    diffopt_b200_ctx* ctx, int64_t k, const double* dx_seeds,
    double atol, double btol, double conlim, int64_t maxiter,
    double* g_out, double* dc_out, double* db_out, double* out_stats, int32_t memspace);

/* Lock-step batch of conic problems: B independent problems of equal size (n, m; any sparsity / solution / cone
 * list without PSD cones), each analysed like conic_setup, then ALL reverse solves advanced by ONE persistent kernel
 * (problem p on its own CTA -- or cluster of `ctas_per_problem` CTAs -- with the gather vectors staged in shared
 * memory).  This is how a training loop calls the reference's one-problem-per-call `reverse_differentiate!`
 * (ConicProgram.jl:336-394) over a minibatch; every problem runs exactly the single-problem iteration (same
 * arithmetic, same stop tests, own iteration count).  Arrays are instance-major: dx_seeds[n,B], g_out[n+m+1,B],
 * dc_out[n,B], db_out[m,B], out_stats[4,B] = (istop, iterations, rnorm, arnorm) per problem. */
int32_t diffopt_b200_conic_batch_begin(diffopt_b200_ctx* ctx, int64_t B, int32_t ctas_per_problem);
int32_t diffopt_b200_conic_batch_add(
    diffopt_b200_ctx* ctx, int64_t n, int64_t m,
    const int64_t* A_colptr, const int64_t* A_rowval, const double* A_nzval,
    const double* b, const double* c, const double* x, const double* s, const double* y,
    int64_t ncones, const int32_t* cone_type, const int64_t* cone_dim, int32_t memspace);
/* conic_batch_add with the per-cone parameters of conic_setup_ex (cone_param may be NULL without power cones) */
int32_t diffopt_b200_conic_batch_add_ex(
    diffopt_b200_ctx* ctx, int64_t n, int64_t m,
    const int64_t* A_colptr, const int64_t* A_rowval, const double* A_nzval,
    const double* b, const double* c, const double* x, const double* s, const double* y,
    int64_t ncones, const int32_t* cone_type, const int64_t* cone_dim, const double* cone_param, int32_t memspace);
int32_t diffopt_b200_conic_batch_reverse(
    diffopt_b200_ctx* ctx, const double* dx_seeds,
    double atol, double btol, double conlim, int64_t maxiter,
    double* g_out, double* dc_out, double* db_out, double* out_stats, int32_t memspace);

/* ---- callers next to the hot path (SURVEY.md 8f) ------------------------------------------------------------------
 *
 * NonLinearProgram backend, `_lu_with_inertia_correction` (NonLinearProgram.jl:356-435): factorise M (host CSC, 1-based);
 * if the factorisation reports a singular matrix (`K.status == 1`), factorise J = M + c st D for c = 1, 2, ... until it
 * succeeds, D = diag(+1 on rows 1..num_w, -1 on the next num_cons rows, +1 on the rest), at most max_corrections
 * corrected factorisations.  corrections_out = c (0: M itself was fine).  Returns 0, or > 0 when the last attempt was
 * still singular (the reference warns "Inertia correction failed." and returns zeros).  The factorisation stays in the
 * ctx: `K \ N` for all parameter columns at once (nlp_utilities.jl:436-444, caller negates) is diffopt_b200_sparse_solve. */
int32_t diffopt_b200_sparse_setup_inertia(
    diffopt_b200_ctx* ctx, int64_t N, const int64_t* colptr, const int64_t* rowval, const double* nzval,
    int64_t num_w, int64_t num_cons, double st, int32_t max_corrections, int32_t* corrections_out);

/* Reverse-mode accumulation into parameters (src/parameters.jl:341-534): out[param] = sum over terms of
 * coef * flat[index], param / index 1-based, term lists in HOST memory (they describe the model), terms of one
 * parameter summed in the order given.  `flat` is a gradient block as diffopt_b200_qp_batch_shared_grads lays it out
 * ([dQ | dq | dG | dh | dA | db], host or device per memspace; device: the batch-summed, all-reduced block is consumed
 * in place).  How the reference's term kinds map to (index, coef): affine p term in constraint row i with coefficient c:
 * (dh_i or db_i, -c) -- the constant of ReverseConstraintFunction is -dh_i (QuadraticProgram.jl:307-314); p v term:
 * (dG_iv / dA_iv / dq_v, c); p p term: (dh_i or db_i, -c * value of the other parameter), once per parameter. */
int32_t diffopt_b200_param_pullback(
    diffopt_b200_ctx* ctx, int64_t nterms, const int64_t* term_param, const int64_t* term_index, const double* term_coef,
    int64_t nflat, const double* flat, int64_t nparams, double* out, int32_t memspace);

#ifdef __cplusplus
}
#endif
#endif /* DIFFOPT_B200_H */
