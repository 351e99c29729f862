// Sparse direct path for general patterns: multifrontal LU with partial pivoting inside the fronts, for ONE large KKT
// system with many right-hand sides -- `LHS \ RHS` of QuadraticProgram.jl:486-492 (UMFPACK in the reference), BASELINE
// config 3.  The reference refactorises for every direction (:438); here the factorisation stays in the ctx.
//
// Host (analysis, once per pattern):
//   * symmetrised pattern; vertices of very high degree (dense rows/columns such as a budget constraint) are set aside
//     and eliminated last in one top front;
//   * nested dissection by BFS level structures (George): a connected region is cut at the smallest level near its
//     middle, thinned to the vertices that actually touch the far side; regions of <= LEAF vertices become leaf fronts,
//     tiny components are packed together into one leaf; every separator is one front;
//   * symbolic factorisation on that supernode partition: row structure of every front, assembly tree, relative
//     indices child -> parent, destination of every matrix entry, tree levels.
// Device (numeric):
//   * factorisation level by level, ONE CTA PER FRONT, fronts of a level batched in one launch: the front is assembled
//     in shared memory (matrix entries + extend-add of the children's contribution blocks in a fixed order, so the
//     result is deterministic), its fully-summed block is eliminated with partial pivoting among the fully-summed rows
//     (threshold test against the whole column; a front that would need a DELAYED pivot is reported, merged into its
//     parent on the host and the factorisation repeated), the Schur complement is passed up;
//   * multi-RHS solves level by level, one CTA per (front, tile of 64 right-hand sides), one thread per column of the
//     tile: leaves gather their rows straight from the caller's column-major block and scatter the solution straight
//     back, so the N x nrhs block crosses HBM four times in total (read b, write y, read y, write x).
// Fronts beyond shared memory are processed in place in global memory by the same code (correct, not tuned).
#include <algorithm>
#include <chrono>
#include <numeric>
#include <vector>

#include "common.cuh"

namespace {

constexpr int MF_TC = 64;            // right-hand sides per solve CTA (one thread each)
constexpr int MF_FACT_THREADS = 256;
constexpr int MF_BIG_THREADS = 1024;
constexpr double MF_PIV_U = 1e-3;    // threshold: |pivot| >= u * max|column| (rows not yet fully summed included)
constexpr size_t MF_SMEM_CAP = 200 * 1024;

struct MfFront {
    int k, s, first, parent;    // fully-summed columns, boundary rows, first permuted position, parent front (-1: root)
    int soff;                   // offset of the boundary list (permuted positions) and of the relative indices into the parent
    int c0, c1;                 // children: child_idx[c0 .. c1)
    int a0, a1;                 // matrix entries: aloc/asrc[a0 .. a1)
    int leaf;
    int u0, un;                 // forward sweep: uptr[u0 .. u0 + nf] delimits, per row of the front (before interchanges), the
                                // workspace rows of the children that are added to it (usrc, un entries in total)
    long long lp, up, cb, w;    // offsets: L panel (nf x k), U panel (k x s), contribution block (s x s), solve workspace row
};

// ---------------------------------------------------------------------------------------------------------------
// numeric factorisation of one front (F: nf x nf column-major with leading dimension ld, in shared or global memory)
template <int THREADS>
__device__ void mf_factor_front(const MfFront fr, double* F, const int ld, double* rinv, const MfFront* fronts, const int* child_idx,
                                const int* rel, const int* aloc, const int* asrc, const double* vals, double* Lp, double* Up,
                                double* CB, int* piv, int* status, const int fid) {
    __shared__ int sh_p, sh_flag;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = fr.k, s = fr.s, nf = k + s;
    for (int i = tid; i < nf * ld; i += THREADS) F[i] = 0.0;
    if (tid == 0) sh_flag = 0;
    __syncthreads();
    for (int e = fr.a0 + tid; e < fr.a1; e += THREADS) {
        const int loc = aloc[e];
        atomicAdd(&F[(loc % nf) + (loc / nf) * ld], vals[asrc[e]]);
    }
    __syncthreads();
    for (int ci = fr.c0; ci < fr.c1; ++ci) {  // extend-add, children in list order (deterministic sums)
        const MfFront ch = fronts[child_idx[ci]];
        const int sc = ch.s;
        const int* r = rel + ch.soff;
        const double* cb = CB + ch.cb;
        for (int b = warp; b < sc; b += THREADS / 32) {   // lanes run down a column of the child's block (coalesced, no div/mod)
            const int rb = r[b] * ld;
            const double* cbb = cb + (size_t)b * sc;
            int a = lane;
            for (; a + 96 < sc; a += 128) {   // four entries in flight (distinct targets: the relative indices are injective)
                double* t0 = F + r[a] + rb;
                double* t1 = F + r[a + 32] + rb;
                double* t2 = F + r[a + 64] + rb;
                double* t3 = F + r[a + 96] + rb;
                const double v0 = cbb[a], v1 = cbb[a + 32], v2 = cbb[a + 64], v3 = cbb[a + 96];
                const double f0 = *t0, f1 = *t1, f2 = *t2, f3 = *t3;
                *t0 = f0 + v0;
                *t1 = f1 + v1;
                *t2 = f2 + v2;
                *t3 = f3 + v3;
            }
            for (; a < sc; a += 32) F[r[a] + rb] += cbb[a];
        }
        __syncthreads();
    }
    for (int j = 0; j < k; ++j) {
        if (warp == 0) {  // pivot search: largest entry among the fully-summed rows, and the column's largest overall
            double best = -1.0, rest = 0.0;
            int bi = j;
            for (int i = j + lane; i < nf; i += 32) {
                const double a = fabs(F[i + j * ld]);
                if (i < k) {
                    if (a > best) { best = a; bi = i; }
                } else if (a > rest) rest = a;
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o), orr = __shfl_xor_sync(0xffffffffu, rest, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
                rest = fmax(rest, orr);
            }
            // a pivot that fails the threshold test is still taken when its ROW has nothing else left (a row singleton,
            // e.g. the row of an inactive inequality in LHS': x = r / D exactly): its multipliers only ever meet zeros
            bool weak = best > 0.0 && best < MF_PIV_U * rest;
            if (weak) {
                double rmax = 0.0;
                for (int c = j + 1 + lane; c < nf; c += 32) rmax = fmax(rmax, fabs(F[bi + c * ld]));
#pragma unroll
                for (int o = 16; o; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
                if (rmax == 0.0) weak = false;
            }
            if (lane == 0) {
                sh_p = bi;
                if (!(best > 0.0)) {
                    if (rest > 0.0) sh_flag |= 2;   // only rows that are not fully summed could pivot: delayed pivot needed
                    else sh_flag |= 1;              // the whole column is zero: the matrix is singular
                } else if (weak) sh_flag |= 2;
            }
        }
        __syncthreads();
        const int p = sh_p;
        if (p != j)
            for (int c = tid; c < nf; c += THREADS) {
                const double t = F[j + c * ld];
                F[j + c * ld] = F[p + c * ld];
                F[p + c * ld] = t;
            }
        __syncthreads();
        const double pv = F[j + j * ld];
        const double ri = pv != 0.0 ? 1.0 / pv : 0.0;
        if (tid == 0) {
            rinv[j] = ri;
            piv[fr.first + j] = p;
        }
        // rank-1 update: lanes <-> rows (their multiplier in a register), warps <-> columns (the pivot-row entry is a broadcast)
        for (int i = j + 1 + lane; i < nf; i += 32) {
            const double l = -(F[i + j * ld] * ri);
            double* Fi = F + i;
            const double* Fj = F + j;
            constexpr int NW = THREADS / 32;
            int c = j + 1 + warp;
            for (; c + 3 * NW < nf; c += 4 * NW) {   // four columns in flight (row j and row i never alias: i > j)
                const double u0 = Fj[c * ld], u1 = Fj[(c + NW) * ld], u2 = Fj[(c + 2 * NW) * ld], u3 = Fj[(c + 3 * NW) * ld];
                const double f0 = Fi[c * ld], f1 = Fi[(c + NW) * ld], f2 = Fi[(c + 2 * NW) * ld], f3 = Fi[(c + 3 * NW) * ld];
                Fi[c * ld] = fma(l, u0, f0);
                Fi[(c + NW) * ld] = fma(l, u1, f1);
                Fi[(c + 2 * NW) * ld] = fma(l, u2, f2);
                Fi[(c + 3 * NW) * ld] = fma(l, u3, f3);
            }
            for (; c < nf; c += NW) Fi[c * ld] = fma(l, Fj[c * ld], Fi[c * ld]);
        }
        __syncthreads();
    }
    // write-back: L panel (unit-lower L11 scaled, U11 on and above the diagonal, L21), U12, contribution block
    for (int c = warp; c < k; c += THREADS / 32) {
        const double rc = rinv[c];
        for (int r = lane; r < nf; r += 32) Lp[fr.lp + r + (size_t)c * nf] = r > c ? F[r + c * ld] * rc : F[r + c * ld];
    }
    for (int t = warp; t < s; t += THREADS / 32) {
        for (int r = lane; r < k; r += 32) Up[fr.up + r + (size_t)t * k] = F[r + (k + t) * ld];
        for (int r = lane; r < s; r += 32) CB[fr.cb + r + (size_t)t * s] = F[(k + r) + (k + t) * ld];
    }
    if (tid == 0) status[fid] = sh_flag;
    __syncthreads();
}

// THREADS follows the front size: a launch group whose fronts leave room for one or two CTAs per SM runs them with 1024 / 512
// threads, so that the SM still has warps to overlap the dependent steps of the elimination.
template <int THREADS>
__global__ void __launch_bounds__(THREADS) mf_factor_kernel(const int* list, const MfFront* fronts, const int* child_idx, const int* rel,
                                                            const int* aloc, const int* asrc, const double* vals, double* Lp,
                                                            double* Up, double* CB, int* piv, int* status) {
    extern __shared__ __align__(16) double mf_smem[];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int nf = fr.k + fr.s, ld = nf | 1;
    mf_factor_front<THREADS>(fr, mf_smem, ld, mf_smem + (size_t)nf * ld, fronts, child_idx, rel, aloc, asrc, vals, Lp, Up, CB, piv, status,
                             fid);
}

// fronts beyond shared memory: the same elimination in a global scratch area (scratch[b]: nf * ld + k doubles)
__global__ void __launch_bounds__(MF_BIG_THREADS) mf_factor_big_kernel(const int* list, const long long* scratch_off, double* scratch,
                                                                       const MfFront* fronts, const int* child_idx, const int* rel,
                                                                       const int* aloc, const int* asrc, const double* vals, double* Lp,
                                                                       double* Up, double* CB, int* piv, int* status) {
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int nf = fr.k + fr.s, ld = nf | 1;
    double* F = scratch + scratch_off[blockIdx.x];
    mf_factor_front<MF_BIG_THREADS>(fr, F, ld, F + (size_t)nf * ld, fronts, child_idx, rel, aloc, asrc, vals, Lp, Up, CB, piv, status,
                                    fid);
}

// ---------------------------------------------------------------------------------------------------------------
// solves.  Y: N x nrhs row-major in PERMUTED row order (y after the forward sweep, x of the separator rows after the
// backward sweep); W: per-front boundary updates (s x nrhs row-major).  SMALL: factor panels and the tile of the
// right-hand sides in shared memory.  BIG: everything stays in global memory (Y itself is the work area).
template <bool BIG>
__global__ void __launch_bounds__(MF_TC) mf_forward_kernel(const int* list, const MfFront* fronts, const int* child_idx, const int* rel,
                                                           const int* perm, const int* piv, const double* Lp, const double* B,
                                                           double* Y, double* W, const long long N, const int nrhs) {
    extern __shared__ __align__(16) double mf_smem[];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int k = fr.k, s = fr.s, nf = k + s;
    const int c0 = blockIdx.y * MF_TC, tid = threadIdx.x, col = c0 + tid;
    const int ncol = min(MF_TC, nrhs - c0);
    const int ldy = (k | 1), ldw = (s | 1);
    double* Ls = mf_smem;                                   // nf x k            (SMALL)
    double* Ys = BIG ? nullptr : Ls + (size_t)nf * k;       // [col][r], ld ldy
    double* Ws = BIG ? nullptr : Ys + (size_t)MF_TC * ldy;  // [col][t], ld ldw
    const double* L = Lp + fr.lp;
    if (!BIG) {
        for (int i = tid; i < nf * k; i += MF_TC) Ls[i] = L[i];
        // own rows from the caller's column-major block: consecutive threads take consecutive rows of one column
        for (int idx = tid; idx < k * ncol; idx += MF_TC) {
            const int r = idx % k, c = idx / k;
            Ys[c * ldy + r] = B[(size_t)perm[fr.first + r] + (size_t)N * (c0 + c)];
        }
        for (int i = tid; i < MF_TC * ldw; i += MF_TC) Ws[i] = 0.0;
        __syncthreads();
        L = Ls;
    } else {
        for (int idx = tid; idx < k * ncol; idx += MF_TC) {
            const int r = idx % k, c = idx / k;
            Y[(size_t)(fr.first + r) * nrhs + c0 + c] = B[(size_t)perm[fr.first + r] + (size_t)N * (c0 + c)];
        }
        __syncthreads();
    }
    if (tid >= ncol) return;
    double* y = BIG ? Y + (size_t)fr.first * nrhs + col : Ys + tid * ldy;
    const size_t ys = BIG ? (size_t)nrhs : 1;
    double* w = BIG ? W + (size_t)fr.w * nrhs + col : Ws + tid * ldw;
    const size_t ws = BIG ? (size_t)nrhs : 1;
    if (BIG)
        for (int t = 0; t < s; ++t) w[t * ws] = 0.0;
    for (int ci = fr.c0; ci < fr.c1; ++ci) {  // updates of the children, in list order
        const MfFront ch = fronts[child_idx[ci]];
        const int* r = rel + ch.soff;
        const double* cw = W + (size_t)ch.w * nrhs + col;
        for (int t = 0; t < ch.s; ++t) {
            const int loc = r[t];
            const double v = cw[(size_t)t * nrhs];
            if (loc < k) y[loc * ys] += v;
            else w[(loc - k) * ws] += v;
        }
    }
    const int* pv = piv + fr.first;
    for (int j = 0; j < k; ++j) {
        const int p = pv[j];
        if (p != j) {
            const double t = y[j * ys];
            y[j * ys] = y[p * ys];
            y[p * ys] = t;
        }
    }
    for (int i = 1; i < k; ++i) {  // unit-lower L11
        double acc = y[i * ys], acc2 = 0.0;
        int j = 0;
        for (; j + 1 < i; j += 2) {
            acc = fma(-L[i + (size_t)j * nf], y[j * ys], acc);
            acc2 = fma(-L[i + (size_t)(j + 1) * nf], y[(j + 1) * ys], acc2);
        }
        if (j < i) acc = fma(-L[i + (size_t)j * nf], y[j * ys], acc);
        y[i * ys] = acc + acc2;
    }
    double* wout = W + (size_t)fr.w * nrhs + col;
    for (int t = 0; t < s; ++t) {  // boundary update  w -= L21 y
        double acc = w[t * ws], acc2 = 0.0;
        int j = 0;
        for (; j + 1 < k; j += 2) {
            acc = fma(-L[k + t + (size_t)j * nf], y[j * ys], acc);
            acc2 = fma(-L[k + t + (size_t)(j + 1) * nf], y[(j + 1) * ys], acc2);
        }
        if (j < k) acc = fma(-L[k + t + (size_t)j * nf], y[j * ys], acc);
        wout[(size_t)t * nrhs] = acc + acc2;
    }
    if (!BIG) {
        double* yo = Y + (size_t)fr.first * nrhs + col;
        for (int r = 0; r < k; ++r) yo[(size_t)r * nrhs] = y[r];
    }
}

template <bool BIG>
__global__ void __launch_bounds__(MF_TC) mf_backward_kernel(const int* list, const MfFront* fronts, const int* strct, const int* perm,
                                                            const double* Lp, const double* Up, double* Y, double* X, const long long N,
                                                            const int nrhs) {
    extern __shared__ __align__(16) double mf_smem[];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int k = fr.k, s = fr.s, nf = k + s;
    const int c0 = blockIdx.y * MF_TC, tid = threadIdx.x, col = c0 + tid;
    const int ncol = min(MF_TC, nrhs - c0);
    if (k == 0) return;                                       // assembly node: nothing to solve
    const int ldy = (k | 1), ldw = (s | 1);
    double* U11s = mf_smem;                                   // k x k (upper part of the L panel), ld k
    double* U12s = BIG ? nullptr : U11s + (size_t)k * k;      // k x s
    double* Ys = BIG ? nullptr : U12s + (size_t)k * s;        // [col][r]
    double* Xs = BIG ? nullptr : Ys + (size_t)MF_TC * ldy;    // [col][t]
    const double* U11 = Lp + fr.lp;
    const double* U12 = Up + fr.up;
    int ldu = nf;
    if (!BIG) {
        for (int i = tid; i < k * k; i += MF_TC) U11s[i] = U11[(i % k) + (size_t)(i / k) * nf];
        for (int i = tid; i < k * s; i += MF_TC) U12s[i] = U12[i];
        __syncthreads();
        U11 = U11s;
        U12 = U12s;
        ldu = k;
    }
    if (tid < ncol) {
        double* y = BIG ? Y + (size_t)fr.first * nrhs + col : Ys + tid * ldy;
        const size_t ys = BIG ? (size_t)nrhs : 1;
        const int* sp = strct + fr.soff;
        if (!BIG) {
            const double* yi = Y + (size_t)fr.first * nrhs + col;
            for (int r = 0; r < k; ++r) y[r] = yi[(size_t)r * nrhs];
            double* x2 = Xs + tid * ldw;
            for (int t = 0; t < s; ++t) x2[t] = Y[(size_t)sp[t] * nrhs + col];
        }
        for (int i = k - 1; i >= 0; --i) {
            double acc = y[i * ys], acc2 = 0.0;
            if (!BIG) {
                const double* x2 = Xs + tid * ldw;
                int t = 0;
                for (; t + 1 < s; t += 2) {
                    acc = fma(-U12[i + (size_t)t * k], x2[t], acc);
                    acc2 = fma(-U12[i + (size_t)(t + 1) * k], x2[t + 1], acc2);
                }
                if (t < s) acc = fma(-U12[i + (size_t)t * k], x2[t], acc);
            } else {
                for (int t = 0; t < s; ++t) acc = fma(-U12[i + (size_t)t * k], Y[(size_t)sp[t] * nrhs + col], acc);
            }
            int j = i + 1;
            for (; j + 1 < k; j += 2) {
                acc = fma(-U11[i + (size_t)j * ldu], y[j * ys], acc);
                acc2 = fma(-U11[i + (size_t)(j + 1) * ldu], y[(j + 1) * ys], acc2);
            }
            if (j < k) acc = fma(-U11[i + (size_t)j * ldu], y[j * ys], acc);
            y[i * ys] = (acc + acc2) / U11[i + (size_t)i * ldu];
        }
        if (!BIG && !fr.leaf) {  // separator rows are read by the fronts below
            double* yo = Y + (size_t)fr.first * nrhs + col;
            for (int r = 0; r < k; ++r) yo[(size_t)r * nrhs] = y[r];
        }
    }
    __syncthreads();
    // solution rows back into the caller's column-major block (consecutive threads: consecutive rows of one column)
    for (int idx = tid; idx < k * ncol; idx += MF_TC) {
        const int r = idx % k, c = idx / k;
        const double v = BIG ? Y[(size_t)(fr.first + r) * nrhs + c0 + c] : Ys[c * ldy + r];
        X[(size_t)perm[fr.first + r] + (size_t)N * (c0 + c)] = v;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Separator fronts that fit shared memory: one CTA per (front, tile of 64 right-hand sides), 256 threads = 64 columns x
// 4 row groups.  The tile of the right-hand sides lives in shared memory as YW[row][column] (rows 0..k-1: the front's
// own unknowns, rows k..nf-1: its boundary), the factor panel streams through shared memory in blocks of MF_NB columns
// (next block in flight in registers while the current one is applied).  Per block every thread solves the MF_NB x MF_NB
// diagonal block for its column redundantly in registers and then updates the rows it owns (row groups interleaved),
// so a front of order k costs k / MF_NB short steps instead of one thread walking k^2 / 2 + k s dependent FMAs.
// Row interchanges enter as the NET permutation of the front (psrc / pdst, mf_netperm_kernel).
constexpr int MF_TT = 256;
constexpr int MF_RG = MF_TT / MF_TC;   // row groups
constexpr int MF_NB = 8;               // columns per block step of the tiled sweeps (16 measured slower: registers)
constexpr int MF_LDT = MF_TC + 1;      // leading dimension of YW: conflict-free by row and by column
constexpr int MF_BT_MIN_BLOCKS = 4;    // resident CTAs per SM the backward tiled kernel is compiled for (64 registers, 24 bytes of spills)
constexpr int MF_US_CAP = 8192;        // update lists up to this many entries are staged in shared memory
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc) {   // one double, global -> shared, no register staging
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ double ld_b(const double* p) { return __ldg(p); }
__device__ __forceinline__ void st_x(double* p, const double v) { *p = v; }

// one CTA per front: net effect of the front's row interchanges.  psrc[first + r] = row (0..k-1, before the interchanges)
// that ends at position r; pdst = inverse.
__global__ void __launch_bounds__(64) mf_netperm_kernel(const MfFront* fronts, const int nfronts, const int* piv, int* psrc, int* pdst) {
    extern __shared__ int np_smem[];
    for (int fid = blockIdx.x; fid < nfronts; fid += gridDim.x) {
        const MfFront fr = fronts[fid];
        const int k = fr.k;
        int* src = np_smem;
        int* pv = np_smem + k;
        for (int r = threadIdx.x; r < k; r += blockDim.x) {
            src[r] = r;
            pv[r] = piv[fr.first + r];
        }
        __syncthreads();
        if (threadIdx.x == 0)
            for (int j = 0; j < k; ++j) {
                const int p = pv[j];
                const int t = src[j];
                src[j] = src[p];
                src[p] = t;
            }
        __syncthreads();
        for (int r = threadIdx.x; r < k; r += blockDim.x) {
            psrc[fr.first + r] = src[r];
            pdst[fr.first + src[r]] = r;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(MF_TT) mf_forward_tiled_kernel(const int* list, const MfFront* fronts, const int* uptr, const int* usrc,
                                                                 const int* perm, const int* psrc, const double* Lp,
                                                                 const double* B, double* Y, double* W, const long long N, const int nrhs) {
    extern __shared__ __align__(16) double mf_smem[];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int k = fr.k, s = fr.s, nf = k + s;
    const int tid = threadIdx.x, c = tid & (MF_TC - 1), q = tid >> 6, lane = tid & 31, wid = tid >> 5;
    const int c0 = blockIdx.y * MF_TC, col = c0 + c;
    const int ncol = min(MF_TC, nrhs - c0);
    const bool live = col < nrhs;
    double* YW = mf_smem;                                  // [nf][MF_LDT]
    double* Lb = YW + (size_t)nf * MF_LDT;                 // [nf][MF_NB]: rows jb.. of the current column block (16-byte aligned:
    Lb += ((size_t)nf * MF_LDT) & 1;                       //  odd offsets are bumped)
    int* rows = reinterpret_cast<int*>(Lb + (size_t)nf * MF_NB);  // original row of position r
    int* locs = rows + k;                                  // row of the front (before the interchanges) at position r
    int* up = locs + k;                                    // nf + 1 offsets into us (children's updates per row)
    int* us = up + nf + 1;                                 // workspace rows of the children, fr.un entries
    const double* L = Lp + fr.lp;
    double lreg[MF_NB];
    auto prefetch = [&](const int jb) {
        const int nbk = min(MF_NB, k - jb);
        const int i = jb + tid;
#pragma unroll
        for (int jj = 0; jj < MF_NB; ++jj) lreg[jj] = (i < nf && jj < nbk) ? L[i + (size_t)(jb + jj) * nf] : 0.0;
    };
    prefetch(0);   // first panel block in flight under the gathers below
    {   // ... and the whole panel on its way into L2: the block steps below then wait for an L2 hit, not for DRAM
        const char* pb = reinterpret_cast<const char*>(L);
        const size_t bytes = (size_t)nf * k * sizeof(double);
        for (size_t off = (size_t)tid * 128; off < bytes; off += (size_t)MF_TT * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pb + off));
    }
    for (int r = tid; r < k; r += MF_TT) {
        const int loc = psrc[fr.first + r];
        locs[r] = loc;
        rows[r] = perm[fr.first + loc];
    }
    {
        const int ub = uptr[fr.u0];
        for (int r = tid; r <= nf; r += MF_TT) up[r] = uptr[fr.u0 + r] - ub;
        if (fr.un <= MF_US_CAP)
            for (int e = tid; e < fr.un; e += MF_TT) us[e] = usrc[ub + e];
    }
    // (a front with thousands of children -- the top front of an arrowhead -- reads its list from global memory)
    const int* const ulist = fr.un <= MF_US_CAP ? us : usrc + uptr[fr.u0];
    __syncthreads();
    // own rows from the caller's column-major block (lanes: consecutive positions of one column), boundary rows zero
    for (int r = lane; r < k; r += 32) {   // asynchronous copies: every entry of the tile in flight at once
        const double* src = B + (size_t)rows[r] + (size_t)N * c0;
        double* dst = YW + r * MF_LDT;
#pragma unroll
        for (int u = 0; u < MF_TC / (MF_TT / 32); ++u) {
            const int cc = wid + u * (MF_TT / 32);
            if (cc < ncol) cp_async8(dst + cc, src + (size_t)N * cc);
        }
    }
    cp_async_wait_all();
    __syncthreads();
    // extend-add as a gather: every row of the tile is owned by one thread per column, which adds the children's
    // workspace rows that land on it in the children's list order (deterministic; no barrier per child)
    // (four rows per pass with the first two entries of each in flight together: a row of a front with two children has
    // at most two entries, so a pass costs one global round trip instead of four)
    if (live)
        for (int pos0 = q; pos0 < nf; pos0 += 4 * MF_RG) {
            int e0[4], e1[4];
            double v0[4], v1[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int pos = pos0 + u * MF_RG;
                const int loc = pos < nf ? (pos < k ? locs[pos] : pos) : 0;
                e0[u] = pos < nf ? up[loc] : 0;
                e1[u] = pos < nf ? up[loc + 1] : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                v0[u] = e0[u] < e1[u] ? W[(size_t)ulist[e0[u]] * nrhs + col] : 0.0;
                v1[u] = e0[u] + 1 < e1[u] ? W[(size_t)ulist[e0[u] + 1] * nrhs + col] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int pos = pos0 + u * MF_RG;
                if (pos >= nf) break;
                double acc = pos < k ? YW[pos * MF_LDT + c] : 0.0;
                acc += v0[u];
                acc += v1[u];
                int e = e0[u] + 2;
                const int ee = e1[u];
                for (; e + 8 <= ee; e += 8) {   // eight loads in flight, added in list order
                    double v[8];
#pragma unroll
                    for (int w = 0; w < 8; ++w) v[w] = W[(size_t)ulist[e + w] * nrhs + col];
#pragma unroll
                    for (int w = 0; w < 8; ++w) acc += v[w];
                }
                for (; e < ee; ++e) acc += W[(size_t)ulist[e] * nrhs + col];
                YW[pos * MF_LDT + c] = acc;
            }
        }
    // blocked forward substitution with the unit-lower L11 and the boundary update w -= L21 y in one sweep over the rows
    for (int jb = 0; jb < k; jb += MF_NB) {
        const int nbk = min(MF_NB, k - jb);
        __syncthreads();   // the previous block's reads of Lb and its row updates are complete
        if (jb + tid < nf) {
            double2* dst = reinterpret_cast<double2*>(Lb + (size_t)tid * MF_NB);
#pragma unroll
            for (int jj = 0; jj < MF_NB; jj += 2) dst[jj >> 1] = make_double2(lreg[jj], lreg[jj + 1]);
        }
        __syncthreads();
        if (jb + MF_NB < k) prefetch(jb + MF_NB);
        double yb[MF_NB];
#pragma unroll
        for (int jj = 0; jj < MF_NB; ++jj) yb[jj] = jj < nbk ? YW[(jb + jj) * MF_LDT + c] : 0.0;
#pragma unroll
        for (int ii = 1; ii < MF_NB; ++ii) {   // diagonal block (block-uniform guard: a short last block stops early)
            if (ii >= nbk) break;
            const double2* l2 = reinterpret_cast<const double2*>(Lb + (size_t)ii * MF_NB);
            double acc = yb[ii], acc2 = 0.0;
#pragma unroll
            for (int jj = 0; jj + 1 < ii; jj += 2) {
                const double2 l = l2[jj >> 1];
                acc = fma(-l.x, yb[jj], acc);
                acc2 = fma(-l.y, yb[jj + 1], acc2);
            }
            if (ii & 1) acc = fma(-Lb[ii * MF_NB + ii - 1], yb[ii - 1], acc);
            yb[ii] = acc + acc2;
        }
        if (q == 0 && live) {   // these rows of y are final
            double* yo = Y + (size_t)(fr.first + jb) * nrhs + col;
#pragma unroll
            for (int ii = 0; ii < MF_NB; ++ii)
                if (ii < nbk) yo[(size_t)ii * nrhs] = yb[ii];
        }
        for (int i = jb + nbk + q; i < nf; i += MF_RG) {
            const double2* l2 = reinterpret_cast<const double2*>(Lb + (size_t)(i - jb) * MF_NB);
            double acc = YW[i * MF_LDT + c], acc2 = 0.0;
#pragma unroll
            for (int jj = 0; jj < MF_NB; jj += 2) {
                const double2 l = l2[jj >> 1];
                acc = fma(-l.x, yb[jj], acc);
                acc2 = fma(-l.y, yb[jj + 1], acc2);
            }
            YW[i * MF_LDT + c] = acc + acc2;
        }
    }
    __syncthreads();
    if (live) {
        double* wout = W + (size_t)fr.w * nrhs + col;
        for (int t = q; t < s; t += MF_RG) wout[(size_t)t * nrhs] = YW[(k + t) * MF_LDT + c];
    }
}

__global__ void __launch_bounds__(MF_TT, MF_BT_MIN_BLOCKS) mf_backward_tiled_kernel(const int* list, const MfFront* fronts, const int* strct, const int* perm,
                                                                  const double* Lp, const double* Up, double* Y, double* X,
                                                                  const long long N, const int nrhs) {
    extern __shared__ __align__(16) double mf_smem[];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int k = fr.k, s = fr.s, nf = k + s;
    const int tid = threadIdx.x, c = tid & (MF_TC - 1), q = tid >> 6, lane = tid & 31, wid = tid >> 5;
    const int c0 = blockIdx.y * MF_TC, col = c0 + c;
    const int ncol = min(MF_TC, nrhs - c0);
    const bool live = col < nrhs;
    if (k == 0) return;                                    // assembly node: nothing to solve
    double* YW = mf_smem;                                  // rows 0..k-1: y -> x; rows k..nf-1: boundary solutions
    double* Ub = YW + (size_t)nf * MF_LDT;                 // [k][MF_NB]: rows of the current column block of [U11 U12]
    Ub += ((size_t)nf * MF_LDT) & 1;
    const double* L = Lp + fr.lp;
    const double* U12 = Up + fr.up;
    const int* sp = strct + fr.soff;
    // the whole tile in flight at once (asynchronous copies: no register staging); the first panel block rides along
    if (live) {
        for (int r = q; r < k; r += MF_RG) cp_async8(&YW[r * MF_LDT + c], &Y[(size_t)(fr.first + r) * nrhs + col]);
#pragma unroll 4
        for (int t = q; t < s; t += MF_RG) cp_async8(&YW[(k + t) * MF_LDT + c], &Y[(size_t)sp[t] * nrhs + col]);
    }
    // column blocks of [U11 U12] from the right: boundary blocks (plain updates), then the blocks of U11 (solve + update)
    const int nbb = (s + MF_NB - 1) / MF_NB, npb = (k + MF_NB - 1) / MF_NB;
    double ureg[MF_NB];
    auto block_col0 = [&](const int b) { return b < nbb ? k + b * MF_NB : (npb - 1 - (b - nbb)) * MF_NB; };
    auto prefetch = [&](const int b) {
        const int jb = block_col0(b);
        const int lim = jb >= k ? nf : k;          // last column of this kind
        const int rows_needed = jb >= k ? k : min(jb + MF_NB, k);
#pragma unroll
        for (int jj = 0; jj < MF_NB; ++jj) {
            const int j = jb + jj;
            double v = 0.0;
            if (tid < rows_needed && j < lim) v = j < k ? L[tid + (size_t)j * nf] : U12[tid + (size_t)(j - k) * k];
            ureg[jj] = v;
        }
    };
    double pend[MF_NB];
    int pend_jb = -1;
    const int nblocks = nbb + npb;
    prefetch(0);
    cp_async_wait_all();
    for (int b = 0; b < nblocks; ++b) {
        const int jb = block_col0(b);
        const bool pivot_block = jb < k;
        const int nbk = pivot_block ? min(MF_NB, k - jb) : min(MF_NB, nf - jb);
        __syncthreads();   // the previous block is applied: its solved rows may be published, Ub may be overwritten
        if (pend_jb >= 0 && q == 0) {
#pragma unroll
            for (int ii = 0; ii < MF_NB; ++ii)
                if (pend_jb + ii < k) YW[(pend_jb + ii) * MF_LDT + c] = pend[ii];
        }
        pend_jb = -1;
        if (tid < k) {
            double2* dst = reinterpret_cast<double2*>(Ub + (size_t)tid * MF_NB);
#pragma unroll
            for (int jj = 0; jj < MF_NB; jj += 2) dst[jj >> 1] = make_double2(ureg[jj], ureg[jj + 1]);
        }
        __syncthreads();
        if (b + 1 < nblocks) prefetch(b + 1);
        double xb[MF_NB];
#pragma unroll
        for (int jj = 0; jj < MF_NB; ++jj) xb[jj] = jj < nbk ? YW[(jb + jj) * MF_LDT + c] : 0.0;
        int top = k;   // rows [0, top) receive this block's update
        if (pivot_block) {
#pragma unroll
            for (int ii = MF_NB - 1; ii >= 0; --ii) {
                if (ii < nbk) {
                    const double* ur = Ub + (size_t)(jb + ii) * MF_NB;
                    double acc = xb[ii], acc2 = 0.0;
#pragma unroll
                    for (int jj = ii + 1; jj < MF_NB; ++jj) {   // columns beyond nbk are zero-padded
                        if ((jj - ii) & 1) acc = fma(-ur[jj], xb[jj], acc);
                        else acc2 = fma(-ur[jj], xb[jj], acc2);
                    }
                    xb[ii] = (acc + acc2) / ur[ii];
                }
            }
#pragma unroll
            for (int ii = 0; ii < MF_NB; ++ii) pend[ii] = xb[ii];
            pend_jb = jb;
            top = jb;
        }
        for (int i = q; i < top; i += MF_RG) {
            const double2* u2 = reinterpret_cast<const double2*>(Ub + (size_t)i * MF_NB);
            double acc = YW[i * MF_LDT + c], acc2 = 0.0;
#pragma unroll
            for (int jj = 0; jj < MF_NB; jj += 2) {
                const double2 u = u2[jj >> 1];
                acc = fma(-u.x, xb[jj], acc);
                acc2 = fma(-u.y, xb[jj + 1], acc2);
            }
            YW[i * MF_LDT + c] = acc + acc2;
        }
    }
    __syncthreads();
    if (pend_jb >= 0 && q == 0) {
#pragma unroll
        for (int ii = 0; ii < MF_NB; ++ii)
            if (pend_jb + ii < k) YW[(pend_jb + ii) * MF_LDT + c] = pend[ii];
    }
    __syncthreads();
    if (!fr.leaf && live)   // separator rows are read by the fronts below
        for (int r = q; r < k; r += MF_RG) Y[(size_t)(fr.first + r) * nrhs + col] = YW[r * MF_LDT + c];
    // solution rows back into the caller's column-major block (lanes: consecutive rows of one column)
    for (int cc = wid; cc < ncol; cc += MF_TT / 32)
        for (int r = lane; r < k; r += 32) X[(size_t)perm[fr.first + r] + (size_t)N * (c0 + cc)] = YW[r * MF_LDT + cc];
}

// ---------------------------------------------------------------------------------------------------------------
// Leaf fronts (tree level 0: no children, k <= KMAX) hold most rows of the matrix, so their sweeps carry the N x nrhs
// block through HBM.  One thread per right-hand side column with ITS k entries in registers (all loops unrolled to
// KMAX, panels zero-padded in shared memory and read as broadcast 16-byte loads), the row interchanges folded into
// the gather, no work area: forward reads the caller's b and writes y / the boundary update, backward reads y and the
// separator solutions and writes the caller's x.
constexpr int MF_KMAX = 32;
constexpr int MF_LLD = MF_KMAX + 2;   // row stride of the panels in shared memory: 16-byte aligned rows, transposing stores 4-way (not 32-way) conflicted
constexpr int MF_LEAF_TC = 128;

__global__ void __launch_bounds__(MF_LEAF_TC) mf_forward_leaf_kernel(const int* list, const MfFront* fronts, const int* perm,
                                                                     const int* piv, const int* psrc, const double* Lp, const double* B,
                                                                     double* Y, double* W, const long long N, const int nrhs) {
    extern __shared__ __align__(16) double mf_smem[];
    __shared__ int rows[MF_KMAX];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int k = fr.k, s = fr.s, nf = k + s;
    const int tid = threadIdx.x, col = blockIdx.y * MF_LEAF_TC + tid;
    constexpr int LDT = MF_KMAX + 1;       // tile leading dimension: conflict-free both ways
    double* Ts = mf_smem;                  // [column][row] tile of b (first), then the L panel (same storage)
    double* Ls = mf_smem;                  // row r of the L panel at Ls[r * KMAX .. ], columns >= k zero
    {   // the panel is read after the gather of b: on its way into L2 meanwhile
        const char* pb = reinterpret_cast<const char*>(Lp + fr.lp);
        const size_t bytes = (size_t)nf * k * sizeof(double);
        for (size_t off = (size_t)tid * 128; off < bytes; off += (size_t)MF_LEAF_TC * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pb + off));
    }
    if (psrc) {      // net effect of the row interchanges, precomputed per front (mf_netperm_kernel)
        if (tid < k) rows[tid] = perm[fr.first + psrc[fr.first + tid]];
    } else if (tid == 0) {  // ... or worked out here: position r of P b comes from row src[r]
        int src[MF_KMAX];
        for (int r = 0; r < k; ++r) src[r] = r;
        for (int j = 0; j < k; ++j) {
            const int p = piv[fr.first + j];
            const int t = src[j];
            src[j] = src[p];
            src[p] = t;
        }
        for (int r = 0; r < k; ++r) rows[r] = perm[fr.first + src[r]];
    }
    __syncthreads();
    // rows of this front from the caller's column-major block: consecutive threads take consecutive rows of one
    // column (the front's rows are sorted runs of the original numbering), transposed through shared memory
    const int c0 = blockIdx.y * MF_LEAF_TC, ncol = min(MF_LEAF_TC, nrhs - c0);
    {   // (k <= 32: lane = position, one warp per column, eight columns in flight per warp)
        const int lane = tid & 31, wid = tid >> 5;
        const size_t row = lane < k ? (size_t)rows[lane] : 0;
#pragma unroll 8
        for (int c = wid; c < ncol; c += MF_LEAF_TC / 32)
            if (lane < k) Ts[c * LDT + lane] = ld_b(B + row + (size_t)N * (c0 + c));
    }
    __syncthreads();
    double y[MF_KMAX];
#pragma unroll
    for (int r = 0; r < MF_KMAX; ++r) y[r] = (r < k && tid < ncol) ? Ts[tid * LDT + r] : 0.0;
    __syncthreads();
    {   // panel: global reads run down the columns (coalesced), rows of the transposed copy are MF_LLD apart
        const int lane = tid & 31, wid = tid >> 5;
#pragma unroll 4
        for (int c = wid; c < MF_KMAX; c += MF_LEAF_TC / 32)
            for (int r = lane; r < nf; r += 32)
                Ls[r * MF_LLD + c] = (c < k && (r >= k || c < r)) ? Lp[fr.lp + r + (size_t)c * nf] : 0.0;
    }
    __syncthreads();
    if (col >= nrhs) return;
#pragma unroll
    for (int i = 1; i < MF_KMAX; ++i) {  // unit-lower L11 (block-uniform guard: rows >= k belong to L21)
        if (i >= k) break;
        double acc = y[i], acc2 = 0.0;
        const double2* l2 = reinterpret_cast<const double2*>(Ls + i * MF_LLD);
#pragma unroll
        for (int j = 0; j + 1 < i; j += 2) {
            const double2 l = l2[j >> 1];
            acc = fma(-l.x, y[j], acc);
            acc2 = fma(-l.y, y[j + 1], acc2);
        }
        if (i & 1) acc = fma(-Ls[i * MF_LLD + i - 1], y[i - 1], acc);
        y[i] = acc + acc2;
    }
    double* yo = Y + (size_t)fr.first * nrhs + col;
#pragma unroll
    for (int r = 0; r < MF_KMAX; ++r)
        if (r < k) yo[(size_t)r * nrhs] = y[r];
    double* wo = W + (size_t)fr.w * nrhs + col;
    for (int t = 0; t < s; ++t) {  // boundary update  w = -L21 y
        const double2* l2 = reinterpret_cast<const double2*>(Ls + (k + t) * MF_LLD);
        double acc = 0.0, acc2 = 0.0;
#pragma unroll
        for (int j = 0; j < MF_KMAX; j += 2) {
            const double2 l = l2[j >> 1];
            acc = fma(-l.x, y[j], acc);
            acc2 = fma(-l.y, y[j + 1], acc2);
        }
        wo[(size_t)t * nrhs] = acc + acc2;
    }
}

__global__ void __launch_bounds__(MF_LEAF_TC) mf_backward_leaf_kernel(const int* list, const MfFront* fronts, const int* strct,
                                                                      const int* perm, const double* Lp, const double* Up,
                                                                      const double* Y, double* X, const long long N, const int nrhs) {
    extern __shared__ __align__(16) double mf_smem[];
    __shared__ int rows[MF_KMAX];
    __shared__ double rdiag[MF_KMAX];
    const int fid = list[blockIdx.x];
    const MfFront fr = fronts[fid];
    const int k = fr.k, s = fr.s, nf = k + s;
    const int tid = threadIdx.x, col = blockIdx.y * MF_LEAF_TC + tid;
    double* U11s = mf_smem;                      // row i at U11s[i * KMAX ..], strictly upper part, zero elsewhere
    double* U12s = U11s + MF_KMAX * MF_LLD;      // boundary column t at U12s[t * KMAX ..] (entries i < k)
#pragma unroll
    for (int i = tid; i < MF_KMAX * MF_KMAX; i += MF_LEAF_TC) {   // global reads run down the columns (coalesced)
        const int c = i / MF_KMAX, r = i % MF_KMAX;
        U11s[r * MF_LLD + c] = (r < k && c < k && c > r) ? Lp[fr.lp + r + (size_t)c * nf] : 0.0;
    }
#pragma unroll 4
    for (int i = tid; i < s * MF_KMAX; i += MF_LEAF_TC) {
        const int t = i / MF_KMAX, r = i % MF_KMAX;
        U12s[i] = r < k ? Up[fr.up + r + (size_t)t * k] : 0.0;
    }
    if (tid < MF_KMAX) {
        rdiag[tid] = tid < k ? 1.0 / Lp[fr.lp + tid + (size_t)tid * nf] : 0.0;
        if (tid < k) rows[tid] = perm[fr.first + tid];
    }
    int* sps = reinterpret_cast<int*>(U12s + (size_t)s * MF_KMAX);   // boundary positions (behind the panels)
    for (int t = tid; t < s; t += MF_LEAF_TC) sps[t] = strct[fr.soff + t];
    __syncthreads();
    double y[MF_KMAX];
    if (col < nrhs) {
    const double* yi = Y + (size_t)fr.first * nrhs + col;
#pragma unroll
    for (int r = 0; r < MF_KMAX; ++r) y[r] = r < k ? yi[(size_t)r * nrhs] : 0.0;
    double xn[4];   // boundary solutions of the next group of four, loaded under the updates of the current one
#pragma unroll
    for (int u4 = 0; u4 < 4; ++u4) xn[u4] = u4 < s ? Y[(size_t)sps[u4] * nrhs + col] : 0.0;
    for (int t0 = 0; t0 < s; t0 += 4) {  // y -= U12 x2
        double x2[4];
#pragma unroll
        for (int u4 = 0; u4 < 4; ++u4) x2[u4] = xn[u4];
#pragma unroll
        for (int u4 = 0; u4 < 4; ++u4) xn[u4] = t0 + 4 + u4 < s ? Y[(size_t)sps[t0 + 4 + u4] * nrhs + col] : 0.0;
#pragma unroll
        for (int u4 = 0; u4 < 4; ++u4) {
            if (t0 + u4 >= s) break;
            const double2* u2 = reinterpret_cast<const double2*>(U12s + (t0 + u4) * MF_KMAX);
#pragma unroll
            for (int i = 0; i < MF_KMAX; i += 2) {
                const double2 u = u2[i >> 1];
                y[i] = fma(-u.x, x2[u4], y[i]);
                y[i + 1] = fma(-u.y, x2[u4], y[i + 1]);
            }
        }
    }
#pragma unroll
    for (int i = MF_KMAX - 1; i >= 0; --i) {
        double acc = y[i], acc2 = 0.0;
        const double* ur = U11s + i * MF_LLD;
        if (!(i & 1)) acc = fma(-ur[i + 1], y[i + 1], acc);   // first entry right of the diagonal sits at an odd column
#pragma unroll
        for (int j = (i + 2) & ~1; j < MF_KMAX; j += 2) {
            const double2 u = *reinterpret_cast<const double2*>(ur + j);
            acc = fma(-u.x, y[j], acc);
            acc2 = fma(-u.y, y[j + 1], acc2);
        }
        y[i] = (acc + acc2) * rdiag[i];
    }
    }
    // solution rows back into the caller's column-major block through a shared-memory transpose (same access shape
    // as the gather of the forward sweep)
    constexpr int LDT = MF_KMAX + 1;
    double* Ts = mf_smem;
    __syncthreads();   // every thread is done with the panels
    if (col < nrhs) {
#pragma unroll
        for (int r = 0; r < MF_KMAX; ++r)
            if (r < k) Ts[tid * LDT + r] = y[r];
    }
    __syncthreads();
    const int c0 = blockIdx.y * MF_LEAF_TC, ncol = min(MF_LEAF_TC, nrhs - c0);
    {
        const int lane = tid & 31, wid = tid >> 5;
        const size_t row = lane < k ? (size_t)rows[lane] : 0;
#pragma unroll 8
        for (int c = wid; c < ncol; c += MF_LEAF_TC / 32)
            if (lane < k) st_x(X + row + (size_t)N * (c0 + c), Ts[c * LDT + lane]);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host analysis
struct Graph {
    int64_t N;
    std::vector<int64_t> ptr;
    std::vector<int32_t> adj;
};

struct Dissector {
    const Graph& g;
    int leaf_max;
    std::vector<int32_t> region;   // region id of every vertex while it is unassigned, -1 once it is ordered
    std::vector<int32_t> level;    // BFS scratch
    std::vector<std::vector<int32_t>> snodes;  // supernodes in elimination order
    int next_region = 1;
    std::vector<int32_t> queue;
    const std::vector<int32_t>* weight = nullptr;  // original vertices behind every (contracted) vertex; nullptr: 1 each

    Dissector(const Graph& gr, int leaf) : g(gr), leaf_max(leaf), region((size_t)gr.N, 0), level((size_t)gr.N, -1) {}
    int64_t wsum(const std::vector<int32_t>& vs) const {
        if (!weight) return (int64_t)vs.size();
        int64_t w = 0;
        for (int32_t v : vs) w += (*weight)[(size_t)v];
        return w;
    }

    // BFS inside region `rid` from `start`; fills queue (visit order) and level[]; returns the number of levels
    int bfs(int32_t start, int32_t rid) {
        queue.clear();
        queue.push_back(start);
        level[(size_t)start] = 0;
        int nl = 1;
        for (size_t head = 0; head < queue.size(); ++head) {
            const int32_t v = queue[head];
            for (int64_t e = g.ptr[(size_t)v]; e < g.ptr[(size_t)v + 1]; ++e) {
                const int32_t w = g.adj[(size_t)e];
                if (region[(size_t)w] == rid && level[(size_t)w] < 0) {
                    level[(size_t)w] = level[(size_t)v] + 1;
                    nl = level[(size_t)w] + 1;
                    queue.push_back(w);
                }
            }
        }
        return nl;
    }
    void clear_levels() {
        for (int32_t v : queue) level[(size_t)v] = -1;
    }
    void emit(std::vector<int32_t>& verts) {
        std::sort(verts.begin(), verts.end());
        for (int32_t v : verts) region[(size_t)v] = -1;
        snodes.push_back(verts);
    }

    // Separators of `group_levels` consecutive dissection levels are collected into ONE front (relaxed amalgamation of
    // the small separator fronts: a tree level costs a kernel launch per sweep, the extra fill is a few dense blocks of
    // separator size).  `sink`: the collecting front of the enclosing group (nullptr: the next cut opens a new group),
    // `remaining`: dissection levels the enclosing group still absorbs.
    int group_levels = 2;

    // orders all vertices of `verts` (all carrying region id rid)
    void dissect(std::vector<int32_t>& verts, int32_t rid, std::vector<int32_t>* sink = nullptr, int remaining = 0) {
        // connected components
        std::vector<std::vector<int32_t>> comps;
        for (int32_t v0 : verts) {
            if (level[(size_t)v0] >= 0 || region[(size_t)v0] != rid) continue;
            bfs(v0, rid);
            comps.emplace_back(queue);
            for (int32_t v : queue) level[(size_t)v] = 1 << 30;  // keep them marked until all components are found
        }
        for (int32_t v : verts) level[(size_t)v] = -1;
        std::vector<int32_t> bin;
        int64_t binw = 0;
        for (auto& comp : comps) {
            const int64_t cw = wsum(comp);
            if (cw <= leaf_max) {  // small component: pack with its small siblings into one leaf front
                if (!bin.empty() && binw + cw > leaf_max) {
                    emit(bin);
                    bin.clear();
                    binw = 0;
                }
                bin.insert(bin.end(), comp.begin(), comp.end());
                binw += cw;
                continue;
            }
            const int32_t cid = next_region++;
            for (int32_t v : comp) region[(size_t)v] = cid;
            split(comp, cid, sink, remaining);
        }
        if (!bin.empty()) emit(bin);
    }

    // connected region larger than a leaf: level-structure bisection
    void split(std::vector<int32_t>& comp, int32_t rid, std::vector<int32_t>* sink, int remaining) {
        // pseudo-peripheral start: repeat BFS from a vertex of the last level
        int32_t start = comp[0];
        int nl = 0;
        for (int it = 0; it < 3; ++it) {
            nl = bfs(start, rid);
            int32_t last = queue.back();
            // smallest degree in the last level
            int64_t bestdeg = INT64_MAX;
            for (size_t i = queue.size(); i-- > 0 && level[(size_t)queue[i]] == nl - 1;) {
                const int64_t d = g.ptr[(size_t)queue[i] + 1] - g.ptr[(size_t)queue[i]];
                if (d < bestdeg) { bestdeg = d; last = queue[i]; }
            }
            if (it == 2) break;
            clear_levels();
            start = last;
        }
        if (nl < 3) {  // no interior level to cut at (clique-like): one dense front
            clear_levels();
            emit(comp);
            return;
        }
        std::vector<int64_t> cnt((size_t)nl, 0);
        for (int32_t v : queue) ++cnt[(size_t)level[(size_t)v]];
        const int64_t total = (int64_t)queue.size();
        int64_t before = cnt[0];
        int best = -1;
        double bestscore = 1e300;
        for (int l = 1; l + 1 < nl; ++l) {
            const double frac = (double)before / (double)total;
            const double imbalance = fabs(frac + 0.5 * (double)cnt[(size_t)l] / (double)total - 0.5);
            // small separators near the middle: size, penalised away from the centre
            const double score = (double)cnt[(size_t)l] * (1.0 + 8.0 * imbalance * imbalance * 4.0) + (imbalance > 0.3 ? 1e9 * imbalance : 0.0);
            if (score < bestscore) { bestscore = score; best = l; }
            before += cnt[(size_t)l];
        }
        // thin the separator: a vertex of level `best` without a neighbour in level best + 1 joins the near side
        std::vector<int32_t> sep, lo, hi;
        for (int32_t v : queue) {
            const int lv = level[(size_t)v];
            if (lv < best) lo.push_back(v);
            else if (lv > best) hi.push_back(v);
            else {
                bool touches = false;
                for (int64_t e = g.ptr[(size_t)v]; e < g.ptr[(size_t)v + 1] && !touches; ++e) {
                    const int32_t w = g.adj[(size_t)e];
                    touches = region[(size_t)w] == rid && level[(size_t)w] == best + 1;
                }
                (touches ? sep : lo).push_back(v);
            }
        }
        clear_levels();
        const int32_t rlo = next_region++, rhi = next_region++, rsep = next_region++;
        for (int32_t v : lo) region[(size_t)v] = rlo;
        for (int32_t v : hi) region[(size_t)v] = rhi;
        for (int32_t v : sep) region[(size_t)v] = rsep;
        if (sink && remaining > 0) {  // inside a group: the separator joins the group's front
            for (int32_t v : sep) region[(size_t)v] = -1;
            sink->insert(sink->end(), sep.begin(), sep.end());
            dissect(lo, rlo, sink, remaining - 1);
            dissect(hi, rhi, sink, remaining - 1);
            return;
        }
        std::vector<int32_t> group;   // this cut opens a group: its separator + those of the next group_levels - 1 levels
        for (int32_t v : sep) region[(size_t)v] = -1;
        dissect(lo, rlo, &group, group_levels - 1);
        dissect(hi, rhi, &group, group_levels - 1);
        group.insert(group.end(), sep.begin(), sep.end());
        emit(group);
    }
};

struct MfLaunch {
    int level, big, offset, count, max_nf, max_k, max_s, max_u;
};

struct MfHost {
    std::vector<MfFront> fronts;
    std::vector<int32_t> perm;       // permuted position -> original index
    std::vector<int32_t> strct, rel, child_idx, aloc, asrc, lists, uptr, usrc;
    std::vector<MfLaunch> launches;  // factorisation order (levels ascending)
    int nlevels = 0;
    long long lp_total = 0, up_total = 0, cb_total = 0, w_rows = 0, big_scratch = 0;
    std::vector<long long> big_off;  // per big launch entry
    double flops = 0.0;
    long long nnz_lu = 0;
    int max_front = 0;
    int nreal = 0;                   // fronts [0, nreal) eliminate supernodes; the others are assembly nodes (k = 0)
};

// symbolic factorisation on a given supernode partition (snodes in elimination order)
bool mf_symbolic(const Graph& g, const std::vector<std::vector<int32_t>>& snodes, int64_t N, const int64_t* colptr, const int64_t* rowval,
                 int trans, MfHost& H, std::string& err) {
    const int S = (int)snodes.size();
    H = MfHost();
    H.perm.resize((size_t)N);
    std::vector<int32_t> pos((size_t)N), sn_of_pos((size_t)N);
    std::vector<int32_t> first((size_t)S + 1, 0);
    {
        int32_t q = 0;
        for (int s = 0; s < S; ++s) {
            first[(size_t)s] = q;
            for (int32_t v : snodes[(size_t)s]) {
                H.perm[(size_t)q] = v;
                pos[(size_t)v] = q;
                sn_of_pos[(size_t)q] = s;
                ++q;
            }
        }
        first[(size_t)S] = q;
        if (q != N) {
            err = "sparse_setup: internal error (ordering does not cover all vertices)";
            return false;
        }
    }
    H.fronts.resize((size_t)S);
    std::vector<std::vector<int32_t>> children((size_t)S);
    std::vector<int32_t> stamp((size_t)N, -1);
    std::vector<int32_t> soff((size_t)S + 1, 0);
    std::vector<int32_t> tmp;
    std::vector<int> lvl((size_t)S, 0);
    for (int s = 0; s < S; ++s) {
        tmp.clear();
        const int32_t end = first[(size_t)s + 1];
        for (int32_t v : snodes[(size_t)s])
            for (int64_t e = g.ptr[(size_t)v]; e < g.ptr[(size_t)v + 1]; ++e) {
                const int32_t q = pos[(size_t)g.adj[(size_t)e]];
                if (q >= end && stamp[(size_t)q] != s) {
                    stamp[(size_t)q] = s;
                    tmp.push_back(q);
                }
            }
        for (int32_t c : children[(size_t)s]) {
            const MfFront& ch = H.fronts[(size_t)c];
            for (int t = 0; t < ch.s; ++t) {
                const int32_t q = H.strct[(size_t)ch.soff + t];
                if (q >= end && stamp[(size_t)q] != s) {
                    stamp[(size_t)q] = s;
                    tmp.push_back(q);
                }
            }
            lvl[(size_t)s] = std::max(lvl[(size_t)s], lvl[(size_t)c] + 1);
        }
        std::sort(tmp.begin(), tmp.end());
        MfFront& f = H.fronts[(size_t)s];
        f.k = (int)snodes[(size_t)s].size();
        f.s = (int)tmp.size();
        f.first = first[(size_t)s];
        f.soff = (int)H.strct.size();
        f.leaf = children[(size_t)s].empty() ? 1 : 0;
        f.parent = tmp.empty() ? -1 : sn_of_pos[(size_t)tmp[0]];
        H.strct.insert(H.strct.end(), tmp.begin(), tmp.end());
        if (f.parent >= 0) children[(size_t)f.parent].push_back(s);
        if (H.strct.size() > (size_t)1 << 30) {
            err = "sparse_setup: factor structure too large";
            return false;
        }
    }
    // Assembly nodes.  A front with very many children (the top front of an arrowhead: thousands of leaves under the
    // dense rows) would add their contribution blocks / boundary updates one after the other on ONE CTA.  Its children
    // are regrouped under intermediate fronts without pivots (k = 0, boundary = all rows of the parent, identity
    // relative indices): they only sum their group, in parallel with each other, and hand ONE block each to the parent
    // (repeated while a front keeps more than MF_MANY children: a tree reduction in a fixed order -- deterministic).
    H.nreal = S;
    {
        constexpr size_t MF_MANY = 32;
        constexpr long long NODE_BUDGET = (long long)1 << 27;   // doubles of extra contribution-block storage (1 GiB)
        for (int s = 0; s < H.nreal; ++s) {
            while (children[(size_t)s].size() > MF_MANY && !getenv("DIFFOPT_B200_MF_NO_ASSEMBLY_NODES")) {
                const std::vector<int32_t> ch = children[(size_t)s];
                const MfFront p = H.fronts[(size_t)s];
                const long long nfp = p.k + p.s;
                size_t fan = 24;
                while ((long long)((ch.size() + fan - 1) / fan) * nfp * nfp > NODE_BUDGET) fan *= 2;
                if (fan >= ch.size()) break;
                std::vector<int32_t> groups;
                for (size_t i0 = 0; i0 < ch.size(); i0 += fan) {
                    MfFront a{};
                    a.k = 0;
                    a.s = (int)nfp;
                    a.first = p.first;
                    a.soff = (int)H.strct.size();
                    a.leaf = 0;
                    a.parent = s;
                    for (int r = 0; r < p.k; ++r) H.strct.push_back(p.first + r);
                    for (int t = 0; t < p.s; ++t) H.strct.push_back(H.strct[(size_t)p.soff + t]);
                    const int32_t id = (int32_t)H.fronts.size();
                    std::vector<int32_t> grp(ch.begin() + (long)i0, ch.begin() + (long)std::min(ch.size(), i0 + fan));
                    for (int32_t c : grp) H.fronts[(size_t)c].parent = id;
                    H.fronts.push_back(a);
                    children.push_back(std::move(grp));
                    groups.push_back(id);
                }
                children[(size_t)s] = groups;
            }
        }
    }
    const int S_all = (int)H.fronts.size();
    if (S_all != S) {   // tree levels again (the nodes sit between their group and the parent)
        lvl.assign((size_t)S_all, -1);
        std::vector<int32_t> stack;
        for (int r = 0; r < S_all; ++r) {
            if (lvl[(size_t)r] >= 0) continue;
            stack.push_back(r);
            while (!stack.empty()) {
                const int32_t f = stack.back();
                int l = 0;
                bool ready = true;
                for (int32_t c : children[(size_t)f]) {
                    if (lvl[(size_t)c] < 0) {
                        stack.push_back(c);
                        ready = false;
                    } else l = std::max(l, lvl[(size_t)c] + 1);
                }
                if (ready) {
                    lvl[(size_t)f] = l;
                    stack.pop_back();
                }
            }
        }
    }
    // relative indices into the parent, children lists, storage offsets
    H.rel.assign(H.strct.size(), 0);
    for (int s = 0; s < S_all; ++s) {
        MfFront& f = H.fronts[(size_t)s];
        f.c0 = (int)H.child_idx.size();
        for (int32_t c : children[(size_t)s]) H.child_idx.push_back(c);
        f.c1 = (int)H.child_idx.size();
        if (f.parent >= 0) {
            const MfFront& p = H.fronts[(size_t)f.parent];
            const int32_t pend = p.first + p.k;
            int t2 = 0;
            for (int t = 0; t < f.s; ++t) {
                const int32_t q = H.strct[(size_t)f.soff + t];
                if (q < pend) H.rel[(size_t)f.soff + t] = q - p.first;
                else {
                    while (t2 < p.s && H.strct[(size_t)p.soff + t2] < q) ++t2;
                    if (t2 >= p.s || H.strct[(size_t)p.soff + t2] != q) {
                        err = "sparse_setup: internal error (child structure not contained in the parent front)";
                        return false;
                    }
                    H.rel[(size_t)f.soff + t] = p.k + t2;
                }
            }
        }
        const long long nf = f.k + f.s;
        f.lp = H.lp_total; H.lp_total += nf * f.k;
        f.up = H.up_total; H.up_total += (long long)f.k * f.s;
        f.cb = H.cb_total; H.cb_total += (long long)f.s * f.s;
        f.w = H.w_rows; H.w_rows += f.s;
        H.nnz_lu += nf * f.k + (long long)f.k * f.s;
        const double k = f.k, s2 = f.s;
        H.flops += 2.0 / 3.0 * k * k * k + 2.0 * k * k * s2 + 2.0 * k * s2 * s2;
        H.max_front = std::max(H.max_front, (int)nf);
        if (nf * nf > ((long long)1 << 31) - 1) {
            err = "sparse_setup: a front is too large";
            return false;
        }
    }
    // matrix entries -> (front, local offset).  Entry (i, j) lives in the front that eliminates min(pos i, pos j).
    {
        std::vector<int32_t> cnt((size_t)S_all + 1, 0);
        const int64_t nnz = colptr[N] - 1;
        std::vector<int32_t> ef((size_t)nnz), el((size_t)nnz);
        for (int64_t c = 0; c < N; ++c)
            for (int64_t e = colptr[c] - 1; e < colptr[c + 1] - 1; ++e) {
                int64_t r = rowval[e] - 1, cc = c;
                if (trans) std::swap(r, cc);
                const int32_t pr = pos[(size_t)r], pc = pos[(size_t)cc];
                const int s = sn_of_pos[(size_t)std::min(pr, pc)];
                const MfFront& f = H.fronts[(size_t)s];
                auto loc = [&](int32_t q) -> int {
                    if (q < f.first + f.k) return q - f.first;
                    const int32_t* b = H.strct.data() + f.soff;
                    const int32_t* it = std::lower_bound(b, b + f.s, q);
                    return f.k + (int)(it - b);
                };
                const int nf = f.k + f.s;
                ef[(size_t)e] = s;
                el[(size_t)e] = loc(pr) + loc(pc) * nf;
                ++cnt[(size_t)s + 1];
            }
        for (int s = 0; s < S_all; ++s) cnt[(size_t)s + 1] += cnt[(size_t)s];
        H.aloc.resize((size_t)nnz);
        H.asrc.resize((size_t)nnz);
        std::vector<int32_t> fill(cnt.begin(), cnt.end() - 1);
        for (int64_t e = 0; e < nnz; ++e) {
            const int32_t d = fill[(size_t)ef[(size_t)e]]++;
            H.aloc[(size_t)d] = el[(size_t)e];
            H.asrc[(size_t)d] = (int32_t)e;
        }
        for (int s = 0; s < S_all; ++s) {
            H.fronts[(size_t)s].a0 = cnt[(size_t)s];
            H.fronts[(size_t)s].a1 = cnt[(size_t)s + 1];
        }
    }
    // forward-sweep update lists: for every row of a front (numbering before the interchanges), the workspace rows of its
    // children that land on it, children in list order (the order the sums are formed in).  uptr holds absolute offsets
    // into usrc.
    if (H.w_rows >= ((long long)1 << 31) - 1) {
        err = "sparse_setup: factor structure too large";
        return false;
    }
    {
        std::vector<int32_t> cnt;
        for (int s = 0; s < S_all; ++s) {
            MfFront& f = H.fronts[(size_t)s];
            const int nf = f.k + f.s;
            f.u0 = (int)H.uptr.size();
            cnt.assign((size_t)nf + 1, 0);
            for (int ci = f.c0; ci < f.c1; ++ci) {
                const MfFront& ch = H.fronts[(size_t)H.child_idx[(size_t)ci]];
                for (int t = 0; t < ch.s; ++t) ++cnt[(size_t)H.rel[(size_t)ch.soff + t] + 1];
            }
            for (int r = 0; r < nf; ++r) cnt[(size_t)r + 1] += cnt[(size_t)r];
            f.un = cnt[(size_t)nf];
            const int32_t base = (int32_t)H.usrc.size();
            for (int r = 0; r <= nf; ++r) H.uptr.push_back(base + cnt[(size_t)r]);
            H.usrc.resize((size_t)base + (size_t)f.un);
            for (int ci = f.c0; ci < f.c1; ++ci) {
                const MfFront& ch = H.fronts[(size_t)H.child_idx[(size_t)ci]];
                for (int t = 0; t < ch.s; ++t) H.usrc[(size_t)base + (size_t)cnt[(size_t)H.rel[(size_t)ch.soff + t]]++] = (int32_t)(ch.w + t);
            }
        }
    }
    // launch groups: per tree level, fronts that fit shared memory (sorted by size) and the others
    H.nlevels = 0;
    for (int s = 0; s < S_all; ++s) H.nlevels = std::max(H.nlevels, lvl[(size_t)s] + 1);
    std::vector<std::vector<int32_t>> bylevel((size_t)H.nlevels);
    for (int s = 0; s < S_all; ++s) bylevel[(size_t)lvl[(size_t)s]].push_back(s);
    for (int l = 0; l < H.nlevels; ++l) {
        auto& v = bylevel[(size_t)l];
        std::stable_sort(v.begin(), v.end(), [&](int32_t a, int32_t b) {
            return H.fronts[(size_t)a].k + H.fronts[(size_t)a].s > H.fronts[(size_t)b].k + H.fronts[(size_t)b].s;
        });
        // size classes so that one huge front does not size the shared memory of thousands of small ones
        size_t i = 0;
        while (i < v.size()) {
            const MfFront& f0 = H.fronts[(size_t)v[i]];
            const int nf0 = f0.k + f0.s;
            const bool big = (size_t)nf0 * (nf0 | 1) * 8 + (size_t)f0.k * 8 > MF_SMEM_CAP;
            MfLaunch L{l, big ? 1 : 0, (int)H.lists.size(), 0, 0, 0, 0, 0};
            size_t j = i;
            for (; j < v.size(); ++j) {
                const MfFront& f = H.fronts[(size_t)v[j]];
                const int nf = f.k + f.s;
                const bool b2 = (size_t)nf * (nf | 1) * 8 + (size_t)f.k * 8 > MF_SMEM_CAP;
                if (b2 != big) break;
                if (!big && j > i && nf * 2 < nf0 && nf0 > 24) break;  // next size class
                H.lists.push_back(v[j]);
                L.max_nf = std::max(L.max_nf, nf);
                L.max_k = std::max(L.max_k, f.k);
                L.max_s = std::max(L.max_s, f.s);
                L.max_u = std::max(L.max_u, f.un);
                if (big) {
                    H.big_off.push_back(H.big_scratch);
                    H.big_scratch += (long long)nf * (nf | 1) + f.k;
                }
            }
            L.count = (int)(j - i);
            // within a size class the fronts run in the order of their rows in the caller's numbering: neighbouring fronts
            // share the sectors at the ends of their row runs (gathers of b, scatters of x), which then meet in L2
            if (!big)
                std::sort(H.lists.begin() + L.offset, H.lists.begin() + L.offset + L.count, [&](int32_t a, int32_t b) {
                    const int32_t ra = H.perm[(size_t)H.fronts[(size_t)a].first], rb = H.perm[(size_t)H.fronts[(size_t)b].first];
                    return ra != rb ? ra < rb : a < b;
                });
            H.launches.push_back(L);
            i = j;
        }
    }
    return true;
}

// symmetrised pattern + ordering (dense vertices last, nested dissection on the rest) -> supernodes in elimination order
bool mf_order(int64_t N, const int64_t* colptr, const int64_t* rowval, const double* nzval, Graph& g,
              std::vector<std::vector<int32_t>>& snodes, std::string& err) {
    // symmetrised pattern without the diagonal, duplicates removed
    g.N = N;
    g.ptr.assign((size_t)N + 1, 0);
    for (int64_t c = 0; c < N; ++c)
        for (int64_t e = colptr[c] - 1; e < colptr[c + 1] - 1; ++e) {
            const int64_t r = rowval[e] - 1;
            if (r < 0 || r >= N) {
                err = "sparse_setup: row index out of range";
                return false;
            }
            if (r != c) {
                ++g.ptr[(size_t)r + 1];
                ++g.ptr[(size_t)c + 1];
            }
        }
    for (int64_t i = 0; i < N; ++i) g.ptr[(size_t)i + 1] += g.ptr[(size_t)i];
    g.adj.resize((size_t)g.ptr[(size_t)N]);
    {
        std::vector<int64_t> fill(g.ptr.begin(), g.ptr.end() - 1);
        for (int64_t c = 0; c < N; ++c)
            for (int64_t e = colptr[c] - 1; e < colptr[c + 1] - 1; ++e) {
                const int64_t r = rowval[e] - 1;
                if (r != c) {
                    g.adj[(size_t)fill[(size_t)r]++] = (int32_t)c;
                    g.adj[(size_t)fill[(size_t)c]++] = (int32_t)r;
                }
            }
        // sort + unique per vertex, compacting in place
        int64_t w = 0;
        std::vector<int64_t> nptr((size_t)N + 1, 0);
        for (int64_t v = 0; v < N; ++v) {
            int32_t* b = g.adj.data() + g.ptr[(size_t)v];
            int32_t* e = g.adj.data() + g.ptr[(size_t)v + 1];
            std::sort(b, e);
            e = std::unique(b, e);
            nptr[(size_t)v] = w;
            for (int32_t* p = b; p < e; ++p) g.adj[(size_t)w++] = *p;
        }
        nptr[(size_t)N] = w;
        g.ptr.swap(nptr);
        g.adj.resize((size_t)w);
    }
    // Weak diagonals (KKT matrices: the multiplier rows) cannot be pivoted inside a front unless a partner row sits in
    // the same front.  Symmetric matching: every vertex whose diagonal is (numerically) zero is paired with the
    // unmatched neighbour u that maximises |a_uv a_vu|; pairs are contracted to one vertex for the ordering, so the
    // dissection never separates them (the compressed-graph ordering of symmetric indefinite solvers).
    std::vector<int32_t> mate((size_t)N, -1);
    if (nzval) {
        std::vector<double> dmag((size_t)N, 0.0), omax((size_t)N, 0.0);
        for (int64_t c = 0; c < N; ++c)
            for (int64_t e = colptr[c] - 1; e < colptr[c + 1] - 1; ++e) {
                const int64_t r = rowval[e] - 1;
                const double a = fabs(nzval[e]);
                if (r == c) dmag[(size_t)c] += a;
                else {
                    omax[(size_t)c] = std::max(omax[(size_t)c], a);
                    omax[(size_t)r] = std::max(omax[(size_t)r], a);
                }
            }
        auto entry = [&](int64_t r, int64_t c) -> double {  // |a_rc| (rows of a column are sorted in Julia's CSC; else linear scan)
            const int64_t* b = rowval + (colptr[c] - 1);
            const int64_t* e = rowval + (colptr[c + 1] - 1);
            const int64_t* it = std::lower_bound(b, e, r + 1);
            if (it != e && *it == r + 1) return fabs(nzval[it - rowval]);
            for (it = b; it != e; ++it)
                if (*it == r + 1) return fabs(nzval[it - rowval]);
            return 0.0;
        };
        std::vector<int32_t> weak;
        for (int64_t v = 0; v < N; ++v)
            if (omax[(size_t)v] > 0.0 && dmag[(size_t)v] <= 1e-8 * omax[(size_t)v]) weak.push_back((int32_t)v);
        std::stable_sort(weak.begin(), weak.end(), [&](int32_t a, int32_t b) {
            return g.ptr[(size_t)a + 1] - g.ptr[(size_t)a] < g.ptr[(size_t)b + 1] - g.ptr[(size_t)b];
        });
        for (int32_t v : weak) {
            if (mate[(size_t)v] >= 0) continue;
            double best = 0.0;
            int32_t bu = -1;
            for (int64_t e = g.ptr[(size_t)v]; e < g.ptr[(size_t)v + 1]; ++e) {
                const int32_t u = g.adj[(size_t)e];
                if (mate[(size_t)u] >= 0) continue;
                const double w = entry(u, v) * entry(v, u);
                if (w > best) {
                    best = w;
                    bu = u;
                }
            }
            if (bu >= 0) {
                mate[(size_t)v] = bu;
                mate[(size_t)bu] = v;
            }
        }
    }
    // contracted graph
    std::vector<int32_t> cmap((size_t)N, -1), cw;
    std::vector<std::vector<int32_t>> members;
    for (int64_t v = 0; v < N; ++v) {
        if (cmap[(size_t)v] >= 0) continue;
        const int32_t id = (int32_t)members.size();
        cmap[(size_t)v] = id;
        members.push_back({(int32_t)v});
        const int32_t u = mate[(size_t)v];
        if (u >= 0) {
            cmap[(size_t)u] = id;
            members.back().push_back(u);
        }
        cw.push_back((int32_t)members.back().size());
    }
    Graph gc;
    gc.N = (int64_t)members.size();
    gc.ptr.assign((size_t)gc.N + 1, 0);
    {
        std::vector<int32_t> tmp;
        for (int64_t c = 0; c < gc.N; ++c) {
            tmp.clear();
            for (int32_t v : members[(size_t)c])
                for (int64_t e = g.ptr[(size_t)v]; e < g.ptr[(size_t)v + 1]; ++e) {
                    const int32_t d = cmap[(size_t)g.adj[(size_t)e]];
                    if (d != c) tmp.push_back(d);
                }
            std::sort(tmp.begin(), tmp.end());
            tmp.erase(std::unique(tmp.begin(), tmp.end()), tmp.end());
            gc.adj.insert(gc.adj.end(), tmp.begin(), tmp.end());
            gc.ptr[(size_t)c + 1] = (int64_t)gc.adj.size();
        }
    }
    // ordering: dense vertices last, nested dissection on the rest
    int leaf = 32;
    if (const char* lf = getenv("DIFFOPT_B200_MF_LEAF")) leaf = std::max(1, atoi(lf));
    {
        Dissector D(gc, leaf);
        D.weight = &cw;
        if (const char* gl = getenv("DIFFOPT_B200_MF_GROUP")) D.group_levels = std::max(1, atoi(gl));
        const double dense_deg = std::max(40.0, 10.0 * std::sqrt((double)N));
        std::vector<int32_t> dense, rest;
        for (int64_t c = 0; c < gc.N; ++c) {
            if ((double)(gc.ptr[(size_t)c + 1] - gc.ptr[(size_t)c]) > dense_deg) {
                dense.push_back((int32_t)c);
                D.region[(size_t)c] = -1;
            } else rest.push_back((int32_t)c);
        }
        D.dissect(rest, 0);
        if (!dense.empty()) D.emit(dense);
        snodes.clear();
        snodes.reserve(D.snodes.size());
        for (auto& sn : D.snodes) {
            std::vector<int32_t> verts;
            for (int32_t c : sn) verts.insert(verts.end(), members[(size_t)c].begin(), members[(size_t)c].end());
            std::sort(verts.begin(), verts.end());
            snodes.push_back(std::move(verts));
        }
    }
    return true;
}

}  // namespace

struct SparseMfImpl {
    MfHost H;
    std::vector<std::vector<int32_t>> snodes;
    Graph g;
    DevBuf fronts, perm, strct, rel, child_idx, aloc, asrc, lists, big_off, big_scratch, vals, Lp, Up, CB, piv, status, Y, W, psrc, pdst, uptr, usrc;
    int retries = 0;
    bool netperm = false;
    double analysis_ms = 0.0;
    void release() {
        for (DevBuf* b : {&fronts, &perm, &strct, &rel, &child_idx, &aloc, &asrc, &lists, &big_off, &big_scratch, &vals, &Lp, &Up, &CB, &piv,
                          &status, &Y, &W, &psrc, &pdst, &uptr, &usrc})
            b->release();
    }
};

void sparse_mf_release(diffopt_b200_ctx* ctx) {
    if (ctx->sparse_mf) {
        ctx->sparse_mf->release();
        delete ctx->sparse_mf;
        ctx->sparse_mf = nullptr;
    }
}

namespace {

template <class T>
cudaError_t upload(diffopt_b200_ctx* ctx, DevBuf& b, const std::vector<T>& v) {
    cudaError_t e = b.reserve(std::max<size_t>(v.size() * sizeof(T), 16));
    if (e != cudaSuccess || v.empty()) return e;
    return cudaMemcpyAsync(b.ptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream);
}

// uploads the symbolic structure and runs the numeric factorisation; returns 0, >0 singular, -5 delayed pivots needed
// (failed_out lists those fronts), <0 error
int32_t mf_numeric(diffopt_b200_ctx* ctx, SparseMfImpl& M, int64_t nnz, std::vector<int32_t>& failed_out) {
    MfHost& H = M.H;
    DO_CUDA(ctx, upload(ctx, M.fronts, H.fronts));
    DO_CUDA(ctx, upload(ctx, M.perm, H.perm));
    DO_CUDA(ctx, upload(ctx, M.strct, H.strct));
    DO_CUDA(ctx, upload(ctx, M.rel, H.rel));
    DO_CUDA(ctx, upload(ctx, M.child_idx, H.child_idx));
    DO_CUDA(ctx, upload(ctx, M.uptr, H.uptr));
    DO_CUDA(ctx, upload(ctx, M.usrc, H.usrc));
    DO_CUDA(ctx, upload(ctx, M.aloc, H.aloc));
    DO_CUDA(ctx, upload(ctx, M.asrc, H.asrc));
    DO_CUDA(ctx, upload(ctx, M.lists, H.lists));
    DO_CUDA(ctx, upload(ctx, M.big_off, H.big_off));
    DO_CUDA(ctx, M.big_scratch.reserve(std::max<size_t>((size_t)H.big_scratch * 8, 16)));
    DO_CUDA(ctx, M.Lp.reserve(std::max<size_t>((size_t)H.lp_total * 8, 16)));
    DO_CUDA(ctx, M.Up.reserve(std::max<size_t>((size_t)H.up_total * 8, 16)));
    DO_CUDA(ctx, M.CB.reserve(std::max<size_t>((size_t)H.cb_total * 8, 16)));
    DO_CUDA(ctx, M.piv.reserve(sizeof(int) * H.perm.size()));
    DO_CUDA(ctx, M.status.reserve(sizeof(int) * H.fronts.size()));
    (void)nnz;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int big_seen = 0;
    for (const MfLaunch& L : H.launches) {
        if (L.count == 0) continue;
        if (!L.big) {
            const size_t smem = ((size_t)L.max_nf * (L.max_nf | 1) + (size_t)L.max_k) * sizeof(double);
            auto launch = [&](auto kernel, const int threads) -> cudaError_t {
                cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024));
                if (e != cudaSuccess) return e;
                kernel<<<(unsigned)L.count, threads, smem, ctx->stream>>>(
                    M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(), M.child_idx.as<int>(), M.rel.as<int>(), M.aloc.as<int>(),
                    M.asrc.as<int>(), M.vals.as<double>(), M.Lp.as<double>(), M.Up.as<double>(), M.CB.as<double>(), M.piv.as<int>(),
                    M.status.as<int>());
                return cudaSuccess;
            };
            if (smem > 100 * 1024) DO_CUDA(ctx, launch(mf_factor_kernel<1024>, 1024));
            else if (smem > 50 * 1024) DO_CUDA(ctx, launch(mf_factor_kernel<512>, 512));
            else DO_CUDA(ctx, launch(mf_factor_kernel<MF_FACT_THREADS>, MF_FACT_THREADS));
        } else {
            mf_factor_big_kernel<<<(unsigned)L.count, MF_BIG_THREADS, 0, ctx->stream>>>(
                M.lists.as<int>() + L.offset, M.big_off.as<long long>() + big_seen, M.big_scratch.as<double>(), M.fronts.as<MfFront>(),
                M.child_idx.as<int>(), M.rel.as<int>(), M.aloc.as<int>(), M.asrc.as<int>(), M.vals.as<double>(), M.Lp.as<double>(),
                M.Up.as<double>(), M.CB.as<double>(), M.piv.as<int>(), M.status.as<int>());
            big_seen += L.count;
        }
        ctx->launches++;
        DO_CUDA(ctx, cudaGetLastError());
    }
    {   // net row permutation of every front (used by the tiled solve kernels)
        DO_CUDA(ctx, M.psrc.reserve(sizeof(int) * H.perm.size()));
        DO_CUDA(ctx, M.pdst.reserve(sizeof(int) * H.perm.size()));
        int maxk = 1;
        for (const MfFront& f : H.fronts) maxk = std::max(maxk, f.k);
        const size_t smem = sizeof(int) * 2 * (size_t)maxk;
        if (smem <= MF_SMEM_CAP) {
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_netperm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
            const int nfr = (int)H.fronts.size();
            mf_netperm_kernel<<<(unsigned)std::min(nfr, ctx->sm_count * 32), 64, smem, ctx->stream>>>(M.fronts.as<MfFront>(), nfr, M.piv.as<int>(),
                                                                                                      M.psrc.as<int>(), M.pdst.as<int>());
            ctx->launches++;
            DO_CUDA(ctx, cudaGetLastError());
            M.netperm = true;
        } else M.netperm = false;
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    std::vector<int> st(H.fronts.size());
    DO_CUDA(ctx, cudaMemcpyAsync(st.data(), M.status.ptr, sizeof(int) * st.size(), cudaMemcpyDeviceToHost, ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    failed_out.clear();
    for (size_t f = 0; f < st.size(); ++f) {
        if (st[f] & 2) failed_out.push_back((int32_t)f);
    }
    if (!failed_out.empty()) return -5;
    for (size_t f = 0; f < st.size(); ++f)
        if (st[f] & 1) return (int32_t)H.fronts[f].first + 1;  // a zero column at this elimination step: singular
    return 0;
}

}  // namespace

extern "C" int32_t diffopt_b200_sparse_setup(diffopt_b200_ctx* ctx, int64_t N, const int64_t* colptr, const int64_t* rowval,
                                             const double* nzval, int32_t trans, int64_t* bandwidth_out) {
    if (!ctx) return -1;
    ctx->sparse_method = 0;
    if (N <= 0 || !colptr || !rowval || !nzval) BAD_ARG(ctx, "sparse_setup: bad argument");
    if (colptr[0] != 1) BAD_ARG(ctx, "sparse_setup: colptr must be 1-based (Julia SparseMatrixCSC)");
    if (N >= (int64_t)1 << 31) BAD_ARG(ctx, "sparse_setup: N too large");
    if (bandwidth_out) *bandwidth_out = -1;
    DeviceGuard guard_(ctx->device);
    const auto t0 = std::chrono::steady_clock::now();
    const int64_t nnz = colptr[N] - 1;
    if (nnz >= ((int64_t)1 << 31) - 1) BAD_ARG(ctx, "sparse_setup: too many nonzeros");
    if (!ctx->sparse_mf) ctx->sparse_mf = new SparseMfImpl();
    SparseMfImpl& M = *ctx->sparse_mf;
    {
        std::string err;
        if (!mf_order(N, colptr, rowval, nzval, M.g, M.snodes, err)) BAD_ARG(ctx, err);
    }
    Graph& g = M.g;
    DO_CUDA(ctx, M.vals.reserve(std::max<size_t>(sizeof(double) * (size_t)nnz, 16)));
    DO_CUDA(ctx, cudaMemcpyAsync(M.vals.ptr, nzval, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream));
    M.retries = 0;
    int32_t rc = 0;
    for (;;) {
        std::string err;
        if (!mf_symbolic(g, M.snodes, N, colptr, rowval, trans, M.H, err)) {
            ctx->err = err;
            return -3;
        }
        M.analysis_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (getenv("DIFFOPT_B200_MF_DEBUG")) {   // how scattered are the rows of a front in the caller's numbering?
            long long rows = 0, sectors = 0, lines = 0, leaves = 0, srows = 0, lists = 0;
            for (const MfFront& f : M.H.fronts) {
                int32_t last = -1, lastl = -1;
                for (int r = 0; r < f.k; ++r) {   // rows of a front are sorted
                    const int32_t v = M.H.perm[(size_t)f.first + r];
                    sectors += (v >> 2) != last;
                    lines += (v >> 4) != lastl;
                    last = v >> 2;
                    lastl = v >> 4;
                }
                rows += f.k;
                leaves += f.leaf != 0;
                srows += f.s;
                lists += f.un;
            }
            fprintf(stderr, "sparse_setup: %zu fronts (%lld leaves), %lld pivot rows in %lld 32-byte sectors / %lld 128-byte lines, %lld boundary rows, %lld update-list entries\n",
                    M.H.fronts.size(), leaves, rows, sectors, lines, srows, lists);
        }
        std::vector<int32_t> failed;
        rc = mf_numeric(ctx, M, nnz, failed);
        if (rc != -5) break;
        if (getenv("DIFFOPT_B200_MF_DEBUG")) {
            const MfFront& f0 = M.H.fronts[(size_t)failed[0]];
            fprintf(stderr, "sparse_setup: pass %d, %zu of %zu fronts need a delayed pivot (first: front %d, k %d, s %d, level-0 leaf %d)\n",
                    M.retries, failed.size(), M.H.fronts.size(), failed[0], f0.k, f0.s, f0.leaf);
        }
        // delayed pivots: merge every failing front into its parent (its columns become fully summed there) and repeat.
        // This ends: a root has no boundary rows, so it never reports a delayed pivot, and every pass removes a front.
        ++M.retries;
        std::vector<char> drop(M.snodes.size(), 0);
        bool progress = false;
        for (int32_t f : failed) {
            int p = M.H.fronts[(size_t)f].parent;
            while (p >= M.H.nreal) p = M.H.fronts[(size_t)p].parent;   // (assembly nodes stand in for their parent)
            if (p < 0) continue;  // a root cannot delay: the pivot is simply unacceptable
            auto& dst = M.snodes[(size_t)p];
            dst.insert(dst.begin(), M.snodes[(size_t)f].begin(), M.snodes[(size_t)f].end());
            drop[(size_t)f] = 1;
            progress = true;
        }
        if (!progress) break;
        std::vector<std::vector<int32_t>> kept;
        for (size_t s = 0; s < M.snodes.size(); ++s)
            if (!drop[s]) kept.push_back(std::move(M.snodes[s]));
        M.snodes.swap(kept);
    }
    if (rc == -5) {   // only if every failing front were a root, which cannot report a delayed pivot
        ctx->err = "sparse_setup: a delayed pivot could not be merged into a parent front";
        return -3;
    }
    if (rc != 0) return rc;
    ctx->sparse_method = 2;
    ctx->sparse_N = N;
    return 0;
}

extern "C" int32_t diffopt_b200_sparse_solve(diffopt_b200_ctx* ctx, int64_t nrhs, const double* rhs, double* x_out, int32_t memspace) {
    if (!ctx) return -1;
    if (ctx->sparse_method != 2 || !ctx->sparse_mf) BAD_ARG(ctx, "sparse_solve: no factorisation (call diffopt_b200_sparse_setup first)");
    if (nrhs <= 0 || !rhs || !x_out) BAD_ARG(ctx, "sparse_solve: bad argument");
    if (nrhs > 65535 * MF_TC) BAD_ARG(ctx, "sparse_solve: too many right-hand sides in one call");
    DeviceGuard guard_(ctx->device);
    SparseMfImpl& M = *ctx->sparse_mf;
    MfHost& H = M.H;
    const int64_t N = ctx->sparse_N;
    const size_t bytes = sizeof(double) * (size_t)N * (size_t)nrhs;
    const void* dB = nullptr;
    void* dX = nullptr;
    DO_CUDA(ctx, stage_in(ctx, ctx->in[5], rhs, bytes, memspace, &dB));
    DO_CUDA(ctx, stage_out_prepare(ctx->out[2], x_out, bytes, memspace, &dX));
    DO_CUDA(ctx, M.Y.reserve(bytes));
    DO_CUDA(ctx, M.W.reserve(std::max<size_t>(sizeof(double) * (size_t)H.w_rows * (size_t)nrhs, 16)));
    const unsigned tiles = (unsigned)((nrhs + MF_TC - 1) / MF_TC);
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const unsigned ltiles = (unsigned)((nrhs + MF_LEAF_TC - 1) / MF_LEAF_TC);
    auto leaf_group = [&](const MfLaunch& L) {
        return L.level == 0 && !L.big && L.max_k <= MF_KMAX && sizeof(double) * (size_t)(MF_KMAX + L.max_nf) * MF_LLD <= MF_SMEM_CAP;
    };
    auto smem_fwd = [](const MfLaunch& L) {
        return ((size_t)L.max_nf * L.max_k + (size_t)MF_TC * (L.max_k | 1) + (size_t)MF_TC * (L.max_s | 1)) * sizeof(double);
    };
    auto smem_bwd = [](const MfLaunch& L) {
        return ((size_t)L.max_k * L.max_k + (size_t)L.max_k * L.max_s + (size_t)MF_TC * (L.max_k | 1) + (size_t)MF_TC * (L.max_s | 1)) *
               sizeof(double);
    };
    auto tiled_smem = [](const MfLaunch& L, bool fwd) {
        return sizeof(double) * ((size_t)L.max_nf * MF_LDT + 1 + (size_t)(fwd ? L.max_nf : L.max_k) * MF_NB) + (fwd ? sizeof(int) * (2 * (size_t)L.max_k + (size_t)L.max_nf + 1 + (size_t)std::min(L.max_u, MF_US_CAP)) : 0);
    };
    auto tiled_group = [&](const MfLaunch& L) {
        return M.netperm && L.max_nf <= MF_TT && tiled_smem(L, true) <= MF_SMEM_CAP && tiled_smem(L, false) <= MF_SMEM_CAP;
    };
    for (const MfLaunch& L : H.launches) {
        if (L.count == 0) continue;
        const dim3 grid((unsigned)L.count, tiles);
        const size_t smem = smem_fwd(L);
        const bool big = L.big || smem > MF_SMEM_CAP;
        if (!leaf_group(L) && tiled_group(L)) {
            const size_t ts = tiled_smem(L, true);
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_forward_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(ts, 1024)));
            mf_forward_tiled_kernel<<<grid, MF_TT, ts, ctx->stream>>>(M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(), M.uptr.as<int>(),
                                                                      M.usrc.as<int>(), M.perm.as<int>(), M.psrc.as<int>(),
                                                                      M.Lp.as<double>(), (const double*)dB, M.Y.as<double>(), M.W.as<double>(), N,
                                                                      (int)nrhs);
        } else if (leaf_group(L)) {
            const size_t ls = sizeof(double) * std::max<size_t>((size_t)L.max_nf * MF_LLD, (size_t)MF_LEAF_TC * (MF_KMAX + 1));
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_forward_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(ls, 1024)));
            mf_forward_leaf_kernel<<<dim3((unsigned)L.count, ltiles), MF_LEAF_TC, ls, ctx->stream>>>(
                M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(), M.perm.as<int>(), M.piv.as<int>(),
                M.netperm ? M.psrc.as<int>() : nullptr, M.Lp.as<double>(), (const double*)dB, M.Y.as<double>(), M.W.as<double>(), N,
                (int)nrhs);
        } else if (!big) {
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_forward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
            mf_forward_kernel<false><<<grid, MF_TC, smem, ctx->stream>>>(M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(),
                                                                         M.child_idx.as<int>(), M.rel.as<int>(), M.perm.as<int>(),
                                                                         M.piv.as<int>(), M.Lp.as<double>(), (const double*)dB,
                                                                         M.Y.as<double>(), M.W.as<double>(), N, (int)nrhs);
        } else {
            mf_forward_kernel<true><<<grid, MF_TC, 0, ctx->stream>>>(M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(),
                                                                     M.child_idx.as<int>(), M.rel.as<int>(), M.perm.as<int>(),
                                                                     M.piv.as<int>(), M.Lp.as<double>(), (const double*)dB, M.Y.as<double>(),
                                                                     M.W.as<double>(), N, (int)nrhs);
        }
        ctx->launches++;
    }
    for (size_t li = H.launches.size(); li-- > 0;) {
        const MfLaunch& L = H.launches[li];
        if (L.count == 0) continue;
        const dim3 grid((unsigned)L.count, tiles);
        const size_t smem = smem_bwd(L);
        const bool big = L.big || smem > MF_SMEM_CAP || smem_fwd(L) > MF_SMEM_CAP;
        if (!leaf_group(L) && tiled_group(L)) {
            const size_t ts = tiled_smem(L, false);
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_backward_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(ts, 1024)));
            mf_backward_tiled_kernel<<<grid, MF_TT, ts, ctx->stream>>>(M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(), M.strct.as<int>(),
                                                                       M.perm.as<int>(), M.Lp.as<double>(), M.Up.as<double>(), M.Y.as<double>(),
                                                                       (double*)dX, N, (int)nrhs);
        } else if (leaf_group(L)) {
            const size_t ls = sizeof(double) * std::max<size_t>((size_t)MF_KMAX * MF_LLD + (size_t)L.max_s * MF_KMAX + (size_t)(L.max_s + 1) / 2 + 1,
                                                                (size_t)MF_LEAF_TC * (MF_KMAX + 1));
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_backward_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(ls, 1024)));
            mf_backward_leaf_kernel<<<dim3((unsigned)L.count, ltiles), MF_LEAF_TC, ls, ctx->stream>>>(
                M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(), M.strct.as<int>(), M.perm.as<int>(), M.Lp.as<double>(),
                M.Up.as<double>(), M.Y.as<double>(), (double*)dX, N, (int)nrhs);
        } else if (!big) {
            DO_CUDA(ctx, cudaFuncSetAttribute(mf_backward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
            mf_backward_kernel<false><<<grid, MF_TC, smem, ctx->stream>>>(M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(),
                                                                          M.strct.as<int>(), M.perm.as<int>(), M.Lp.as<double>(),
                                                                          M.Up.as<double>(), M.Y.as<double>(), (double*)dX, N, (int)nrhs);
        } else {
            mf_backward_kernel<true><<<grid, MF_TC, 0, ctx->stream>>>(M.lists.as<int>() + L.offset, M.fronts.as<MfFront>(),
                                                                      M.strct.as<int>(), M.perm.as<int>(), M.Lp.as<double>(),
                                                                      M.Up.as<double>(), M.Y.as<double>(), (double*)dX, N, (int)nrhs);
        }
        ctx->launches++;
    }
    DO_CUDA(ctx, cudaGetLastError());
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DO_CUDA(ctx, stage_out_finish(ctx, dX, x_out, bytes, memspace));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    return 0;
}

// Host-only analysis (no GPU involved): ordering + symbolic factorisation of a pattern, for inspection and tests.
extern "C" int32_t diffopt_b200_sparse_analyze(int64_t N, const int64_t* colptr, const int64_t* rowval, const double* nzval,
                                               int32_t trans, double* out8) {
    if (N <= 0 || !colptr || !rowval || !out8 || colptr[0] != 1) return -1;
    Graph g;
    std::vector<std::vector<int32_t>> snodes;
    MfHost H;
    std::string err;
    const auto t0 = std::chrono::steady_clock::now();
    if (!mf_order(N, colptr, rowval, nzval, g, snodes, err)) return -1;
    if (!mf_symbolic(g, snodes, N, colptr, rowval, trans, H, err)) return -3;
    out8[0] = 2.0;
    out8[1] = (double)H.fronts.size();
    out8[2] = (double)H.nlevels;
    out8[3] = (double)H.max_front;
    out8[4] = (double)H.nnz_lu;
    out8[5] = H.flops;
    out8[6] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    out8[7] = (double)H.launches.size();
    return 0;
}

extern "C" int32_t diffopt_b200_sparse_stats(diffopt_b200_ctx* ctx, double* out8) {
    if (!ctx || !out8) return -1;
    for (int i = 0; i < 8; ++i) out8[i] = 0.0;
    out8[0] = (double)ctx->sparse_method;
    if (ctx->sparse_method == 2 && ctx->sparse_mf) {
        const SparseMfImpl& M = *ctx->sparse_mf;
        out8[1] = (double)M.H.fronts.size();
        out8[2] = (double)M.H.nlevels;
        out8[3] = (double)M.H.max_front;
        out8[4] = (double)M.H.nnz_lu;
        out8[5] = M.H.flops;
        out8[6] = M.analysis_ms;
        out8[7] = (double)M.retries;
    }
    return 0;
}
