// Fast path of the batched KKT sensitivity solve for ANY shape (n, m, p): the same pivot-free blocked LDL' of the symmetric
// quasi-definite reduced system as qp_batch_sqd.cu (column singletons of inactive inequalities removed, one factorisation
// for forward and reverse mode, every pivot checked, failures re-solved by the pivoted-LU kernel), with the shape read at
// run time.  The factorisation and the backward substitution are the shared code of qp_sqd_dev.cuh; the assembly here is
// written with plain coalesced loops instead of the tile-shaped register pipeline of the headline kernel.
//
// Reference: LHS = [Q G'diag(lam) A'; G diag(Gz-h) 0; A 0 0] (QuadraticProgram.jl:256-282), reverse mode
// LHS x = [dl_dz;0;0] (:324-335), forward mode LHS' x = rhs (:429-438), outputs -x.
//
// Reduced ordering: z (n rows, padded to n8 = 8 ceil(n/8) with identity rows so that the sign change of the pivots falls
// on a tile boundary), active inequalities (ma), equalities (p), padding to a multiple of 8 with -1 on the diagonal.
#include <stdlib.h>

#include "qp_sqd_dev.cuh"

int32_t qp_generic_launch_list(diffopt_b200_ctx* ctx, const QpSolveArgs& a, const int* list, const int* count);
size_t qp_generic_smem_bytes(int n, int m, int p);

namespace {

using namespace sqd;

__host__ __device__ inline int even(int x) { return (x + 1) & ~1; }

// shared-memory carve-up (doubles unless stated), identical on host and device
struct Layout {
    int npc, n8, m2, p2;
    int vecs;     // 8 work vectors of npc
    int zs, lams, dvec, nus, rowq, gcol, acol, rowg, arow, part, apos /* ints, m2 */, scal /* 4 ints */, tiles, total;
    __host__ __device__ Layout(int n, int m, int p, int nt_cap) {
        npc = nt_cap * 8;
        n8 = (n + 7) & ~7;
        m2 = even(m);
        p2 = even(p);
        int o = 0;
        vecs = o; o += 8 * npc;
        zs = o; o += n8;
        lams = o; o += m2;
        dvec = o; o += m2;
        nus = o; o += p2;
        rowq = o; o += n8;
        gcol = o; o += n8;
        acol = o; o += n8;
        rowg = o; o += m2;
        arow = o; o += p2;
        part = o; o += THREADS;
        apos = o; o += even(m2 / 2);
        scal = o; o += 2;
        tiles = o; o += (nt_cap * (nt_cap + 1) / 2) * 64;
        total = o;
    }
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// out[r] = sum_j X[r + j R] zc[j], r < R, for a column-major R x n matrix in global memory.  One owner per row and a fixed
// summation order (bitwise reproducible): rows go to threads, the columns are dealt to 128 / RP thread groups whose
// partial sums meet in shared memory.  Called by all threads; synchronises.
// Optional scatter (T != nullptr): row r with apos[r] >= 0 is also written to row n8 + apos[r] of the tile grid T while it
// passes through the registers (the active rows of G), so G is not read a second time for that.
__device__ void rows_times(const double* __restrict__ X, const int R, const int n, const double* zc, double* out, double* part,
                           double* T = nullptr, const int* apos = nullptr, const int n8 = 0) {
    const int tid = threadIdx.x;
    const int RP = R >= 96 ? 128 : (R > 32 ? 64 : 32), ngrp = THREADS / RP;
    const int ri = tid % RP, grp = tid / RP;
    for (int r0 = 0; r0 < R; r0 += RP) {
        const int r = r0 + ri;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        if (X && r < R) {
            const double* x = X + r;
            const int ar = T ? apos[r] : -1;
            double* trow = nullptr;  // element (n8 + ar, 0) of the tile grid; column c adds (c >> 3) * 64 + the swizzled in-tile offset
            const int Rt = n8 + ar;
            if (ar >= 0) trow = T + tix(Rt >> 3, 0) * 64;
            int j = grp;
            for (; j + 7 * ngrp < n; j += 8 * ngrp) {  // eight independent loads in flight per thread
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldg(x + (size_t)(j + u * ngrp) * R);
                s0 = fma(v[0], zc[j], s0);
                s1 = fma(v[1], zc[j + ngrp], s1);
                s2 = fma(v[2], zc[j + 2 * ngrp], s2);
                s3 = fma(v[3], zc[j + 3 * ngrp], s3);
                s0 = fma(v[4], zc[j + 4 * ngrp], s0);
                s1 = fma(v[5], zc[j + 5 * ngrp], s1);
                s2 = fma(v[6], zc[j + 6 * ngrp], s2);
                s3 = fma(v[7], zc[j + 7 * ngrp], s3);
                if (trow) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int c = j + u * ngrp;
                        trow[(c >> 3) * 64 + el(Rt & 7, c & 7)] = v[u];
                    }
                }
            }
            for (; j < n; j += ngrp) {
                const double v = __ldg(x + (size_t)j * R);
                s0 = fma(v, zc[j], s0);
                if (trow) trow[(j >> 3) * 64 + el(Rt & 7, j & 7)] = v;
            }
        }
        part[tid] = (s0 + s1) + (s2 + s3);
        __syncthreads();
        if (tid < RP && r < R) {
            double s = part[tid];
            for (int q = 1; q < ngrp; ++q) s += part[tid + q * RP];
            out[r] = s;
        }
        __syncthreads();
    }
}

// out[j] = sum_r X[r + j R] wr[r], j < n: one warp per column, lanes over the rows, fixed shuffle tree
__device__ void cols_times(const double* __restrict__ X, const int R, const int n, const double* wr, double* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j0 = 4 * warp; j0 < n; j0 += 4 * NWARP) {  // four columns per pass: their loads and shuffle trees overlap
        double c[4] = {0.0, 0.0, 0.0, 0.0};
        if (X)
            for (int r = lane; r < R; r += 32) {
                const double w = wr[r];
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (j0 + u < n) c[u] = fma(__ldg(X + (size_t)(j0 + u) * R + r), w, c[u]);
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int u = 0; u < 4; ++u) c[u] += __shfl_xor_sync(FULL, c[u], o);
        }
        if (lane < 4 && j0 + lane < n) out[j0 + lane] = lane == 0 ? c[0] : (lane == 1 ? c[1] : (lane == 2 ? c[2] : c[3]));
    }
}

// pull a range of global memory towards L2 (128-byte lines dealt to the CTA's threads)
__device__ __forceinline__ void prefetch_l2(const void* p, const size_t bytes) {
    if (!p) return;
    const char* c = reinterpret_cast<const char*>(p);
    for (size_t o = (size_t)threadIdx.x * 128; o < bytes; o += (size_t)THREADS * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(c + o));
}

// STORE (qp_batch_factorize): no right-hand sides and no outputs; the factor of every instance that passes the pivot test is
// written to `store` (FactorLayout, `stride` doubles per instance) instead of being used, every other instance is listed in
// fb_list and marked in the store.
template <bool STORE>
__global__ void __launch_bounds__(THREADS, 4) qp_kkt_sqd_any_kernel(QpSolveArgs a, int* fb_list, int* fb_count, const int nt_cap,
                                                                     int* max_active, const int max_tag, double* store,
                                                                     const int64_t stride) {
    extern __shared__ __align__(16) double sm[];
    const int n = a.n, m = a.m, p = a.p, N = n + m + p;
    const Layout lay(n, m, p, nt_cap);
    const int n8 = lay.n8, ntz = n8 >> 3, npc = lay.npc;
    const Vecs V = {sm + lay.vecs,           sm + lay.vecs + npc,     sm + lay.vecs + 2 * npc, sm + lay.vecs + 3 * npc, sm + lay.vecs + 4 * npc,
                    sm + lay.vecs + 5 * npc, sm + lay.vecs + 6 * npc, sm + lay.vecs + 7 * npc, reinterpret_cast<int*>(sm + lay.scal) + 2};
    double *const zs = sm + lay.zs, *const lams = sm + lay.lams, *const dvec = sm + lay.dvec, *const nus = sm + lay.nus;
    double *const rowq = sm + lay.rowq, *const gcol = sm + lay.gcol, *const acol = sm + lay.acol, *const rowg = sm + lay.rowg;
    double *const arow = sm + lay.arow, *const part = sm + lay.part, *const T = sm + lay.tiles;
    int* const apos = reinterpret_cast<int*>(sm + lay.apos);
    int* const scal = reinterpret_cast<int*>(sm + lay.scal);  // [0] ma, [1] nt, [2] fail
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int fo = el(g, 2 * t);
    const bool do_fwd = !STORE && a.fwd != nullptr, do_rev = !STORE && a.rev != nullptr;
#ifdef QP_PROFILE
    long long sub[6] = {0, 0, 0, 0, 0, 0};
    long long pc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    long long tprev = clock64();
#define APROF(i)                  \
    do {                          \
        long long _n = clock64(); \
        pc[i] += _n - tprev;      \
        tprev = _n;               \
    } while (0)
#else
#define APROF(i)
#endif

    for (int64_t inst = blockIdx.x; inst < a.B; inst += gridDim.x) {
        const size_t b = (size_t)inst;
        const size_t bm = (a.shared & 1) ? 0 : b, bd = (a.shared & 2) ? 0 : b;
        const double* Q = a.Q + bm * n * n;
        const double* G = m ? a.G + bm * m * n : nullptr;
        const double* A = p ? a.A + bm * p * n : nullptr;
        if (do_fwd && !a.rhs_pre) {  // this instance's direction is consumed a few microseconds from now: pull it into L2
            if (a.dQ) prefetch_l2(a.dQ + bd * n * n, sizeof(double) * n * n);
            if (a.dG && m) prefetch_l2(a.dG + bd * m * n, sizeof(double) * m * n);
            if (a.dA && p) prefetch_l2(a.dA + bd * p * n, sizeof(double) * p * n);
        }
        // ---- vectors, active set
        for (int i = tid; i < n8; i += THREADS) {
            zs[i] = i < n ? a.z[b * n + i] : 0.0;
            V.yb[i] = (do_rev && i < n) ? a.seed[b * n + i] : 0.0;
        }
        for (int i = tid; i < p; i += THREADS) nus[i] = a.nu[b * p + i];
        if (warp == NWARP - 1) {
            int run = 0;
            for (int i0 = 0; i0 < m; i0 += 32) {
                const int i = i0 + lane;
                const double l = i < m ? a.lam[b * m + i] : 0.0;
                const unsigned mask = __ballot_sync(FULL, l != 0.0);
                if (i < m) {
                    lams[i] = l;
                    apos[i] = (l != 0.0) ? run + __popc(mask & ((1u << lane) - 1u)) : -1;
                }
                run += __popc(mask);
            }
            if (lane == 0) {
                scal[0] = run;
                if (max_active) atomicMax(max_active, max_tag | run);
                scal[1] = (n8 + run + p + 7) >> 3;
                scal[2] = 0;
            }
        }
        __syncthreads();
        const int ma = scal[0], nt = scal[1];
        const int nred = n8 + ma + p, np = nt << 3;
        if (nt > nt_cap) {  // larger than this launch was configured for: the pivoted-LU kernel takes it
            if (tid == 0) {
                fb_list[atomicAdd(fb_count, 1)] = (int)inst;
                if (STORE) reinterpret_cast<int*>(store + b * stride)[0] = -1;
            }
            __syncthreads();
            continue;
        }
        // ---- clear the tile grid and the work vectors
        {
            double2* T2 = reinterpret_cast<double2*>(T);
            const int cnt = ((nt * (nt + 1)) >> 1) * 32;
            for (int i = tid; i < cnt; i += THREADS) T2[i] = make_double2(0.0, 0.0);
            for (int i = tid; i < np; i += THREADS) {
                V.yf[i] = 0.0;
                if (i >= n8) V.yb[i] = 0.0;
                V.sf[i] = 0.0;
                V.sb[i] = 0.0;
                V.sf2[i] = 0.0;
                V.sb2[i] = 0.0;
            }
        }
        __syncthreads();
        APROF(0);
        // ---- Q (lower triangle), identity padding, A
#pragma unroll 2
        for (int c = warp; c < n; c += NWARP) {  // a warp per column; six row chunks loaded before their first store
            const double* qc = Q + (size_t)c * n;
            for (int rb = (c & ~31) + lane; rb < n; rb += 192) {
                double v[6];
#pragma unroll
                for (int u = 0; u < 6; ++u) {
                    const int r = rb + 32 * u;
                    v[u] = (r >= c && r < n) ? __ldg(qc + r) : 0.0;
                }
#pragma unroll
                for (int u = 0; u < 6; ++u) {
                    const int r = rb + 32 * u;
                    if (r >= c && r < n) {
                        T[tix(r >> 3, c >> 3) * 64 + el(r & 7, c & 7)] = v[u];
                        if (r == c) V.ref[c] = fabs(v[u]);
                    }
                }
            }
        }
        if (tid < n8 - n) {
            const int r = n + tid;
            T[tix(r >> 3, r >> 3) * 64 + el(r & 7, r & 7)] = 1.0;
            V.ref[r] = 1.0;
        }
        if (tid < np - nred) {
            const int r = nred + tid;
            T[tix(nt - 1, nt - 1) * 64 + el(r & 7, r & 7)] = -1.0;
        }
        for (int e0 = tid; e0 < p * n; e0 += 4 * THREADS) {  // A: p x n entries, four loads in flight per thread
            double v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = e0 + u * THREADS < p * n ? __ldg(A + e0 + u * THREADS) : 0.0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * THREADS;
                if (e < p * n) {
                    const int c = e / p, R = n8 + ma + (e - c * p);
                    T[tix(R >> 3, c >> 3) * 64 + el(R & 7, c & 7)] = v[u];
                }
            }
        }
        APROF(1);
        // ---- D = G z - h; the (2,2) diagonal D_a / lam_a
        rows_times(G, m, n, zs, dvec, part, T, apos, n8);  // ... and the active rows of G into the tile grid
        APROF(2);
        for (int i = tid; i < m; i += THREADS) {
            const double d = dvec[i] - a.h[b * m + i];
            dvec[i] = d;
            const int ar = apos[i];
            if (ar >= 0) {
                const int R = n8 + ar;
                T[tix(R >> 3, R >> 3) * 64 + el(R & 7, R & 7)] = d * fast_rcp(lams[i]);
            } else if (d == 0.0) {
                scal[2] = 1;  // lam_i = D_i = 0: singular column, the LU path reports it
            }
        }
        // ---- forward right-hand side (QuadraticProgram.jl:429-433), symmetric-form scaling
        if (do_fwd && a.rhs_pre) {  // assembled from sparse triplets by qp_coo_rhs_kernel
            const double* r = a.rhs_pre + b * N;
            for (int i = tid; i < n; i += THREADS) V.yf[i] = r[i];
            for (int i = tid; i < m; i += THREADS) {
                const int ar = apos[i];
                if (ar >= 0) V.yf[n8 + ar] = r[n + i];
            }
            for (int i = tid; i < p; i += THREADS) V.yf[n8 + ma + i] = r[n + m + i];
        } else if (do_fwd) {
            const double* dQp = a.dQ ? a.dQ + bd * n * n : nullptr;
            const double* dGp = (a.dG && m) ? a.dG + bd * m * n : nullptr;
            const double* dAp = (a.dA && p) ? a.dA + bd * p * n : nullptr;
            rows_times(dQp, n, n, zs, rowq, part);
            rows_times(dGp, m, n, zs, rowg, part);
            rows_times(dAp, p, n, zs, arow, part);
            cols_times(dGp, m, n, lams, gcol);
            cols_times(dAp, p, n, nus, acol);
            __syncthreads();
            for (int i = tid; i < n; i += THREADS) V.yf[i] = (rowq[i] + (a.dq ? a.dq[b * n + i] : 0.0)) + gcol[i] + acol[i];
            for (int i = tid; i < m; i += THREADS) {
                const int ar = apos[i];
                if (ar >= 0) V.yf[n8 + ar] = rowg[i] - (a.dh ? a.dh[b * m + i] : 0.0);
            }
            for (int i = tid; i < p; i += THREADS) V.yf[n8 + ma + i] = arow[i] - (a.db ? a.db[b * p + i] : 0.0);
        }
        __syncthreads();

        APROF(3);
        factor<0>(T, V, nt, np, ntz, tid, lane, warp, g, t, fo SQD_SUB_ARG);
        __syncthreads();
        APROF(4);
        if constexpr (STORE) {
            double* F = store + b * stride;
            int* Fi = reinterpret_cast<int*>(F);
            const FactorLayout fl(m, nt_cap);
            if (scal[2] == 0) {
                const double2* T2 = reinterpret_cast<const double2*>(T);
                double2* F2 = reinterpret_cast<double2*>(F + fl.tiles);
                const int cnt = ((nt * (nt + 1)) >> 1) * 32;
                for (int i = tid; i < cnt; i += THREADS) F2[i] = T2[i];
                for (int i = tid; i < np; i += THREADS) F[fl.rd + i] = V.rd[i];
                for (int i = tid; i < m; i += THREADS) {
                    F[fl.dvec + i] = dvec[i];
                    Fi[1 + i] = apos[i];
                }
                if (tid == 0) {
                    Fi[0] = ma;
                    if (a.info) a.info[inst] = 0;
                }
            } else if (tid == 0) {
                fb_list[atomicAdd(fb_count, 1)] = (int)inst;
                Fi[0] = -1;
            }
            __syncthreads();
            continue;
        }
        {
            const int lines = (int)(((size_t)m * n * sizeof(double) + 127) / 128);
            backward(T, V, nt, lane, warp, (do_rev && G) ? (const char*)G : nullptr, lines < 1024 ? lines : 1024);
        }
        __syncthreads();
        APROF(5);

        {   // the next instance's problem data travel to L2 while this one is written out (any earlier and the resident CTAs'
            // prefetched lines evict each other: 444 CTAs x 360 KB exceed L2 at n = 100)
            const int64_t nxt = inst + gridDim.x;
            if (nxt < a.B) {
                if (!(a.shared & 1)) {
                    prefetch_l2(a.Q + (size_t)nxt * n * n, sizeof(double) * n * n);
                    if (m) prefetch_l2(a.G + (size_t)nxt * m * n, sizeof(double) * m * n);
                    if (p) prefetch_l2(a.A + (size_t)nxt * p * n, sizeof(double) * p * n);
                }
                prefetch_l2(a.z + (size_t)nxt * n, sizeof(double) * n);
                if (m) prefetch_l2(a.lam + (size_t)nxt * m, sizeof(double) * m);
                if (m) prefetch_l2(a.h + (size_t)nxt * m, sizeof(double) * m);
                if (p) prefetch_l2(a.nu + (size_t)nxt * p, sizeof(double) * p);
                if (do_rev) prefetch_l2(a.seed + (size_t)nxt * n, sizeof(double) * n);
            }
        }
        // ---- outputs (dz, dlam, dnu) = -x; inactive inequalities recovered from their singleton columns
        if (scal[2] == 0) {
            double* rev = do_rev ? a.rev + b * N : nullptr;
            double* fwd = do_fwd ? a.fwd + b * N : nullptr;
            if (do_rev) {
                rows_times(G, m, n, V.yb, rowg, part);  // G x_z
                for (int i = tid; i < n; i += THREADS) rev[i] = -V.yb[i];
                for (int i = tid; i < m; i += THREADS) {
                    const int ar = apos[i];
                    rev[n + i] = ar >= 0 ? -V.yb[n8 + ar] * fast_rcp(lams[i]) : rowg[i] * fast_rcp(dvec[i]);
                }
                for (int i = tid; i < p; i += THREADS) rev[n + m + i] = -V.yb[n8 + ma + i];
            }
            if (do_fwd) {
                for (int i = tid; i < n; i += THREADS) fwd[i] = -V.yf[i];
                for (int i = tid; i < m; i += THREADS) {
                    const int ar = apos[i];
                    fwd[n + i] = ar >= 0 ? -V.yf[n8 + ar] : 0.0;
                }
                for (int i = tid; i < p; i += THREADS) fwd[n + m + i] = -V.yf[n8 + ma + i];
            }
            if (a.info && tid == 0) a.info[inst] = 0;
        } else if (tid == 0) {
            fb_list[atomicAdd(fb_count, 1)] = (int)inst;
        }
        __syncthreads();
        APROF(6);
    }
#ifdef QP_PROFILE
    if (a.prof && blockIdx.x == 0 && tid == 0)
        for (int i = 0; i < 7; ++i) a.prof[i] = pc[i];
#endif
}

__global__ void max_active_any_kernel(int64_t B, int m, const double* __restrict__ lam, int* out) {
    int best = 0;
    const int lane = threadIdx.x & 31;
    for (int64_t b = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); b < B; b += (int64_t)gridDim.x * (blockDim.x >> 5)) {
        int c = 0;
        for (int i = lane; i < m; i += 32) c += lam[b * m + i] != 0.0;
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
        best = max(best, c);
    }
    if (lane == 0 && best > 0) atomicMax(out, best);
}

}  // namespace

// tile order of the reduced system when `active` inequalities are active
int qp_sqd_any_nt(const QpSolveArgs& a, int active) { return (((a.n + 7) & ~7) + active + a.p + 7) / 8; }

// Largest tile order whose shared-memory layout fits one CTA (0: not even the z block plus one constraint tile fits).
int qp_sqd_any_nt_limit(diffopt_b200_ctx* ctx, const QpSolveArgs& a) {
    const int ntz = (a.n + 7) / 8;
    int nt = qp_sqd_any_nt(a, a.m);  // all inequalities active
    while (nt > ntz && (size_t)Layout(a.n, a.m, a.p, nt).total * sizeof(double) > ctx->smem_optin) --nt;
    if ((size_t)Layout(a.n, a.m, a.p, nt).total * sizeof(double) > ctx->smem_optin) return 0;
    return nt;
}

// The fast path serves a shape when the reduced system of an instance with no active inequality fits one CTA's shared
// memory; instances whose active set outgrows what fits are handed to the pivoted-LU kernel like any other reject (that
// kernel keeps the matrix in shared memory up to N = 165 and in global memory beyond).
bool qp_sqd_any_supported(diffopt_b200_ctx* ctx, const QpSolveArgs& a) {
    if (a.m > 255) return false;  // the active-set report carries the size in one byte
    return qp_sqd_any_nt_limit(ctx, a) >= qp_sqd_any_nt(a, 0);
}

int32_t qp_max_active_any_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a, int* dmax) {
    int64_t blocks = (a.B + 7) / 8;
    if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
    if (blocks < 1) blocks = 1;
    max_active_any_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(a.B, a.m, a.lam, dmax);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// Launches the shape-generic LDL' fast path followed by the generic pivoted-LU kernel over the instances it rejected.
int32_t qp_sqd_any_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a, int nt_cap, bool* handled, int* max_active, int max_tag) {
    *handled = false;
    const Layout lay(a.n, a.m, a.p, nt_cap);
    const size_t smem = (size_t)lay.total * sizeof(double);
    if (smem > ctx->smem_optin) return 0;
    DO_CUDA(ctx, ctx->qp_fb.reserve(sizeof(int) * ((size_t)a.B + 1)));
    int* fb_count = ctx->qp_fb.as<int>();
    int* fb_list = fb_count + 1;
    DO_CUDA(ctx, cudaMemsetAsync(fb_count, 0, sizeof(int), ctx->stream));
    int per_sm = 1;
    DO_CUDA(ctx, kernel_config((const void*)qp_kkt_sqd_any_kernel<false>, ctx->device, THREADS, smem, &per_sm));
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)ctx->sm_count * per_sm;
    if (grid > a.B) grid = a.B;
    if (grid < 1) grid = 1;
    QpSolveArgs aa = a;
    long long* dprof = nullptr;
    const bool profile = getenv("DIFFOPT_B200_PROFILE") != nullptr;
    if (profile) {
        DO_CUDA(ctx, cudaMalloc(&dprof, 16 * sizeof(long long)));
        DO_CUDA(ctx, cudaMemsetAsync(dprof, 0, 16 * sizeof(long long), ctx->stream));
        aa.prof = dprof;
    }
    qp_kkt_sqd_any_kernel<false><<<(unsigned)grid, THREADS, smem, ctx->stream>>>(aa, fb_list, fb_count, nt_cap, max_active, max_tag,
                                                                                 nullptr, 0);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    if (profile) {  // per-phase clocks of CTA 0 (profile build: DIFFOPT_B200_BUILD_PROFILE=1)
        long long h[16];
        DO_CUDA(ctx, cudaMemcpyAsync(h, dprof, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
        DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(dprof);
        const long long ninst = (a.B + grid - 1) / grid;
        fprintf(stderr, "[qp_sqd_any profile, CTA 0, %lld instances, %d CTA/SM, nt_cap %d, smem %zu] clocks/instance: vectors+clear %lld, "
                        "scatter Q/G/A %lld, G z %lld, forward rhs %lld, factor %lld, backward %lld, output %lld\n",
                ninst, per_sm, nt_cap, smem, h[0] / ninst, h[1] / ninst, h[2] / ninst, h[3] / ninst, h[4] / ninst, h[5] / ninst, h[6] / ninst);
    }
    *handled = true;
    return qp_generic_launch_list(ctx, a, fb_list, fb_count);
}

// Store mode (qp_batch_factorize): the same factorisation of every instance of `a` (no right-hand sides), factors written to
// `store` (FactorLayout(m, nt_cap), `stride` doubles per instance); instances that fail the pivot test or exceed nt_cap are
// appended to fb_list / *fb_count (cleared here).  a.info[b] = 0 for every stored instance.
int32_t qp_sqd_any_store_launch(diffopt_b200_ctx* ctx, const QpSolveArgs& a, int nt_cap, double* store, int64_t stride, int* fb_list,
                                int* fb_count) {
    const size_t smem = (size_t)Layout(a.n, a.m, a.p, nt_cap).total * sizeof(double);
    DO_CUDA(ctx, cudaMemsetAsync(fb_count, 0, sizeof(int), ctx->stream));
    int per_sm = 1;
    DO_CUDA(ctx, kernel_config((const void*)qp_kkt_sqd_any_kernel<true>, ctx->device, THREADS, smem, &per_sm));
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)ctx->sm_count * per_sm;
    if (grid > a.B) grid = a.B;
    if (grid < 1) grid = 1;
    QpSolveArgs aa = a;
    aa.fwd = aa.rev = nullptr;
    aa.prof = nullptr;
    qp_kkt_sqd_any_kernel<true><<<(unsigned)grid, THREADS, smem, ctx->stream>>>(aa, fb_list, fb_count, nt_cap, nullptr, 0, store, stride);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    return 0;
}
