// Persistent cooperative LSQR kernel + the conic matrix-free operator.  See lsqr.cuh.
#include <cooperative_groups.h>

#include <algorithm>
#include <thread>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "lsqr.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int LSQR_THREADS = 256;

#ifdef LSQR_PROF
__device__ long long g_prof[8192];
__device__ int g_prof_n;
__device__ __forceinline__ long long gtimer() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

struct Dev {
    cg::grid_group grid;
    double* partials;  // [LSQR_NSLOTS][nblk]
    double* red;       // shared scratch (>= 2 * warps doubles)
    int tid, lane, warp, nwarp, nblk, gtid, gthreads;
    bool cluster = false;  // the whole grid is ONE thread-block cluster: hardware barrier instead of grid.sync()
    // batched launches (one problem per cluster of `nblk` CTAs, lsqr_batch_kernel): rank of this CTA inside its problem
    // (-1: the grid is one problem, rank = blockIdx.x) and whether the problem lives in a single CTA (barrier = bar.sync)
    int cta = -1;
    bool cta_only = false;
    __device__ __forceinline__ int rank() const { return cta >= 0 ? cta : (int)blockIdx.x; }
    // All-CTA barrier with release/acquire ordering of global memory.  The cluster barrier costs ~0.2 us (and
    // invalidates L1, so plain loads after it see the other CTAs' stores); cooperative grid.sync() costs 2-3 us.
    __device__ __forceinline__ void sync() {
#ifdef LSQR_PROF
        if (gtid == 0 && g_prof_n < 8190) g_prof[g_prof_n++] = gtimer();
#endif
        sync_();
#ifdef LSQR_PROF
        if (gtid == 0 && g_prof_n < 8190) g_prof[g_prof_n++] = gtimer();
#endif
    }
    __device__ __forceinline__ void sync_() {
        if (cta_only)
            __syncthreads();
        else if (cluster)
            asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        else
            grid.sync();
    }
};

// Dev of a problem solved by the whole grid, its partial sums in columns of `nblk`
__device__ __forceinline__ Dev make_dev(double* partials, double* red, int nblk) {
    return Dev{cg::this_grid(), partials, red, (int)threadIdx.x, (int)(threadIdx.x & 31), (int)(threadIdx.x >> 5),
               (int)(blockDim.x >> 5), nblk, (int)(blockIdx.x * blockDim.x + threadIdx.x), (int)(gridDim.x * blockDim.x)};
}

__device__ __forceinline__ double warp_sum_all(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-level sum of `v`, result stored as this CTA's partial in `slot`
__device__ void block_partial(Dev& d, int slot, double v) {
    v = warp_sum_all(v);
    if (d.lane == 0) d.red[d.warp] = v;
    __syncthreads();
    if (d.tid == 0) {
        double s = 0.0;
        for (int w = 0; w < d.nwarp; ++w) s += d.red[w];
        d.partials[slot * d.nblk + d.rank()] = s;
    }
    __syncthreads();
}

// after a grid.sync(): fixed-order sum of all CTA partials of `slot` (bitwise identical in every thread)
__device__ double total_of(Dev& d, int slot) {
    const double* p = d.partials + slot * d.nblk;
    double s = 0.0;
    for (int i = d.lane; i < d.nblk; i += 32) s += __ldcg(p + i);
    return warp_sum_all(s);
}

constexpr int SP_THREADS = 128;                   // threads of a streaming-SpMV CTA (8 CTAs per SM)
constexpr int ST_NPT = 8;                         // nonzeros per thread in flight
constexpr int ST_CHUNK = SP_THREADS * ST_NPT;     // nonzeros per row block
// cluster-synchronised kernel (small operators): one cluster of CL_THREADS-thread CTAs, same SpMV with bigger blocks
#ifndef CL_THREADS_DEF
#define CL_THREADS_DEF 512
#endif
constexpr int CL_THREADS = CL_THREADS_DEF;
constexpr int CL_NPT = 8;
constexpr int CL_CHUNK = CL_THREADS * CL_NPT;
constexpr int CL_MAX_CTAS = 16;
// the 256-thread persistent kernel (problems with PSD cones) and conic_M_kernel run on the row blocks of the streaming
// driver (CsrDev::blk / t_blk): <= ST_CHUNK nonzeros and <= SP_THREADS rows per block, or one longer row
constexpr int LSQR_NPT = 4;
static_assert(LSQR_THREADS * LSQR_NPT == ST_CHUNK && LSQR_THREADS >= SP_THREADS, "shape does not fit the blk lists");
constexpr int ST_STRIDE = 2048;  // capacity of one partial slot = upper bound of every streaming grid

// Row-block ("CSR-stream") SpMV, the sparse product of every LSQR driver.  The host cuts the rows into blocks of
// <= THREADS * NPT nonzeros (and <= THREADS rows, or one longer row) and stores (first row, first nonzero) per block.
// A CTA owns a CONTIGUOUS range of blocks, so the part of x it gathers from slides slowly and stays in L1 when the
// matrix has any locality (the kernels keep shared memory small to leave L1 its capacity).  Per block: NPT independent,
// fully coalesced (val, colind) loads per thread -- no dependence on row pointers, so the HBM pipe stays full regardless
// of the row lengths -- then the x gathers (read-only path) with the row's epilogue operands loaded underneath them
// (`pre(b, row)`), products parked in shared memory, one row per thread reduced in storage order (deterministic),
// `epi(b, row, value, operands)` once per row.
// sel(b, A, x, lb): matrix, gather vector and local block index of global block b.
// XCG: x was written earlier in the SAME launch (persistent kernels) -> gather with ld.global.cg, not the read-only path.
// XM: how x is gathered.  0: read-only path (x constant during the launch); 1: ld.global.cg (x was written earlier in the
// SAME launch by other CTAs: persistent kernels); 2: plain generic loads -- x is a copy staged in SHARED memory by the
// caller (one problem per CTA: the whole gather vector fits, and shared-memory gathers are not bound by the one-sector-
// per-request rate of L1TEX that caps the global-memory forms at ~50 % of HBM).  The matrix streams evict-first for 0, 2.
// cta / ncta: this CTA's rank among the CTAs that share the blocks.
template <int THREADS, int NPT, int XM, class Sel, class Pre, class Epi>
__device__ __forceinline__ void spmv_stream(int cta, int ncta, int nblk_total, double* prod, double* red, Sel&& sel, Pre&& pre,
                                            Epi&& epi) {
    constexpr int CHUNK = THREADS * NPT;
    constexpr bool XCG = XM == 1;
    const int tid = threadIdx.x;
    const int per = (nblk_total + ncta - 1) / ncta;
    const int b_end = min(nblk_total, (cta + 1) * per);
    for (int b = cta * per; b < b_end; ++b) {
        const CsrView* A;
        const double* x;
        int lb;
        sel(b, A, x, lb);
        const int2 d0 = __ldg(reinterpret_cast<const int2*>(A->blk) + lb);
        const int2 d1 = __ldg(reinterpret_cast<const int2*>(A->blk) + lb + 1);
        const int r0 = d0.x, s = d0.y, r1 = d1.x, cnt = d1.y - d0.y;
        if (cnt > CHUNK) {  // one long row: whole CTA, fixed-order reduction
            double acc = 0.0;
            for (int k = tid; k < cnt; k += THREADS)
                {
                const double* xp = x + (XCG ? __ldg(A->colind + s + k) : __ldcs(A->colind + s + k));
                acc = fma(XCG ? __ldg(A->val + s + k) : __ldcs(A->val + s + k), XM == 2 ? *xp : (XCG ? __ldcg(xp) : __ldg(xp)), acc);
            }
            acc = warp_sum_all(acc);
            if ((tid & 31) == 0) red[32 + (tid >> 5)] = acc;
            __syncthreads();
            if (tid == 0) {
                double t = 0.0;
                for (int w = 0; w < THREADS / 32; ++w) t += red[32 + w];
                epi(b, r0, t, pre(b, r0));
            }
        } else {
            double av[NPT];
            int ci[NPT];
            int ps[NPT];  // slot of the product in `prod` (CSR position inside the block)
            const bool sorted = XM == 0 && A->spos != nullptr;  // column-ordered copy of the block (large operators)
#pragma unroll
            for (int u = 0; u < NPT; ++u) {
                const int k = tid + u * THREADS;
                av[u] = 0.0;
                ci[u] = 0;
                ps[u] = k;
                if (k < cnt) {  // streamed once per pass (evict-first) unless the operator lives in L2 (XCG kernels)
                    if (sorted) {
                        av[u] = __ldcs(A->sval + s + k);
                        ci[u] = __ldcs(A->scol + s + k);
                        ps[u] = __ldcs(A->spos + s + k);
                    } else {
                        av[u] = XCG ? __ldg(A->val + s + k) : __ldcs(A->val + s + k);
                        ci[u] = XCG ? __ldg(A->colind + s + k) : __ldcs(A->colind + s + k);
                    }
                }
            }
            // T threads per row (power of two, as many as the block's row count allows): rows of a few hundred nonzeros
            // (KKT matrices with dense blocks) are not summed by one thread; fixed order either way
            int T = 1;
            while (T < 32 && (r1 - r0) * T * 2 <= THREADS) T <<= 1;
            const int row = r0 + tid / T, sub = tid & (T - 1);
            int ra = 0, rb = 0;
            if (row < r1) {
                ra = __ldg(A->rowptr + row) - s;
                rb = __ldg(A->rowptr + row + 1) - s;
            }
            double xv[NPT];
#pragma unroll
            for (int u = 0; u < NPT; ++u)
                xv[u] = (tid + u * THREADS < cnt) ? (XM == 2 ? x[ci[u]] : (XCG ? __ldcg(x + ci[u]) : __ldg(x + ci[u]))) : 0.0;
            double4 opnd = make_double4(0.0, 0.0, 0.0, 0.0);
            if (row < r1 && sub == 0) opnd = pre(b, row);
#pragma unroll
            for (int u = 0; u < NPT; ++u)
                if (tid + u * THREADS < cnt) prod[ps[u]] = av[u] * xv[u];
            __syncthreads();
            double t = 0.0;
            for (int k = ra + sub; k < rb; k += T) t += prod[k];
            for (int o = T >> 1; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (row < r1 && sub == 0) epi(b, row, t, opnd);
        }
        __syncthreads();  // prod / red are free again
    }
}

// ---- SOC block of Dpi applied to y (symmetric block, so it serves Dpi and Dpi') ------------------
// group of `T` lanes handles cone `c`; writes out[off .. off+dim)
__device__ void soc_apply(const ConicOpView& op, int c, bool valid, const double* __restrict__ y, double* out,
                          int lig, int T) {
    int off = 0, dim = 0, cs = 0;
    double nx = 1.0, t = 0.0;
    if (valid) {
        off = op.soc_off[c];
        dim = op.soc_dim[c];
        cs = op.soc_case[c];
        nx = op.soc_nx[c];
        t = op.v[off];
    }
    double xy = 0.0;
    if (valid && cs == 2)
        for (int k = 1 + lig; k < dim; k += T) xy += op.v[off + k] * __ldcg(y + off + k);
    for (int o = T >> 1; o > 0; o >>= 1) xy += __shfl_xor_sync(0xffffffffu, xy, o);
    if (!valid) return;
    if (cs == 0) {
        for (int k = lig; k < dim; k += T) out[off + k] = __ldcg(y + off + k);
    } else if (cs == 1) {
        for (int k = lig; k < dim; k += T) out[off + k] = 0.0;
    } else {
        const double y0 = __ldcg(y + off);
        const double inv2 = 1.0 / (2.0 * nx);
        const double coef = t / (nx * nx) * xy;
        for (int k = lig; k < dim; k += T) {
            double r;
            if (k == 0)
                r = nx * y0 + xy;
            else {
                double xk = op.v[off + k];
                r = xk * y0 + (nx + t) * __ldcg(y + off + k) - coef * xk;
            }
            out[off + k] = r * inv2;
        }
    }
}

// ---- PSD block: out = Dpi*y (transpose=false) or Dpi'*y (true), whole grid cooperates ------------
// Dpi' y = vec(F(unvec(y)));  Dpi y = S' F T' y  (diag of unvec doubled on the way in, halved on the way out),
// F(X) = U (B o (U' X U)) U'.  Four GEMM phases on the FP64 tensor pipe (mma.sync m8n8k4), 3 barriers inside:
//   W1 = U' X        (X read straight from the triangle y)
//   W2 = (W1 U) o B
//   W1 = U W2
//   out = vec(W1 U') (upper-triangle tiles only, written straight into the triangle)
// Work unit = one 32 x 32 output tile of one cone (tiles of all cones in one list, so 512 small cones fill the grid as
// well as one 200 x 200 cone does); a 256-thread CTA stages 32-deep operand panels in shared memory ([k][i] layout,
// leading dimension 36: fragment reads are bank-conflict free), next panel prefetched into registers under the MMAs.
constexpr int PT = 32;        // tile side
constexpr int PLD = PT + 4;   // panel leading dimension (doubles)

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

// C(i0.., j0..) = sum_k la(i, k) * lb(k, j); st(i, j, value) for every in-range element of the tile.
// a_ic / b_kc: which index is contiguous in memory for the A / B operand (chooses the coalesced load mapping).
template <class LA, class LB, class ST>
__device__ __forceinline__ void psd_tile_gemm(int dd, int i0, int j0, bool a_ic, bool b_kc, double* As, double* Bs,
                                              LA&& la, LB&& lb, ST&& st) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int iw = (warp & 3) * 8, jw = (warp >> 2) * 16;
    const int f = tid & 31, s8 = tid >> 5;  // fast / slow index of the load mapping (slow: s8 + 8 r)
    double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
    double ra[4], rb[4];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int sl = s8 + 8 * r;
            const int ia = a_ic ? f : sl, ka = a_ic ? sl : f;
            const int kb = b_kc ? f : sl, jb = b_kc ? sl : f;
            ra[r] = (i0 + ia < dd && k0 + ka < dd) ? la(i0 + ia, k0 + ka) : 0.0;
            rb[r] = (k0 + kb < dd && j0 + jb < dd) ? lb(k0 + kb, j0 + jb) : 0.0;
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < dd; k0 += PT) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int sl = s8 + 8 * r;
            const int ia = a_ic ? f : sl, ka = a_ic ? sl : f;
            const int kb = b_kc ? f : sl, jb = b_kc ? sl : f;
            As[ka * PLD + ia] = ra[r];
            Bs[kb * PLD + jb] = rb[r];
        }
        __syncthreads();
        if (k0 + PT < dd) fetch(k0 + PT);
#pragma unroll
        for (int kk = 0; kk < PT; kk += 4) {
            const int kr = (kk + (lane & 3)) * PLD;
            const double av = As[kr + iw + (lane >> 2)];
            const double b0 = Bs[kr + jw + (lane >> 2)];
            const double b1 = Bs[kr + jw + 8 + (lane >> 2)];
            dmma884(c00, c01, av, b0);
            dmma884(c10, c11, av, b1);
        }
        __syncthreads();
    }
    const int i = i0 + iw + (lane >> 2), j = j0 + jw + 2 * (lane & 3);
    if (i < dd) {
        if (j < dd) st(i, j, c00);
        if (j + 1 < dd) st(i, j + 1, c01);
        if (j + 8 < dd) st(i, j + 8, c10);
        if (j + 9 < dd) st(i, j + 9, c11);
    }
}

__device__ void psd_apply_all(Dev& d, const ConicOpView& op, const double* __restrict__ y, double* out,
                              bool transpose) {
    if (op.npsd == 0) return;
    __shared__ double As[PT * PLD], Bs[PT * PLD];
    const double dscale = transpose ? 1.0 : 2.0, oscale = transpose ? 1.0 : 0.5;
    for (int phase = 0; phase < 4; ++phase) {
        for (int t = blockIdx.x; t < op.psd_ntiles; t += gridDim.x) {
            // cone of tile t: last c with toff[c] <= t
            int lo = 0, hi = op.npsd - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (__ldg(op.psd_toff + mid) <= t) lo = mid; else hi = mid - 1;
            }
            const int c = lo, dd = op.psd_d[c], off = op.psd_off[c];
            const int nt = (dd + PT - 1) / PT, lt = t - __ldg(op.psd_toff + c);
            const int i0 = (lt % nt) * PT, j0 = (lt / nt) * PT;
            const long long uo = op.psd_uoff[c];
            const double* U = op.psd_U + uo;
            double* W1 = op.psd_w1 + uo;
            double* W2 = op.psd_w2 + uo;
            const double* yc = y + off;
            if (op.psd_ident[c]) {  // Dpi = I on this cone
                if (phase == 3)
                    for (int e = threadIdx.x; e < PT * PT; e += blockDim.x) {
                        const int i = i0 + e % PT, j = j0 + e / PT;
                        if (i <= j && j < dd) out[off + (long long)j * (j + 1) / 2 + i] = __ldcg(yc + (long long)j * (j + 1) / 2 + i);
                    }
                continue;
            }
            if (phase == 0) {  // W1 = U' X
                psd_tile_gemm(dd, i0, j0, false, true, As, Bs,
                    [&](int i, int k) { return U[k + (long long)i * dd]; },
                    [&](int k, int j) {
                        const int r = k < j ? k : j, cc = k < j ? j : k;
                        const double v = __ldcg(yc + (long long)cc * (cc + 1) / 2 + r);
                        return k == j ? v * dscale : v;
                    },
                    [&](int i, int j, double v) { W1[i + (long long)j * dd] = v; });
            } else if (phase == 1) {  // W2 = (W1 U) o B
                const double* Bm = op.psd_Bm + uo;
                psd_tile_gemm(dd, i0, j0, true, true, As, Bs,
                    [&](int i, int k) { return __ldcg(W1 + i + (long long)k * dd); },
                    [&](int k, int j) { return U[k + (long long)j * dd]; },
                    [&](int i, int j, double v) { W2[i + (long long)j * dd] = v * Bm[i + (long long)j * dd]; });
            } else if (phase == 2) {  // W1 = U W2
                psd_tile_gemm(dd, i0, j0, true, true, As, Bs,
                    [&](int i, int k) { return U[i + (long long)k * dd]; },
                    [&](int k, int j) { return __ldcg(W2 + k + (long long)j * dd); },
                    [&](int i, int j, double v) { W1[i + (long long)j * dd] = v; });
            } else if (i0 <= j0 + PT - 1) {  // out = vec(W1 U'), tiles touching the upper triangle
                psd_tile_gemm(dd, i0, j0, true, false, As, Bs,
                    [&](int i, int k) { return __ldcg(W1 + i + (long long)k * dd); },
                    [&](int k, int j) { return U[j + (long long)k * dd]; },
                    [&](int i, int j, double v) {
                        if (i <= j) out[off + (long long)j * (j + 1) / 2 + i] = i == j ? v * oscale : v;
                    });
            }
        }
        if (phase < 3) d.sync();
    }
    // caller syncs
}

// Dpi (or Dpi') applied to y -> out, for all cones; ends WITHOUT a grid sync when there is no PSD cone
// PSD = false compiles the PSD-cone phases out (the cluster, gstream and batch kernels and the streaming driver never
// run problems with PSD cones; their kernels stay small).
template <bool PSD>
__device__ void dpi_apply(Dev& d, const ConicOpView& op, const double* __restrict__ y, double* out, bool transpose) {
    for (int i = d.gtid; i < op.m; i += d.gthreads) {
        const int k = op.kind[i];
        if (k == 0) {
            out[i] = op.diag[i] * __ldcg(y + i);
        } else if (k >= 4) {  // row k - 4 of a symmetric 3 x 3 block (exp cones): the same for Dpi and Dpi'
            const double* br = op.blk3 + 3 * (long long)i;
            const double* yc = y + (i - (k - 4));
            out[i] = br[0] * __ldcg(yc) + br[1] * __ldcg(yc + 1) + br[2] * __ldcg(yc + 2);
        }
    }
    {
        const int T = 8;
        const int lig = d.lane & (T - 1);
        const int ngroups = d.gthreads / T;
        const int g = d.gtid / T;
        for (int base = 0; base < op.nsoc; base += ngroups) {
            int c = base + g;
            soc_apply(op, c, c < op.nsoc, y, out, lig, T);
        }
    }
    if constexpr (PSD) psd_apply_all(d, op, y, out, transpose);
}

// ------------------------------------------------------------------------------------------------
// Operator application  dst = OP(src)*s_src + s_dst*dst  with ||dst||^2 reduced into `slot`.
// CSR:   OP = A (rows) or its transpose view (the caller hands the right CsrView).
// CONIC: OP = M or M'.
// All functions are called by the whole grid and contain grid syncs.

extern __shared__ double cl_prod[];  // THREADS * NPT products (dynamic shared memory of the persistent launches)

// THREADS / NPT: row-block shape of the launch (the block list the host hands over is cut for it), see spmv_stream.
template <int THREADS, int NPT>
__device__ void csr_apply(Dev& d, const CsrView& A, const double* __restrict__ src, double s_src, double* dst,
                          double s_dst, int slot) {
    double acc = 0.0;
    spmv_stream<THREADS, NPT, 1>(
        d.rank(), d.nblk, A.nblk, cl_prod, d.red, [&](int b, const CsrView*& M, const double*& x, int& lb) { M = &A; x = src; lb = b; },
        [&](int, int row) { return make_double4(s_dst != 0.0 ? __ldcg(dst + row) : 0.0, 0.0, 0.0, 0.0); },
        [&](int, int row, double t, const double4& o) {
            t = t * s_src + s_dst * o.x;
            dst[row] = t;
            acc += t * t;
        });
    block_partial(d, slot, acc);
}

// ---- Row-block phases of the conic operator, shared by conic_apply and the streaming kernels.  The CTAs
// that share the row blocks number `ncta`, this one is `cta`; prod / red: shared scratch of spmv_stream.  xw / xs: the
// vectors the products gather from (wc and src or src + n, or their copies staged in shared memory for XM = 2).
// Partial sums accumulate into acc (||dst||^2) and dot.  dst is read with ld.global.cg where other CTAs of the same
// launch wrote it (XM != 0), with plain loads in the one-kernel-per-phase streaming driver.
template <int XM>
__device__ __forceinline__ double ld_dst(const double* p) { return XM == 0 ? *p : __ldcg(p); }

// M src: rows 0..n-1 (A' wc)_j + c_j t3, rows n..n+m-1 -(A t1)_i + t2_i - wc_i + b_i t3; dst = s_src * row + s_dst * dst,
// dot += c't1 + b'wc
template <int THREADS, int NPT, int XM>
__device__ __forceinline__ void conic_M_rows(const ConicOpView& op, int cta, int ncta, double* prod, double* red,
                                             const double* __restrict__ src, const double* xw, const double* xs, double t3,
                                             double s_src, double* dst, double s_dst, double& acc, double& dot) {
    const int n = op.n, nbt = op.At.nblk;
    spmv_stream<THREADS, NPT, XM>(
        cta, ncta, nbt + op.A.nblk, prod, red,
        [&](int b, const CsrView*& A, const double*& x, int& lb) {
            if (b < nbt) { A = &op.At; x = xw; lb = b; }
            else { A = &op.A; x = xs; lb = b - nbt; }
        },
        [&](int b, int row) {
            return b < nbt ? make_double4(op.c[row], ld_dst<XM>(dst + row), __ldcg(src + row), 0.0)
                           : make_double4(__ldcg(op.wc + row), __ldcg(src + n + row), op.b[row], ld_dst<XM>(dst + n + row));
        },
        [&](int b, int row, double t, const double4& o) {
            if (b < nbt) {
                t = (t + o.x * t3) * s_src + s_dst * o.y;
                dst[row] = t;
                acc += t * t;
                dot += o.x * o.z;
            } else {
                t = (-t + o.y - o.x + o.z * t3) * s_src + s_dst * o.w;
                dst[n + row] = t;
                acc += t * t;
                dot += o.z * o.x;
            }
        });
}

// M' src, phase 1: wc = A u1 - u2 - b u3, dot += b'u2
template <int THREADS, int NPT, int XM>
__device__ __forceinline__ void conic_Mt_A(const ConicOpView& op, int cta, int ncta, double* prod, double* red,
                                           const double* __restrict__ src, const double* xs, double u3, double& dot) {
    const int n = op.n;
    spmv_stream<THREADS, NPT, XM>(
        cta, ncta, op.A.nblk, prod, red,
        [&](int b, const CsrView*& A, const double*& x, int& lb) { A = &op.A; x = xs; lb = b; },
        [&](int, int row) { return make_double4(__ldcg(src + n + row), op.b[row], 0.0, 0.0); },
        [&](int, int row, double t, const double4& o) {
            op.wc[row] = t - o.x - o.y * u3;
            dot += o.y * o.x;
        });
}

// M' src, phase 3 (after r2 = Dpi' wc, stored behind wc): rows 0..n-1 -(A' u2)_j - c_j u3, rows n..n+m-1 r2_i + u2_i;
// dst = s_src * row + s_dst * dst, dot += c'u1
template <int THREADS, int NPT, int XM>
__device__ __forceinline__ void conic_Mt_rows(const ConicOpView& op, int cta, int ncta, double* prod, double* red,
                                              const double* __restrict__ src, const double* xs, double u3, double s_src,
                                              double* dst, double s_dst, double& acc, double& dot) {
    const int n = op.n, m = op.m;
    spmv_stream<THREADS, NPT, XM>(
        cta, ncta, op.At.nblk, prod, red,
        [&](int b, const CsrView*& A, const double*& x, int& lb) { A = &op.At; x = xs; lb = b; },
        [&](int, int row) { return make_double4(op.c[row], ld_dst<XM>(dst + row), __ldcg(src + row), 0.0); },
        [&](int, int row, double t, const double4& o) {
            t = (-t - o.x * u3) * s_src + s_dst * o.y;
            dst[row] = t;
            acc += t * t;
            dot += o.x * o.z;
        });
    const double* r2 = op.wc + m;
    for (int i = cta * THREADS + (int)threadIdx.x; i < m; i += ncta * THREADS) {
        const double t = (__ldcg(r2 + i) + __ldcg(src + n + i)) * s_src + s_dst * ld_dst<XM>(dst + n + i);
        dst[n + i] = t;
        acc += t * t;
    }
}

// dst = s_src * (M src) + s_dst * dst ; slots: slot (norm), slot+1 (last-row dot)
// `src_last` / `dst_last` are every thread's private copies of src[N-1] / dst[N-1] (all threads compute the last row
// identically): nobody reads those entries from memory, so thread 0 may store the new one right after the barrier
// that publishes the partial sums, and ||dst||^2 (returned in `norm2`) is complete without another barrier.
// SM (batched launches, one problem per CTA): the vectors the products gather from are first copied into shared memory
// (behind the THREADS * NPT products: n + m doubles), see spmv_stream XM = 2.
template <int THREADS, int NPT, bool PSD, bool SM = false>
__device__ __forceinline__ void conic_apply(Dev& d, const ConicOpView& op, bool transpose, const double* __restrict__ src,
                            double s_src, double* dst, double s_dst, int slot, double src_last, double& dst_last,
                            double& norm2) {
    const int n = op.n, m = op.m, N = n + m + 1;
    double* xs_m = cl_prod + THREADS * NPT;  // staged gather vectors (SM): m entries, then n entries
    double* xs_n = xs_m + m;
    constexpr int XM = SM ? 2 : 1;
    // (one problem per CTA: every producer of these vectors ran on this SM, so the L1-allocating cp.async sees them;
    // the copies are in flight together, each thread waits for its own and the caller's barrier publishes them)
    auto stage = [&](double* to, const double* from, int len) {
        for (int i = d.tid; i < len; i += THREADS)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(to + i)), "l"(from + i)
                         : "memory");
        asm volatile("cp.async.commit_group;\n\tcp.async.wait_all;" ::: "memory");
    };
    double acc = 0.0, dotacc = 0.0;
    if (!transpose) {
        dpi_apply<PSD>(d, op, src + n, op.wc, false);  // wc = Dpi t2
        d.sync();
        if constexpr (SM) {
            stage(xs_m, op.wc, m);
            stage(xs_n, src, n);
            __syncthreads();
        }
        conic_M_rows<THREADS, NPT, XM>(op, d.rank(), d.nblk, cl_prod, d.red, src, SM ? xs_m : op.wc, SM ? xs_n : src, src_last,
                                       s_src, dst, s_dst, acc, dotacc);
        block_partial(d, slot, acc);
        block_partial(d, slot + 1, dotacc);
        d.sync();
        const double last = -total_of(d, slot + 1) * s_src + s_dst * dst_last;  // -(c't1 + b'wc)
        dst_last = last;
        if (d.gtid == 0) dst[N - 1] = last;
        norm2 = total_of(d, slot) + last * last;
    } else {
        const double u3 = src_last;
        if constexpr (SM) {
            stage(xs_n, src, n);
            __syncthreads();
        }
        conic_Mt_A<THREADS, NPT, XM>(op, d.rank(), d.nblk, cl_prod, d.red, src, SM ? xs_n : src, u3, dotacc);
        d.sync();
        dpi_apply<PSD>(d, op, op.wc, op.wc + m, true);
        if constexpr (SM) stage(xs_m, src + n, m);   // (src is not touched by dpi_apply: no barrier needed before)
        d.sync();
        conic_Mt_rows<THREADS, NPT, XM>(op, d.rank(), d.nblk, cl_prod, d.red, src, SM ? xs_m : src + n, u3, s_src, dst, s_dst,
                                        acc, dotacc);
        block_partial(d, slot, acc);
        block_partial(d, slot + 1, dotacc);
        d.sync();
        const double last = total_of(d, slot + 1) * s_src + s_dst * dst_last;
        dst_last = last;
        if (d.gtid == 0) dst[N - 1] = last;
        norm2 = total_of(d, slot) + last * last;
    }
}

struct OpArgs {
    int kind;  // 0 csr, 1 conic
    CsrView fwd, adj;  // csr: matrix for A*v and for A'*u
    ConicOpView conic;
    int conic_trans;   // solve with M' instead of M
    int nrows, ncols;
};

// Returns ||dst||^2 (after the update).  The conic operator ends behind its own barrier; the CSR one needs a barrier
// here before its partial sums can be read.  Inlined with conic_apply: called out of line, they make the kernel copy
// its OpArgs parameter to a stack frame (600 B in the PSD build).
template <int THREADS, int NPT, bool PSD, bool SM = false>
__device__ __forceinline__ double op_apply(Dev& d, const OpArgs& o, bool adjoint, const double* src, double s_src, double* dst,
                           double s_dst, int slot, double src_last, double& dst_last) {
    if (o.kind == 0) {
        csr_apply<THREADS, NPT>(d, adjoint ? o.adj : o.fwd, src, s_src, dst, s_dst, slot);
        d.sync();
        return total_of(d, slot);
    }
    double norm2 = 0.0;
    conic_apply<THREADS, NPT, PSD, SM>(d, o.conic, adjoint != (o.conic_trans != 0), src, s_src, dst, s_dst, slot, src_last, dst_last, norm2);
    return norm2;
}

// u = b, x = v = w = 0; ||b||^2 into slot 0
__device__ __forceinline__ void lsqr_init(Dev& d, int nr, int nc, const double* __restrict__ rhs, const LsqrVectors& vec) {
    double acc = 0.0;
    for (int i = d.gtid; i < nr; i += d.gthreads) {
        const double t = rhs[i];
        vec.u[i] = t;
        acc += t * t;
    }
    for (int i = d.gtid; i < nc; i += d.gthreads) {
        vec.x[i] = 0.0;
        vec.v[i] = 0.0;
        vec.w[i] = 0.0;
    }
    block_partial(d, 0, acc);
}

// LSQR's deferred vector update: w = sv v on the first call, later x += t1 w and w = sv v + t2 w; ||w / rho||^2 into
// slot 4.  ilast >= 0: v[ilast] is read from the register copy v_last (see conic_apply).
__device__ __forceinline__ void lsqr_update(Dev& d, const LsqrScalars& s, bool first, int nc, const LsqrVectors& vec, int ilast,
                                            double v_last) {
    double *v = vec.v, *w = vec.w, *x = vec.x;
    const double sv = s.sv, t1 = s.t1, t2 = s.t2;
    double dd = 0.0;
    if (first) {
        for (int i = d.gtid; i < nc; i += d.gthreads) w[i] = sv * (i == ilast ? v_last : v[i]);
    } else {
        const double irho = 1.0 / s.rho;
        int i = d.gtid;
        for (; i + 3 * d.gthreads < nc; i += 4 * d.gthreads) {   // four independent elements in flight per thread
            double wi[4], vi[4], xi[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = i + q * d.gthreads;
                wi[q] = w[k];
                vi[q] = k == ilast ? v_last : v[k];
                xi[q] = x[k];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = i + q * d.gthreads;
                const double dk = wi[q] * irho;
                dd += dk * dk;
                x[k] = xi[q] + t1 * wi[q];
                w[k] = sv * vi[q] + t2 * wi[q];
            }
        }
        for (; i < nc; i += d.gthreads) {
            double wi = w[i];
            double dk = wi * irho;
            dd += dk * dk;
            x[i] += t1 * wi;
            w[i] = sv * (i == ilast ? v_last : v[i]) + t2 * wi;
        }
    }
    block_partial(d, 4, dd);
}

// The whole LSQR iteration (Paige-Saunders) for one operator; called by every thread of the CTAs that share the problem
// (the whole grid, one cluster, or -- batched launches -- one cluster / CTA per problem).  zero_below: right-hand sides of
// norm <= zero_below give x = 0 without iterating (ConicProgram.jl:369 tests 1e-4 on the reverse seed; -1 disables).
template <int THREADS, int NPT, bool PSD, bool SM>
__device__ void lsqr_body(Dev& d, const OpArgs& o, const double* __restrict__ rhs, const LsqrParams prm, const LsqrVectors vec,
                          const double zero_below) {
    const int nr = o.nrows, nc = o.ncols;
    double *u = vec.u, *v = vec.v;

    // private copies of the last entries of u and v (see conic_apply)
    double u_last = nr > 0 ? rhs[nr - 1] : 0.0, v_last = 0.0;
    lsqr_init(d, nr, nc, rhs, vec);
    d.sync();
    LsqrScalars s;
    const bool op1 = s.start(total_of(d, 0), zero_below);
    s.first_alpha(op1 ? op_apply<THREADS, NPT, PSD, SM>(d, o, true, u, s.su, v, 0.0, 2, u_last, v_last) : 0.0);  // v_mem = A' u_true
    bool first = true;
    bool pending = false;  // an iteration whose x/w update and stop tests are still to be applied

    if (s.arnorm != 0.0) {
        while (true) {
            // deferred vector update of the previous iteration (or w = v at start), fused with the next
            // bidiagonalisation product (conic operator: the last entry of v is read from its register copy, see conic_apply)
            lsqr_update(d, s, first, nc, vec, o.kind == 1 ? nc - 1 : -1, v_last);
            const bool more = s.itn < prm.maxiter;
            double unorm2 = 0.0;
            if (more) unorm2 = op_apply<THREADS, NPT, PSD, SM>(d, o, false, v, s.sv, u, -s.alpha * s.su, 0, v_last, u_last);  // u_mem = A v_true - alpha u_true
            else d.sync();  // the partial sums of the update above
            if (pending) {
                s.stop_tests(total_of(d, 4), prm);
                pending = false;
            }
            first = false;
            if (s.istop > 0 || !more) break;
            if (s.next_beta(unorm2))
                s.next_alpha(op_apply<THREADS, NPT, PSD, SM>(d, o, true, u, s.su, v, -s.beta * s.sv, 2, u_last, v_last));  // v_mem = A' u_true - beta v_true
            s.rotate();
            pending = true;
        }
    }
#ifdef LSQR_PROF
    if (d.gtid == 0) {
        const int n0 = g_prof_n > 400 ? 300 : 0;
        for (int k = n0; k + 1 < g_prof_n && k < n0 + 44; ++k)
            printf("%s %lld ns\n", (k & 1) ? "  compute" : "barrier", g_prof[k + 1] - g_prof[k]);
        g_prof_n = 0;
    }
#endif
    if (d.gtid == 0) s.write_stats(vec.stats);
}

template <int THREADS, int NPT, int MINB, bool CLUSTER, bool PSD>
__global__ void __launch_bounds__(THREADS, MINB) lsqr_kernel_t(OpArgs o, const double* __restrict__ rhs, LsqrParams prm,
                                                               LsqrVectors vec) {
    __shared__ double red[64];
    // (Dev built in place in the persistent kernels: from make_dev, ptxas allocates their registers worse and spills more)
    Dev d{cg::this_grid(), vec.partials, red, (int)threadIdx.x, (int)(threadIdx.x & 31), (int)(threadIdx.x >> 5),
          (int)(blockDim.x >> 5), (int)gridDim.x, (int)(blockIdx.x * blockDim.x + threadIdx.x),
          (int)(gridDim.x * blockDim.x), CLUSTER};
    lsqr_body<THREADS, NPT, PSD, false>(d, o, rhs, prm, vec, -1.0);
}

// Lock-step batch: problem p = blockIdx.x / C is solved by the C CTAs of one cluster (C = 1: one CTA, the gather vectors
// staged in shared memory); every problem has its own operator, right-hand side and work vectors.  No barrier spans
// problems: a problem that converges early simply retires its CTAs.
template <bool SM>
__global__ void __launch_bounds__(CL_THREADS, 1) lsqr_batch_kernel(const OpArgs* __restrict__ ops, const double* const* __restrict__ rhs,
                                                                   LsqrParams prm, const LsqrVectors* __restrict__ vecs, const int C,
                                                                   const double zero_below) {
    __shared__ double red[64];
    __shared__ OpArgs so;
    __shared__ LsqrVectors sv;
    const int p = blockIdx.x / C, cta = blockIdx.x - p * C;
    for (int i = threadIdx.x; i < (int)(sizeof(OpArgs) / sizeof(int)); i += blockDim.x)
        reinterpret_cast<int*>(&so)[i] = reinterpret_cast<const int*>(ops + p)[i];
    for (int i = threadIdx.x; i < (int)(sizeof(LsqrVectors) / sizeof(int)); i += blockDim.x)
        reinterpret_cast<int*>(&sv)[i] = reinterpret_cast<const int*>(vecs + p)[i];
    __syncthreads();
    Dev d{cg::this_grid(), sv.partials, red, (int)threadIdx.x, (int)(threadIdx.x & 31), (int)(threadIdx.x >> 5),
          (int)(blockDim.x >> 5), C, (int)(cta * blockDim.x + threadIdx.x), (int)(C * blockDim.x), true, cta, C == 1};
    lsqr_body<CL_THREADS, CL_NPT, false, SM>(d, so, rhs[p], prm, sv, zero_below);
}

// stand-alone operator kernels (C-ABI conic_M_apply / conic_dpi_apply; also used by tests)
__global__ void __launch_bounds__(LSQR_THREADS) conic_M_kernel(ConicOpView op, int transpose, const double* t, double* out,
                                                              double* partials) {
    __shared__ double red[64];
    Dev d = make_dev(partials, red, (int)gridDim.x);
    double last = 0.0, norm2 = 0.0;
    conic_apply<LSQR_THREADS, LSQR_NPT, true>(d, op, transpose != 0, t, 1.0, out, 0.0, 0, __ldcg(t + op.n + op.m), last, norm2);
}

__global__ void __launch_bounds__(LSQR_THREADS) conic_dpi_kernel(ConicOpView op, int transpose, const double* t, double* out,
                                                                double* partials) {
    __shared__ double red[64];
    Dev d = make_dev(partials, red, (int)gridDim.x);
    dpi_apply<true>(d, op, t, out, transpose != 0);
}


// ================================================================================================================
// Streaming LSQR for LARGE conic operators (working set beyond L2): the same iteration as lsqr_body, but every
// phase is its own kernel at full occupancy (the persistent kernel is capped at a few hundred CTAs by grid.sync and
// its register footprint, far too few loads in flight to cover HBM latency).  The LsqrScalars and the `done` flag
// live in a device struct: the host only enqueues iterations in batches and looks at the flag between batches;
// kernels of an iteration after convergence return at once.  The phases call the persistent kernel's own code
// (LsqrScalars, lsqr_init, lsqr_update, the conic row-block phases) with the same deterministic reductions (per-CTA
// partials, fixed-order sums).  No PSD cones here.
struct LsqrState {
    LsqrScalars sc;
    double op_src, op_dst;  // scalars of the operator application in flight: dst = op_src * OP(src) + op_dst * dst
    int first, pending, done, more, do_op1;
};

constexpr int ST_THREADS = 256;

__device__ double st_total(const double* partials, int slot, int stride, int count, double* red) {
    // fixed-order sum of `count` CTA partials by one 256-thread block
    double s = 0.0;
    for (int i = threadIdx.x; i < count; i += blockDim.x) s += partials[slot * stride + i];
    s = warp_sum_all(s);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    __syncthreads();
    return t;
}

// three totals in one pass (independent loads, one shared-memory exchange): the single-CTA scalar kernels are pure
// latency, three sequential st_total calls were most of it
__device__ void st_total3(const double* partials, int stride, int s0, int c0, int s1, int c1, int s2, int c2, double* red,
                          double& t0, double& t1, double& t2) {
    double a = 0.0, b = 0.0, c = 0.0;
    const int cmax = max(c0, max(c1, c2));
    for (int i = threadIdx.x; i < cmax; i += blockDim.x) {
        const double x0 = i < c0 ? partials[s0 * stride + i] : 0.0;
        const double x1 = i < c1 ? partials[s1 * stride + i] : 0.0;
        const double x2 = i < c2 ? partials[s2 * stride + i] : 0.0;
        a += x0;
        b += x1;
        c += x2;
    }
    a = warp_sum_all(a);
    b = warp_sum_all(b);
    c = warp_sum_all(c);
    const int nw = blockDim.x >> 5, w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        red[w] = a;
        red[8 + w] = b;
        red[16 + w] = c;
    }
    __syncthreads();
    t0 = t1 = t2 = 0.0;
    for (int k = 0; k < nw; ++k) {
        t0 += red[k];
        t1 += red[8 + k];
        t2 += red[16 + k];
    }
}

__global__ void __launch_bounds__(ST_THREADS) st_init_kernel(int nr, int nc, const double* __restrict__ rhs, LsqrVectors vec) {
    __shared__ double red[64];
    Dev d = make_dev(vec.partials, red, ST_STRIDE);
    lsqr_init(d, nr, nc, rhs, vec);
}

// after st_init_kernel: beta, su; sets up v = A' u (op1 with s_dst = 0)
__global__ void __launch_bounds__(ST_THREADS) st_init_fin_kernel(LsqrVectors vec, int stride, int cnt0, LsqrState* S) {
    __shared__ double red[64];
    const double t0 = st_total(vec.partials, 0, stride, cnt0, red);
    if (threadIdx.x == 0) {
        LsqrState s{};
        s.do_op1 = s.sc.start(t0, -1.0);
        s.op_src = s.sc.su;
        s.op_dst = 0.0;
        s.first = 1;
        *S = s;
    }
}

// x, w update of the previous iteration (LSQR's deferred vector update), ||w / rho||^2 into slot 4
__global__ void __launch_bounds__(ST_THREADS) st_update_kernel(int nc, LsqrVectors vec, LsqrState* S) {
    if (S->done) return;
    __shared__ double red[64];
    Dev d = make_dev(vec.partials, red, ST_STRIDE);
    const LsqrScalars s = S->sc;
    lsqr_update(d, s, S->first, nc, vec, -1, 0.0);
}

// ---- M src (non-transposed), phase 1: wc = Dpi src2
__global__ void __launch_bounds__(ST_THREADS) st_dpi_kernel(ConicOpView op, const double* __restrict__ y, double* out, int transpose,
                                                            const LsqrState* S, int which) {
    if (S->done || (which == 0 ? !S->more : !S->do_op1)) return;
    __shared__ double red[64];
    Dev d = make_dev(nullptr, red, ST_STRIDE);
    dpi_apply<false>(d, op, y, out, transpose != 0);
}

// ---- M src, phase 2: both sparse products, dst updated in place; slots 0 (norm) and 1 (last-row dot)
__global__ void __launch_bounds__(SP_THREADS, 8) st_M_rows_kernel(ConicOpView op, const double* __restrict__ src, double* dst, double* partials,
                                                               const LsqrState* S) {
    if (S->done || !S->more) return;
    __shared__ double red[64], prod[ST_CHUNK];
    Dev d = make_dev(partials, red, ST_STRIDE);
    double acc = 0.0, dotacc = 0.0;
    conic_M_rows<SP_THREADS, ST_NPT, 0>(op, (int)blockIdx.x, (int)gridDim.x, prod, red, src, op.wc, src, __ldcg(src + op.n + op.m),
                                        S->op_src, dst, S->op_dst, acc, dotacc);
    block_partial(d, 0, acc);
    block_partial(d, 1, dotacc);
}

// ---- after M v: last row of u, pending stop tests, beta, scalars of the transposed application
__global__ void __launch_bounds__(ST_THREADS) st_mid_kernel(int N, LsqrVectors vec, int stride, int cnt_rows, int cnt_upd, LsqrParams prm,
                                                            LsqrState* S) {
    if (S->done) return;
    __shared__ double red[64];
    double tot0, tot1, tot4;
    st_total3(vec.partials, stride, 0, cnt_rows, 1, cnt_rows, 4, cnt_upd, red, tot0, tot1, tot4);
    if (threadIdx.x != 0) return;
    LsqrState s = *S;
    double unorm2 = tot0;
    if (s.more) {
        const double last = -tot1 * s.op_src + s.op_dst * vec.u[N - 1];
        vec.u[N - 1] = last;
        unorm2 += last * last;
    }
    if (s.pending) {
        s.sc.stop_tests(tot4, prm);
        s.pending = 0;
    }
    s.first = 0;
    if (s.sc.istop > 0 || !s.more) {
        s.done = 1;
        *S = s;
        return;
    }
    s.do_op1 = s.sc.next_beta(unorm2);
    if (s.do_op1) {
        s.op_src = s.sc.su;
        s.op_dst = -s.sc.beta * s.sc.sv;
    }
    *S = s;
}

// ---- M' src, phase 1: wc = A src1 - src2 - b src3 ; slot 3 = b . src2
__global__ void __launch_bounds__(SP_THREADS, 8) st_Mt_A_kernel(ConicOpView op, const double* __restrict__ src, double* partials,
                                                             const LsqrState* S) {
    if (S->done || !S->do_op1) return;
    __shared__ double red[64], prod[ST_CHUNK];
    Dev d = make_dev(partials, red, ST_STRIDE);
    double dotacc = 0.0;
    conic_Mt_A<SP_THREADS, ST_NPT, 0>(op, (int)blockIdx.x, (int)gridDim.x, prod, red, src, src, __ldcg(src + op.n + op.m), dotacc);
    block_partial(d, 3, dotacc);
}

// ---- M' src, phase 3 (after Dpi' wc -> r2): rows of A' and the elementwise block; slots 2 (norm) and 5 (c . src1)
__global__ void __launch_bounds__(SP_THREADS, 8) st_Mt_rows_kernel(ConicOpView op, const double* __restrict__ src, double* dst, double* partials,
                                                                const LsqrState* S) {
    if (S->done || !S->do_op1) return;
    __shared__ double red[64], prod[ST_CHUNK];
    Dev d = make_dev(partials, red, ST_STRIDE);
    double acc = 0.0, dotacc = 0.0;
    conic_Mt_rows<SP_THREADS, ST_NPT, 0>(op, (int)blockIdx.x, (int)gridDim.x, prod, red, src, src + op.n, __ldcg(src + op.n + op.m),
                                         S->op_src, dst, S->op_dst, acc, dotacc);
    block_partial(d, 2, acc);
    block_partial(d, 5, dotacc);
}

// ---- after M' u: last row of v, alpha, plane rotations (or, at start-up, the initial scalars)
__global__ void __launch_bounds__(ST_THREADS) st_end_kernel(int N, LsqrVectors vec, int stride, int cnt_a, int cnt_rows, LsqrParams prm,
                                                            LsqrState* S, int startup) {
    if (S->done) return;
    __shared__ double red[64];
    double tot2, tot3, tot5;
    st_total3(vec.partials, stride, 2, cnt_rows, 3, cnt_a, 5, cnt_rows, red, tot2, tot3, tot5);
    if (threadIdx.x != 0) return;
    LsqrState s = *S;
    double alpha2 = 0.0;
    if (s.do_op1) {
        const double last = (tot3 + tot5) * s.op_src + s.op_dst * vec.v[N - 1];
        vec.v[N - 1] = last;
        alpha2 = tot2 + last * last;
    }
    if (startup) {
        s.sc.first_alpha(alpha2);
        if (s.sc.arnorm == 0.0) s.done = 1;
    } else {
        if (s.do_op1) s.sc.next_alpha(alpha2);
        s.sc.rotate();
        s.pending = 1;
    }
    s.more = s.sc.itn < prm.maxiter ? 1 : 0;
    s.op_src = s.sc.sv;
    s.op_dst = -s.sc.alpha * s.sc.su;
    *S = s;
}

__global__ void st_stats_kernel(const LsqrState* S, double* stats) { S->sc.write_stats(stats); }

// ================================================================================================================
// Multi-right-hand-side LSQR (diffopt_b200_conic_forward_multi / _reverse_multi): KB right-hand sides against the SAME
// conic operator M advance in lock-step in one persistent kernel.  Everything but the vectors is shared: one pass over
// (val, colind) of A and A' per phase serves all KB directions, and the vectors are stored interleaved ([row][KB]), so
// one gathered sector carries the values of several directions.  Per direction the arithmetic is that of lsqr_body
// (the same LsqrScalars methods in the same order, fixed-order reductions), and no value of one direction depends on
// another's: direction j gives the same bits whatever the other directions of its group hold.  A direction whose stop
// test fired, or whose right-hand side failed the zero test, is frozen (its x and statistics are final, its vectors are
// no longer written); the group ends when every direction is frozen.
// Shape: 256-thread CTAs (the PSD GEMM phases are written for them) on the blk / t_blk row blocks (<= ST_CHUNK nonzeros,
// <= SP_THREADS rows, or one longer row), KB products per nonzero parked in shared memory.
constexpr int MR_THREADS = LSQR_THREADS;
constexpr int MR_NPT = LSQR_NPT;
constexpr int MR_PLD = ST_CHUNK + 1;  // products of direction j at prod[j * MR_PLD ..] (odd stride: row sums of the
                                      // directions of one row fall into different banks)

// Work of one group of KB directions against an operator of order N = n + m + 1 (offsets in doubles, all multiples of KB):
// u, v, w (N KB each) | wc (2 m KB: Dpi t2 / r and Dpi' r) | PSD scratch W1, W2 (sumd2 KB each) | partial sums
// (LSQR_NSLOTS KB ctas).
struct MultiArgs {
    ConicOpView op;            // row blocks blk / t_blk; op.wc and op.psd_w* are unused (per group, in `work`)
    const double* rhs;         // [group][N][KB]
    const double* rhs_norm2;   // [group][KB] squared norms of the right-hand sides (zero test)
    double zero_below;         // a direction whose right-hand side has norm <= zero_below is not iterated
    double* x;                 // [group][N][KB] solutions
    double* stats;             // [group][KB][4] istop, itn, rnorm, arnorm
    double* work;              // one region of `work_stride` doubles per group running concurrently
    size_t work_stride;
    long long sumd2;
    int group0;                // first group of the launch
    int ctas;                  // CTAs per group (cluster route; the cooperative route uses the whole grid)
};

template <int KB>
__device__ __forceinline__ void mr_block_partial(Dev& d, int slot, double v) {
    // thread t accumulates for direction t % KB: lanes of one direction are KB apart
#pragma unroll
    for (int o = 16; o >= KB; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (d.lane < KB) d.red[d.warp * KB + d.lane] = v;
    __syncthreads();
    if (d.tid < KB) {
        double s = 0.0;
        for (int w = 0; w < d.nwarp; ++w) s += d.red[w * KB + d.tid];
        d.partials[(size_t)(slot * KB + d.tid) * d.nblk + d.rank()] = s;
    }
    __syncthreads();
}

// after a barrier: fixed-order sum of the CTA partials of (slot, direction j), identical in every CTA
template <int KB>
__device__ __forceinline__ double mr_total(const Dev& d, int slot, int j) {
    const double* p = d.partials + (size_t)(slot * KB + j) * d.nblk;
    double s = 0.0;
    for (int i = 0; i < d.nblk; ++i) s += __ldcg(p + i);
    return s;
}

// Row-block SpMM: spmv_stream for KB interleaved vectors.  Each (val, colind) is loaded once and KB contiguous values are
// gathered with 16-byte loads; every row is summed per direction in storage order by one thread (direction j = thread
// index % KB).  pre(b, row) / epi(b, row, t, operands) see the direction of the calling thread.
template <int KB, class Sel, class Pre, class Epi>
__device__ __forceinline__ void spmm_stream(int cta, int ncta, int nblk_total, double* prod, double* red, Sel&& sel, Pre&& pre,
                                            Epi&& epi) {
    constexpr int THREADS = MR_THREADS, NPT = MR_NPT, CHUNK = THREADS * NPT, KH = KB / 2;
    const int tid = threadIdx.x;
    const int per = (nblk_total + ncta - 1) / ncta;
    const int b_end = min(nblk_total, (cta + 1) * per);
    for (int b = cta * per; b < b_end; ++b) {
        const CsrView* A;
        const double* x;
        int lb;
        sel(b, A, x, lb);
        const int2 d0 = __ldg(reinterpret_cast<const int2*>(A->blk) + lb);
        const int2 d1 = __ldg(reinterpret_cast<const int2*>(A->blk) + lb + 1);
        const int r0 = d0.x, s = d0.y, r1 = d1.x, cnt = d1.y - d0.y;
        if (cnt > CHUNK) {  // one long row: whole CTA, fixed-order reduction per direction
            double acc[KB];
#pragma unroll
            for (int j = 0; j < KB; ++j) acc[j] = 0.0;
            for (int k = tid; k < cnt; k += THREADS) {
                const double a = __ldg(A->val + s + k);
                const double2* xp = reinterpret_cast<const double2*>(x + (size_t)__ldg(A->colind + s + k) * KB);
#pragma unroll
                for (int q = 0; q < KH; ++q) {
                    const double2 xv = __ldcg(xp + q);
                    acc[2 * q] = fma(a, xv.x, acc[2 * q]);
                    acc[2 * q + 1] = fma(a, xv.y, acc[2 * q + 1]);
                }
            }
#pragma unroll
            for (int j = 0; j < KB; ++j) {
                const double t = warp_sum_all(acc[j]);
                if ((tid & 31) == 0) red[(tid >> 5) * KB + j] = t;
            }
            __syncthreads();
            if (tid < KB) {
                double t = 0.0;
                for (int w = 0; w < THREADS / 32; ++w) t += red[w * KB + tid];
                epi(b, r0, t, pre(b, r0));
            }
        } else {
            double av[NPT];
            int ci[NPT];
#pragma unroll
            for (int u = 0; u < NPT; ++u) {
                const int k = tid + u * THREADS;
                av[u] = 0.0;
                ci[u] = 0;
                if (k < cnt) {
                    av[u] = __ldg(A->val + s + k);
                    ci[u] = __ldg(A->colind + s + k);
                }
            }
            double2 xv[NPT][KH];
#pragma unroll
            for (int u = 0; u < NPT; ++u) {
                const double2* xp = reinterpret_cast<const double2*>(x + (size_t)ci[u] * KB);
#pragma unroll
                for (int q = 0; q < KH; ++q) xv[u][q] = tid + u * THREADS < cnt ? __ldcg(xp + q) : make_double2(0.0, 0.0);
            }
#pragma unroll
            for (int u = 0; u < NPT; ++u) {
                const int k = tid + u * THREADS;
                if (k < cnt) {
#pragma unroll
                    for (int q = 0; q < KH; ++q) {
                        prod[(2 * q) * MR_PLD + k] = av[u] * xv[u][q].x;
                        prod[(2 * q + 1) * MR_PLD + k] = av[u] * xv[u][q].y;
                    }
                }
            }
            __syncthreads();
            const int nrow = r1 - r0;
            for (int it = tid; it < nrow * KB; it += THREADS) {
                const int row = r0 + it / KB;
                const double* pj = prod + (it % KB) * MR_PLD;
                const int ra = __ldg(A->rowptr + row) - s, rb = __ldg(A->rowptr + row + 1) - s;
                const double4 o = pre(b, row);
                double t = 0.0;
                for (int k = ra; k < rb; ++k) t += pj[k];
                epi(b, row, t, o);
            }
        }
        __syncthreads();  // prod / red are free again
    }
}

// soc_apply for direction j of interleaved vectors
template <int KB>
__device__ void soc_apply_multi(const ConicOpView& op, int c, int j, bool valid, const double* __restrict__ y, double* out,
                                int lig, int T) {
    int off = 0, dim = 0, cs = 0;
    double nx = 1.0, t = 0.0;
    if (valid) {
        off = op.soc_off[c];
        dim = op.soc_dim[c];
        cs = op.soc_case[c];
        nx = op.soc_nx[c];
        t = op.v[off];
    }
    auto at = [&](int k) { return (size_t)(off + k) * KB + j; };
    double xy = 0.0;
    if (valid && cs == 2)
        for (int k = 1 + lig; k < dim; k += T) xy += op.v[off + k] * __ldcg(y + at(k));
    for (int o = T >> 1; o > 0; o >>= 1) xy += __shfl_xor_sync(0xffffffffu, xy, o);
    if (!valid) return;
    if (cs == 0) {
        for (int k = lig; k < dim; k += T) out[at(k)] = __ldcg(y + at(k));
    } else if (cs == 1) {
        for (int k = lig; k < dim; k += T) out[at(k)] = 0.0;
    } else {
        const double y0 = __ldcg(y + at(0));
        const double inv2 = 1.0 / (2.0 * nx);
        const double coef = t / (nx * nx) * xy;
        for (int k = lig; k < dim; k += T) {
            double r;
            if (k == 0)
                r = nx * y0 + xy;
            else {
                double xk = op.v[off + k];
                r = xk * y0 + (nx + t) * __ldcg(y + at(k)) - coef * xk;
            }
            out[at(k)] = r * inv2;
        }
    }
}

// psd_apply_all for KB interleaved vectors: one flattened tile list over (direction, cone), so the four GEMM phases of
// every direction share the three barriers; W1, W2 of direction j at w1 / w2 + j * sumd2
template <int KB>
__device__ void psd_apply_multi(Dev& d, const ConicOpView& op, const double* __restrict__ y, double* out, bool transpose,
                                double* w1, double* w2, long long sumd2) {
    if (op.npsd == 0) return;
    __shared__ double As[PT * PLD], Bs[PT * PLD];
    const double dscale = transpose ? 1.0 : 2.0, oscale = transpose ? 1.0 : 0.5;
    const int ntot = op.psd_ntiles * KB;
    for (int phase = 0; phase < 4; ++phase) {
        for (int tt = blockIdx.x; tt < ntot; tt += gridDim.x) {
            const int j = tt / op.psd_ntiles, t = tt - j * op.psd_ntiles;
            int lo = 0, hi = op.npsd - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (__ldg(op.psd_toff + mid) <= t) lo = mid; else hi = mid - 1;
            }
            const int c = lo, dd = op.psd_d[c], off = op.psd_off[c];
            const int nt = (dd + PT - 1) / PT, lt = t - __ldg(op.psd_toff + c);
            const int i0 = (lt % nt) * PT, j0 = (lt / nt) * PT;
            const long long uo = op.psd_uoff[c];
            const double* U = op.psd_U + uo;
            double* W1 = w1 + j * sumd2 + uo;
            double* W2 = w2 + j * sumd2 + uo;
            auto tri = [&](int r, int cc) { return (size_t)(off + (long long)cc * (cc + 1) / 2 + r) * KB + j; };
            if (op.psd_ident[c]) {
                if (phase == 3)
                    for (int e = threadIdx.x; e < PT * PT; e += blockDim.x) {
                        const int i = i0 + e % PT, jj = j0 + e / PT;
                        if (i <= jj && jj < dd) out[tri(i, jj)] = __ldcg(y + tri(i, jj));
                    }
                continue;
            }
            if (phase == 0) {
                psd_tile_gemm(dd, i0, j0, false, true, As, Bs,
                    [&](int i, int k) { return U[k + (long long)i * dd]; },
                    [&](int k, int jj) {
                        const int r = k < jj ? k : jj, cc = k < jj ? jj : k;
                        const double v = __ldcg(y + tri(r, cc));
                        return k == jj ? v * dscale : v;
                    },
                    [&](int i, int jj, double v) { W1[i + (long long)jj * dd] = v; });
            } else if (phase == 1) {
                const double* Bm = op.psd_Bm + uo;
                psd_tile_gemm(dd, i0, j0, true, true, As, Bs,
                    [&](int i, int k) { return __ldcg(W1 + i + (long long)k * dd); },
                    [&](int k, int jj) { return U[k + (long long)jj * dd]; },
                    [&](int i, int jj, double v) { W2[i + (long long)jj * dd] = v * Bm[i + (long long)jj * dd]; });
            } else if (phase == 2) {
                psd_tile_gemm(dd, i0, j0, true, true, As, Bs,
                    [&](int i, int k) { return U[i + (long long)k * dd]; },
                    [&](int k, int jj) { return __ldcg(W2 + k + (long long)jj * dd); },
                    [&](int i, int jj, double v) { W1[i + (long long)jj * dd] = v; });
            } else if (i0 <= j0 + PT - 1) {
                psd_tile_gemm(dd, i0, j0, true, false, As, Bs,
                    [&](int i, int k) { return __ldcg(W1 + i + (long long)k * dd); },
                    [&](int k, int jj) { return U[jj + (long long)k * dd]; },
                    [&](int i, int jj, double v) {
                        if (i <= jj) out[tri(i, jj)] = i == jj ? v * oscale : v;
                    });
            }
        }
        if (phase < 3) d.sync();
    }
}

// dpi_apply for KB interleaved vectors (diagonal and 3 x 3 block rows: one thread per row and direction; SOC: 8 lanes per
// cone and direction; PSD: psd_apply_multi)
template <int KB, bool PSD>
__device__ __forceinline__ void dpi_apply_multi(Dev& d, const ConicOpView& op, const double* __restrict__ y, double* out,
                                                bool transpose, double* w1, double* w2, long long sumd2) {
    for (int e = d.gtid; e < op.m * KB; e += d.gthreads) {
        const int i = e / KB;
        const int k = op.kind[i];
        if (k == 0) {
            out[e] = op.diag[i] * __ldcg(y + e);
        } else if (k >= 4) {
            const double* br = op.blk3 + 3 * (long long)i;
            const double* yc = y + (e - (k - 4) * KB);
            out[e] = br[0] * __ldcg(yc) + br[1] * __ldcg(yc + KB) + br[2] * __ldcg(yc + 2 * KB);
        }
    }
    {
        const int T = 8;
        const int lig = d.lane & (T - 1);
        const int ngroups = d.gthreads / T;
        const int g = d.gtid / T;
        const int npair = op.nsoc * KB;
        for (int base = 0; base < npair; base += ngroups) {
            const int p = base + g;
            soc_apply_multi<KB>(op, p / KB, p % KB, p < npair, y, out, lig, T);
        }
    }
    if constexpr (PSD) psd_apply_multi<KB>(d, op, y, out, transpose, w1, w2, sumd2);
}

// Per-direction scalars of one operator application, read by every thread for its direction t % KB
struct MrScal {
    double s_src, s_dst, src_last;
    int write;  // 0: the direction's dst is not written (frozen, or beta = 0 before an M' application)
};

// dst = s_src * OP(src) + s_dst * dst for the KB directions (OP = M, or M' when `transpose`); partial sums of ||dst||^2
// (without the last row) into `slot`, of the last-row dot product into slot + 1; ends behind a barrier.
template <int KB, bool PSD>
__device__ __forceinline__ void conic_apply_multi(Dev& d, const ConicOpView& op, bool transpose, const double* __restrict__ src,
                                                  double* dst, const MrScal& sc, int slot, double* wc, double* w1, double* w2,
                                                  long long sumd2) {
    const int n = op.n, m = op.m;
    const double ss = sc.s_src, sd = sc.s_dst, t3 = sc.src_last;
    const bool wr = sc.write != 0;
    const int j = d.tid % KB;
    double acc = 0.0, dot = 0.0;
    auto at = [&](int row) { return (size_t)row * KB + j; };
    if (!transpose) {
        dpi_apply_multi<KB, PSD>(d, op, src + (size_t)n * KB, wc, false, w1, w2, sumd2);  // wc = Dpi t2
        d.sync();
        const int nbt = op.At.nblk;
        spmm_stream<KB>(
            d.rank(), d.nblk, nbt + op.A.nblk, cl_prod, d.red,
            [&](int b, const CsrView*& A, const double*& x, int& lb) {
                if (b < nbt) { A = &op.At; x = wc; lb = b; }
                else { A = &op.A; x = src; lb = b - nbt; }
            },
            [&](int b, int row) {
                return b < nbt ? make_double4(op.c[row], __ldcg(dst + at(row)), __ldcg(src + at(row)), 0.0)
                               : make_double4(__ldcg(wc + at(row)), __ldcg(src + at(n + row)), op.b[row], __ldcg(dst + at(n + row)));
            },
            [&](int b, int row, double t, const double4& o) {
                if (b < nbt) {
                    t = (t + o.x * t3) * ss + sd * o.y;
                    if (wr) dst[at(row)] = t;
                    acc += t * t;
                    dot += o.x * o.z;
                } else {
                    t = (-t + o.y - o.x + o.z * t3) * ss + sd * o.w;
                    if (wr) dst[at(n + row)] = t;
                    acc += t * t;
                    dot += o.z * o.x;
                }
            });
    } else {
        spmm_stream<KB>(   // wc = A u1 - u2 - b u3
            d.rank(), d.nblk, op.A.nblk, cl_prod, d.red,
            [&](int b, const CsrView*& A, const double*& x, int& lb) { A = &op.A; x = src; lb = b; },
            [&](int, int row) { return make_double4(__ldcg(src + at(n + row)), op.b[row], 0.0, 0.0); },
            [&](int, int row, double t, const double4& o) {
                wc[at(row)] = t - o.x - o.y * t3;
                dot += o.y * o.x;
            });
        d.sync();
        double* r2 = wc + (size_t)m * KB;
        dpi_apply_multi<KB, PSD>(d, op, wc, r2, true, w1, w2, sumd2);
        d.sync();
        const double* src2 = src + (size_t)n * KB;
        spmm_stream<KB>(
            d.rank(), d.nblk, op.At.nblk, cl_prod, d.red,
            [&](int b, const CsrView*& A, const double*& x, int& lb) { A = &op.At; x = src2; lb = b; },
            [&](int, int row) { return make_double4(op.c[row], __ldcg(dst + at(row)), __ldcg(src + at(row)), 0.0); },
            [&](int, int row, double t, const double4& o) {
                t = (-t - o.x * t3) * ss + sd * o.y;
                if (wr) dst[at(row)] = t;
                acc += t * t;
                dot += o.x * o.z;
            });
        for (int e = d.rank() * MR_THREADS + d.tid; e < m * KB; e += d.nblk * MR_THREADS) {
            const double t = (__ldcg(r2 + e) + __ldcg(src2 + e)) * ss + sd * __ldcg(dst + (size_t)n * KB + e);
            if (wr) dst[(size_t)n * KB + e] = t;
            acc += t * t;
        }
    }
    mr_block_partial<KB>(d, slot, acc);
    mr_block_partial<KB>(d, slot + 1, dot);
    d.sync();
}

// The LSQR iteration of lsqr_body for the KB directions of group g.
template <int KB, bool CLUSTER>
__global__ void __launch_bounds__(MR_THREADS, 2) lsqr_multi_kernel(MultiArgs a, LsqrParams prm) {
    constexpr bool PSD = !CLUSTER;  // problems with PSD cones take the cooperative route
    __shared__ double red[(MR_THREADS / 32) * KB];
    __shared__ LsqrScalars sc[KB];
    __shared__ MrScal fw[KB], bw[KB];   // scalars of the next M v / M' u application
    __shared__ double ulast[KB], vlast[KB];  // last entries of u and v (never read from memory, see conic_apply)
    __shared__ int active[KB];
    const ConicOpView& op = a.op;
    const int n = op.n, m = op.m, N = n + m + 1;
    const int slot = CLUSTER ? (int)blockIdx.x / a.ctas : 0;
    const int g = a.group0 + slot;
    const int C = CLUSTER ? a.ctas : (int)gridDim.x;
    const int cta = CLUSTER ? (int)blockIdx.x - slot * a.ctas : (int)blockIdx.x;
    double* u = a.work + (size_t)slot * a.work_stride;
    double* v = u + (size_t)N * KB;
    double* w = v + (size_t)N * KB;
    double* wc = w + (size_t)N * KB;
    double* w1 = wc + (size_t)2 * m * KB;
    double* w2 = w1 + (size_t)a.sumd2 * KB;
    double* partials = w2 + (size_t)a.sumd2 * KB;
    const double* rhs = a.rhs + (size_t)g * N * KB;
    double* x = a.x + (size_t)g * N * KB;
    double* stats = a.stats + (size_t)g * KB * 4;
    Dev d{cg::this_grid(), partials, red, (int)threadIdx.x, (int)(threadIdx.x & 31), (int)(threadIdx.x >> 5),
          (int)(blockDim.x >> 5), C, cta * MR_THREADS + (int)threadIdx.x, C * MR_THREADS, CLUSTER, CLUSTER ? cta : -1, false};
    const int NK = N * KB;
    const int jt = d.tid % KB;  // this thread's direction in every element-wise loop and row epilogue
    auto freeze = [&](int j) {  // by thread j of every CTA
        active[j] = 0;
        bw[j].write = 0;
        if (d.rank() == 0) {
            stats[j * 4 + 0] = (double)sc[j].istop;
            stats[j * 4 + 1] = (double)sc[j].itn;
            stats[j * 4 + 2] = sc[j].rnorm;
            stats[j * 4 + 3] = sc[j].arnorm;
        }
    };

    double acc = 0.0;  // u = b, x = v = w = 0
    for (int e = d.gtid; e < NK; e += d.gthreads) {
        const double t = rhs[e];
        u[e] = t;
        acc += t * t;
        x[e] = 0.0;
        v[e] = 0.0;
        w[e] = 0.0;
    }
    mr_block_partial<KB>(d, 0, acc);
    d.sync();
    if (d.tid < KB) {
        const int j = d.tid;
        const bool zero = sqrt(a.rhs_norm2[(size_t)g * KB + j]) <= a.zero_below;
        ulast[j] = rhs[(size_t)(N - 1) * KB + j];
        vlast[j] = 0.0;
        const bool op1 = sc[j].start(zero ? 0.0 : mr_total<KB>(d, 0, j), -1.0);
        bw[j] = MrScal{sc[j].su, 0.0, ulast[j], op1 ? 1 : 0};
    }
    __syncthreads();
    bool any = false;
    for (int j = 0; j < KB; ++j) any |= bw[j].write != 0;
    if (any) conic_apply_multi<KB, PSD>(d, op, true, u, v, bw[jt], 2, wc, w1, w2, a.sumd2);  // v_mem = M' u_true
    if (d.tid < KB) {
        const int j = d.tid;
        double a2 = 0.0;
        if (bw[j].write) {
            const double last = mr_total<KB>(d, 3, j) * bw[j].s_src;
            vlast[j] = last;
            a2 = mr_total<KB>(d, 2, j) + last * last;
        }
        sc[j].first_alpha(a2);
        active[j] = 1;
        if (sc[j].arnorm == 0.0) freeze(j);
        fw[j] = MrScal{sc[j].sv, -sc[j].alpha * sc[j].su, vlast[j], active[j]};
    }
    bool first = true;
    long long itn = 0;
    while (true) {
        __syncthreads();
        any = false;
        for (int j = 0; j < KB; ++j) any |= active[j] != 0;
        if (!any) break;
        {   // deferred x / w update of the active directions (w = sv v at start); ||w / rho||^2 into slot 4
            const bool act = active[jt] != 0;
            const double svj = sc[jt].sv, t1 = sc[jt].t1, t2 = sc[jt].t2, irho = 1.0 / sc[jt].rho;
            const double vl = vlast[jt];
            double dd = 0.0;
            if (act) {
                for (int e = d.gtid; e < NK; e += d.gthreads) {
                    const double ve = e >= NK - KB ? vl : v[e];
                    if (first) {
                        w[e] = svj * ve;
                    } else {
                        const double wi = w[e];
                        const double dk = wi * irho;
                        dd += dk * dk;
                        x[e] += t1 * wi;
                        w[e] = svj * ve + t2 * wi;
                    }
                }
            }
            mr_block_partial<KB>(d, 4, dd);
        }
        const bool more = itn < prm.maxiter;
        if (more) conic_apply_multi<KB, PSD>(d, op, false, v, u, fw[jt], 0, wc, w1, w2, a.sumd2);  // u = M v_true - alpha u_true
        else d.sync();
        if (d.tid < KB && active[d.tid]) {
            const int j = d.tid;
            double unorm2 = 0.0;
            if (more) {
                const double last = -mr_total<KB>(d, 1, j) * fw[j].s_src + fw[j].s_dst * ulast[j];
                ulast[j] = last;
                unorm2 = mr_total<KB>(d, 0, j) + last * last;
            }
            if (!first) sc[j].stop_tests(mr_total<KB>(d, 4, j), prm);
            if (sc[j].istop > 0 || !more) {
                freeze(j);
            } else {
                const bool op1 = sc[j].next_beta(unorm2);
                bw[j] = MrScal{sc[j].su, -sc[j].beta * sc[j].sv, ulast[j], op1 ? 1 : 0};
            }
        }
        first = false;
        __syncthreads();
        any = false;
        bool live = false;
        for (int j = 0; j < KB; ++j) {
            any |= bw[j].write != 0 && active[j] != 0;
            live |= active[j] != 0;
        }
        if (!live) break;
        if (any) conic_apply_multi<KB, PSD>(d, op, true, u, v, bw[jt], 2, wc, w1, w2, a.sumd2);  // v = M' u_true - beta v_true
        if (d.tid < KB && active[d.tid]) {
            const int j = d.tid;
            if (bw[j].write) {
                const double last = mr_total<KB>(d, 3, j) * bw[j].s_src + bw[j].s_dst * vlast[j];
                vlast[j] = last;
                sc[j].next_alpha(mr_total<KB>(d, 2, j) + last * last);
            }
            sc[j].rotate();
            fw[j] = MrScal{sc[j].sv, -sc[j].alpha * sc[j].su, vlast[j], 1};
        }
        ++itn;
    }
}

CsrView view_of(const DevBuf& rp, const DevBuf& ci, const DevBuf& v, int64_t nrows, int64_t ncols,
                const DevBuf* blk = nullptr, int64_t nblk = 0, const DevBuf* sval = nullptr, const DevBuf* scol = nullptr,
                const DevBuf* spos = nullptr) {
    return CsrView{(int)nrows, (int)ncols, rp.as<int>(), ci.as<int>(), v.as<double>(),
                   blk ? blk->as<int>() : nullptr, (int)nblk,
                   sval ? sval->as<double>() : nullptr, scol ? scol->as<int>() : nullptr,
                   spos ? spos->as<unsigned short>() : nullptr};
}

}  // namespace

ConicOpView conic_view(diffopt_b200_ctx* ctx, bool stream_blocks = false) {
    ConicState& s = ctx->conic;
    ConicOpView o{};
    o.n = (int)s.n;
    o.m = (int)s.m;
    if (stream_blocks) {
        const bool so = s.A.sorted;
        o.A = view_of(s.A.rowptr, s.A.colind, s.A.val, s.m, s.n, &s.A.blk, s.A.nblk, so ? &s.A.sval : nullptr,
                      so ? &s.A.scol : nullptr, so ? &s.A.spos : nullptr);
        o.At = view_of(s.A.t_rowptr, s.A.t_colind, s.A.t_val, s.n, s.m, &s.A.t_blk, s.A.t_nblk, so ? &s.A.t_sval : nullptr,
                       so ? &s.A.t_scol : nullptr, so ? &s.A.t_spos : nullptr);
    } else {
        o.A = view_of(s.A.rowptr, s.A.colind, s.A.val, s.m, s.n, &s.A.cblk, s.A.ncblk);
        o.At = view_of(s.A.t_rowptr, s.A.t_colind, s.A.t_val, s.n, s.m, &s.A.t_cblk, s.A.t_ncblk);
    }
    o.b = s.b.as<double>();
    o.c = s.c.as<double>();
    o.diag = s.nn_scale.as<double>();
    o.kind = s.row_kind.as<signed char>();
    o.blk3 = s.blk3.as<double>();
    o.nsoc = (int)s.nsoc;
    o.soc_off = s.soc_off.as<int>();
    o.soc_dim = s.soc_dim.as<int>();
    o.soc_case = s.soc_case.as<int>();
    o.soc_nx = s.soc_nx.as<double>();
    o.v = s.v.as<double>();
    o.npsd = (int)s.npsd;
    o.psd_off = s.psd_off.as<int>();
    o.psd_d = s.psd_d.as<int>();
    o.psd_uoff = s.psd_uoff.as<long long>();
    o.psd_U = s.psd_U.as<double>();
    o.psd_Bm = s.psd_Bm.as<double>();
    o.psd_ident = s.psd_ident.as<int>();
    o.psd_toff = s.psd_toff.as<int>();
    o.psd_ntiles = (int)s.psd_ntiles;
    o.psd_w0 = s.psd_work.as<double>();
    o.psd_w1 = o.psd_w0 + s.psd_sumd2;
    o.psd_w2 = o.psd_w1 + s.psd_sumd2;
    o.wc = s.w1.as<double>();
    return o;
}

static int coop_grid(diffopt_b200_ctx* ctx, const void* kernel, size_t dyn, int64_t work) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, LSQR_THREADS, dyn);
    if (per_sm < 1) per_sm = 1;
    int64_t want = (work + LSQR_THREADS * 4 - 1) / (LSQR_THREADS * 4);
    // small problems: one CTA per SM keeps grid.sync cheap; large ones (beyond L2) need every resident CTA to cover HBM latency
    int64_t cap = (int64_t)ctx->sm_count * (work > (int64_t)4 << 20 ? per_sm : 1);
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return (int)want;
}

// Cluster-synchronised variant for operators that a single cluster can chew through (a few 10^5 nonzeros, everything
// L2 resident): ONE cluster of 16 (or 8) CTAs x 1024 threads, every phase boundary is a hardware cluster barrier.
constexpr int64_t CL_CLUSTER_WORK = (int64_t)512 << 10;

// launch of `grid` CL_THREADS-thread CTAs in thread-block clusters of `cs`; `at` stores the cluster attribute
static cudaLaunchConfig_t cluster_config(unsigned grid, unsigned cs, size_t dyn, cudaStream_t stream, cudaLaunchAttribute& at) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(CL_THREADS);
    cfg.dynamicSmemBytes = dyn;
    cfg.stream = stream;
    at = cudaLaunchAttribute{};
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = cs;
    at.val.clusterDim.y = 1;
    at.val.clusterDim.z = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    return cfg;
}

static int cluster_size_for(diffopt_b200_ctx* ctx, const void* kernel) {
    static int cached = -1;  // per process; every B200 in a box is the same part
    if (cached >= 0) return cached;
    cached = 0;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        cudaGetLastError();
    }
    for (int cs : {16, 8}) {
        cudaLaunchAttribute at;
        const cudaLaunchConfig_t cfg = cluster_config((unsigned)cs, (unsigned)cs, CL_CHUNK * sizeof(double), nullptr, at);
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) == cudaSuccess && n >= 1) {
            cached = cs;
            break;
        }
        cudaGetLastError();
    }
    (void)ctx;
    return cached;
}

static int32_t lsqr_launch(diffopt_b200_ctx* ctx, OpArgs& o, int64_t work, const double* rhs_dev, LsqrParams prm,
                           double* x_dev, double* stats_host7) {
    LsqrWork& wk = ctx->lsqr;
    const size_t d = sizeof(double);
    DO_CUDA(ctx, wk.u.reserve(d * (size_t)o.nrows));
    DO_CUDA(ctx, wk.v.reserve(d * (size_t)o.ncols));
    DO_CUDA(ctx, wk.w.reserve(d * (size_t)o.ncols));
    const void* k_cluster = (const void*)lsqr_kernel_t<CL_THREADS, CL_NPT, 1, true, false>;
    const void* k_gstream = (const void*)lsqr_kernel_t<CL_THREADS, CL_NPT, 1, false, false>;
    // problems with PSD cones: 256 threads (the GEMM phases of the PSD apply are written for them), 2 CTAs per SM
    const void* k_grid = (const void*)lsqr_kernel_t<LSQR_THREADS, LSQR_NPT, 2, false, true>;
    // Three persistent variants, all with the row-block SpMV (`work` ~ nonzeros + vector lengths):
    //   cluster : <= CL_CLUSTER_WORK  one 16-CTA cluster, hardware barriers (16 SMs are enough)
    //   gstream : larger              one CTA per SM, grid.sync() (L1 gather rate of 16 SMs is not enough)
    //   grid    : PSD cones           256-thread CTAs, up to 2 per SM, grid.sync()
    const char* mode = getenv("DIFFOPT_B200_LSQR");
    const bool psd = o.kind == 1 && o.conic.npsd > 0;
    int variant = psd || (mode && strcmp(mode, "grid") == 0) ? 0 : work <= CL_CLUSTER_WORK ? 1 : 2;  // 0 grid, 1 cluster, 2 gstream
    if (mode && strcmp(mode, "cluster") == 0 && !psd) variant = 1;
    if (mode && strcmp(mode, "gstream") == 0 && !psd) variant = 2;
    int cs = variant == 1 ? cluster_size_for(ctx, k_cluster) : 0;
    if (variant == 1 && cs == 0) variant = 2;
    const size_t dyn = (variant ? CL_CHUNK : ST_CHUNK) * sizeof(double);
    int grid = cs;
    if (variant == 0) grid = coop_grid(ctx, k_grid, dyn, work);
    if (variant == 2) {
        DO_CUDA(ctx, cudaFuncSetAttribute(k_gstream, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        grid = ctx->sm_count;
    }
    {   // the row-block lists cut for the launch's block shape
        auto pick = [&](CsrView& v, const CsrDev& M, bool t) {
            const DevBuf* lists[3][2] = {{&M.blk, &M.t_blk}, {&M.cblk, &M.t_cblk}, {&M.gblk, &M.t_gblk}};
            const int64_t counts[3][2] = {{M.nblk, M.t_nblk}, {M.ncblk, M.t_ncblk}, {M.ngblk, M.t_ngblk}};
            v.blk = lists[variant][t]->as<int>();
            v.nblk = (int)counts[variant][t];
        };
        if (o.kind == 1) {
            pick(o.conic.A, ctx->conic.A, false);
            pick(o.conic.At, ctx->conic.A, true);
        } else {
            const bool fwd_is_t = o.fwd.rowptr == ctx->lsqr_mat.t_rowptr.as<int>();
            pick(o.fwd, ctx->lsqr_mat, fwd_is_t);
            pick(o.adj, ctx->lsqr_mat, !fwd_is_t);
        }
    }
    DO_CUDA(ctx, wk.tmp.reserve(d * (size_t)LSQR_NSLOTS * (size_t)grid));
    DO_CUDA(ctx, wk.scal.reserve(d * 8));
    DO_CUDA(ctx, cudaMemsetAsync(wk.tmp.ptr, 0, d * (size_t)LSQR_NSLOTS * (size_t)grid, ctx->stream));
    LsqrVectors vec{wk.u.as<double>(), wk.v.as<double>(), wk.w.as<double>(), x_dev, wk.tmp.as<double>(),
                    wk.scal.as<double>()};
    void* args[] = {&o, (void*)&rhs_dev, &prm, &vec};
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (variant == 1) {
        cudaLaunchAttribute at;
        const cudaLaunchConfig_t cfg = cluster_config((unsigned)cs, (unsigned)cs, dyn, ctx->stream, at);
        DO_CUDA(ctx, cudaLaunchKernelExC(&cfg, k_cluster, args));
    } else if (variant == 2) {
        DO_CUDA(ctx, cudaLaunchCooperativeKernel(k_gstream, dim3(grid), dim3(CL_THREADS), args, dyn, ctx->stream));
    } else {
        DO_CUDA(ctx, cudaLaunchCooperativeKernel(k_grid, dim3(grid), dim3(LSQR_THREADS), args, dyn, ctx->stream));
    }
    ctx->launches++;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    double st[7];
    DO_CUDA(ctx, cudaMemcpyAsync(st, wk.scal.ptr, sizeof st, cudaMemcpyDeviceToHost, ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    if (stats_host7) memcpy(stats_host7, st, sizeof st);
    return 0;
}

int32_t lsqr_run_csr(diffopt_b200_ctx* ctx, const CsrDev& M, bool trans, const double* rhs_dev, LsqrParams prm,
                     double* x_dev, double* stats_host7) {
    OpArgs o{};
    o.kind = 0;
    CsrView a = view_of(M.rowptr, M.colind, M.val, M.nrows, M.ncols, &M.cblk, M.ncblk);
    CsrView at = view_of(M.t_rowptr, M.t_colind, M.t_val, M.ncols, M.nrows, &M.t_cblk, M.t_ncblk);
    o.fwd = trans ? at : a;
    o.adj = trans ? a : at;
    o.nrows = (int)(trans ? M.ncols : M.nrows);
    o.ncols = (int)(trans ? M.nrows : M.ncols);
    return lsqr_launch(ctx, o, M.nnz + M.nrows + M.ncols, rhs_dev, prm, x_dev, stats_host7);
}

static int32_t lsqr_stream_conic(diffopt_b200_ctx* ctx, const double* rhs_dev, LsqrParams prm, double* x_dev, double* stats_host7) {
    ConicState& cs = ctx->conic;
    LsqrWork& wk = ctx->lsqr;
    ConicOpView op = conic_view(ctx, true);
    const int n = (int)cs.n, m = (int)cs.m, N = n + m + 1;
    const size_t dsz = sizeof(double);
    DO_CUDA(ctx, wk.u.reserve(dsz * (size_t)N));
    DO_CUDA(ctx, wk.v.reserve(dsz * (size_t)N));
    DO_CUDA(ctx, wk.w.reserve(dsz * (size_t)N));
    const int stride = ST_STRIDE;
    DO_CUDA(ctx, wk.tmp.reserve(dsz * (size_t)LSQR_NSLOTS * (size_t)stride));
    DO_CUDA(ctx, wk.scal.reserve(dsz * 8 + sizeof(LsqrState) + 64));
    double* stats = wk.scal.as<double>();
    LsqrState* S = reinterpret_cast<LsqrState*>(stats + 8);
    LsqrVectors vec{wk.u.as<double>(), wk.v.as<double>(), wk.w.as<double>(), x_dev, wk.tmp.as<double>(), stats};
    auto blocks_for = [&](int64_t items) {
        int64_t b = (items + ST_THREADS - 1) / ST_THREADS;
        if (b > stride) b = stride;
        if (b < 1) b = 1;
        return (unsigned)b;
    };
    // Dpi: one thread per row (diagonal and 3 x 3 block rows), 8 lanes per SOC cone
    const unsigned g_vec = blocks_for(N), g_dpi = blocks_for(std::max<int64_t>(m, (int64_t)cs.nsoc * 8));
    // SpMV kernels: persistent over the row blocks, every resident CTA slot filled exactly once (8 CTAs per SM)
    auto blocks_spmv = [&](int64_t nblk) {
        int per_sm = 8;
        if (const char* e = getenv("DIFFOPT_B200_SPMV_CTAS")) per_sm = std::max(1, atoi(e));
        int64_t b = std::min<int64_t>(nblk, (int64_t)ctx->sm_count * per_sm);
        return (unsigned)std::max<int64_t>(1, std::min<int64_t>(b, stride));
    };
    const unsigned g_rows = blocks_spmv(cs.A.nblk + cs.A.t_nblk), g_a = blocks_spmv(cs.A.nblk);
    const unsigned g_trows = blocks_spmv(std::max<int64_t>(cs.A.t_nblk, ((int64_t)m + SP_THREADS * 8 - 1) / (SP_THREADS * 8)));
    cudaStream_t st = ctx->stream;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
    st_init_kernel<<<g_vec, ST_THREADS, 0, st>>>(N, N, rhs_dev, vec);
    st_init_fin_kernel<<<1, ST_THREADS, 0, st>>>(vec, stride, (int)g_vec, S);
    auto apply_Mt = [&](int startup) {  // v = su M' u + op_dst v
        st_Mt_A_kernel<<<g_a, SP_THREADS, 0, st>>>(op, vec.u, vec.partials, S);
        st_dpi_kernel<<<g_dpi, ST_THREADS, 0, st>>>(op, op.wc, op.wc + m, 1, S, 1);
        st_Mt_rows_kernel<<<g_trows, SP_THREADS, 0, st>>>(op, vec.u, vec.v, vec.partials, S);
        st_end_kernel<<<1, ST_THREADS, 0, st>>>(N, vec, stride, (int)g_a, (int)g_trows, prm, S, startup);
        ctx->launches += 4;
    };
    apply_Mt(1);
    ctx->launches += 2;
    LsqrState hs{};
    const long long batch = 16;
    for (long long it = 0; it <= prm.maxiter; it += batch) {
        for (long long k = 0; k < batch; ++k) {
            st_update_kernel<<<g_vec, ST_THREADS, 0, st>>>(N, vec, S);
            st_dpi_kernel<<<g_dpi, ST_THREADS, 0, st>>>(op, vec.v + n, op.wc, 0, S, 0);
            st_M_rows_kernel<<<g_rows, SP_THREADS, 0, st>>>(op, vec.v, vec.u, vec.partials, S);
            st_mid_kernel<<<1, ST_THREADS, 0, st>>>(N, vec, stride, (int)g_rows, (int)g_vec, prm, S);
            ctx->launches += 4;
            apply_Mt(0);
        }
        DO_CUDA(ctx, cudaMemcpyAsync(&hs, S, sizeof hs, cudaMemcpyDeviceToHost, st));
        DO_CUDA(ctx, cudaStreamSynchronize(st));
        if (hs.done) break;
    }
    st_stats_kernel<<<1, 1, 0, st>>>(S, stats);
    ctx->launches++;
    DO_CUDA(ctx, cudaGetLastError());
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
    double stv[7];
    DO_CUDA(ctx, cudaMemcpyAsync(stv, stats, sizeof stv, cudaMemcpyDeviceToHost, st));
    DO_CUDA(ctx, cudaStreamSynchronize(st));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    if (stats_host7) memcpy(stats_host7, stv, sizeof stv);
    return 0;
}

int32_t lsqr_run_conic(diffopt_b200_ctx* ctx, const double* rhs_dev, LsqrParams prm, double* x_dev,
                       double* stats_host7) {
    ConicState& s = ctx->conic;
    OpArgs o{};
    o.kind = 1;
    o.conic = conic_view(ctx);
    o.conic_trans = 0;
    o.nrows = o.ncols = (int)(s.n + s.m + 1);
    int64_t work = s.A.nnz * 2 + s.n + 2 * s.m + s.psd_sumd2 * 8;
    // large operators without PSD cones: one kernel per phase at full occupancy (see lsqr_stream_conic)
    const char* mode = getenv("DIFFOPT_B200_LSQR");
    const bool want_stream = mode ? strcmp(mode, "stream") == 0 : work > ((int64_t)4 << 20);
    if (want_stream && s.npsd == 0 && !(mode && strcmp(mode, "persistent") == 0))
        return lsqr_stream_conic(ctx, rhs_dev, prm, x_dev, stats_host7);
    return lsqr_launch(ctx, o, work, rhs_dev, prm, x_dev, stats_host7);
}

// dyn: dynamic shared memory of the kernel (conic_M_kernel: the products of its row blocks)
static int32_t conic_small_launch(diffopt_b200_ctx* ctx, const void* kernel, size_t dyn, const double* t_dev, bool transpose,
                                  double* out_dev) {
    ConicState& s = ctx->conic;
    ConicOpView op = conic_view(ctx, true);  // the streaming row blocks, cut for the LSQR_THREADS x LSQR_NPT shape
    int64_t work = s.A.nnz * 2 + s.n + 2 * s.m + s.psd_sumd2 * 8;
    int grid = coop_grid(ctx, kernel, dyn, work);
    DO_CUDA(ctx, ctx->lsqr.tmp.reserve(sizeof(double) * (size_t)LSQR_NSLOTS * (size_t)grid));
    double* partials = ctx->lsqr.tmp.as<double>();
    int tr = transpose ? 1 : 0;
    void* args[] = {&op, &tr, (void*)&t_dev, &out_dev, &partials};
    DO_CUDA(ctx, cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(LSQR_THREADS), args, dyn, ctx->stream));
    ctx->launches++;
    return 0;
}

int32_t conic_apply_M(diffopt_b200_ctx* ctx, const double* t_dev, bool transpose, double* out_dev) {
    return conic_small_launch(ctx, (const void*)conic_M_kernel, ST_CHUNK * sizeof(double), t_dev, transpose, out_dev);
}
int32_t conic_apply_dpi(diffopt_b200_ctx* ctx, const double* t_dev, bool transpose, double* out_dev) {
    return conic_small_launch(ctx, (const void*)conic_dpi_kernel, 0, t_dev, transpose, out_dev);
}

// Lock-step batch of conic problems (diffopt_b200_conic_batch_reverse): one persistent kernel, problem p on the C CTAs of
// cluster p.  `work` holds one region per problem, laid out by L.  With C == 1 and `stage` the gather vectors are staged
// in shared memory.
int32_t lsqr_run_conic_batch(diffopt_b200_ctx* ctx, std::vector<ConicState>& states, int C, bool stage, double* work,
                             const LsqrBatchLayout& L, LsqrParams prm, double zero_below, DevBuf& ops_buf, DevBuf& vecs_buf,
                             DevBuf& rhs_buf) {
    const int B = (int)states.size();
    if (B == 0) return 0;
    const int n = (int)states[0].n, m = (int)states[0].m, N = n + m + 1;
    std::vector<OpArgs> ops((size_t)B);
    std::vector<LsqrVectors> vecs((size_t)B);
    std::vector<const double*> rhs((size_t)B);
    for (int p = 0; p < B; ++p) {
        std::swap(ctx->conic, states[(size_t)p]);
        OpArgs o{};
        o.kind = 1;
        o.conic = conic_view(ctx);
        o.conic_trans = 0;
        o.nrows = o.ncols = N;
        ops[(size_t)p] = o;
        std::swap(ctx->conic, states[(size_t)p]);
        double* base = work + (size_t)p * L.stride;
        rhs[(size_t)p] = base;
        vecs[(size_t)p] = LsqrVectors{base + L.u, base + L.v, base + L.w, base + L.x, base + L.partials, base + L.stats};
    }
    DO_CUDA(ctx, ops_buf.reserve(sizeof(OpArgs) * (size_t)B));
    DO_CUDA(ctx, vecs_buf.reserve(sizeof(LsqrVectors) * (size_t)B));
    DO_CUDA(ctx, rhs_buf.reserve(sizeof(double*) * (size_t)B));
    DO_CUDA(ctx, cudaMemcpyAsync(ops_buf.ptr, ops.data(), sizeof(OpArgs) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    DO_CUDA(ctx, cudaMemcpyAsync(vecs_buf.ptr, vecs.data(), sizeof(LsqrVectors) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    DO_CUDA(ctx, cudaMemcpyAsync(rhs_buf.ptr, rhs.data(), sizeof(double*) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // host vectors die at return
    stage = stage && C == 1;
    const size_t dyn = sizeof(double) * ((size_t)CL_CHUNK + (stage ? (size_t)(n + m) : 0));
    if (dyn > ctx->smem_optin) stage = false;
    const size_t dyn2 = sizeof(double) * ((size_t)CL_CHUNK + (stage ? (size_t)(n + m) : 0));
    const void* kern = stage ? (const void*)lsqr_batch_kernel<true> : (const void*)lsqr_batch_kernel<false>;
    DO_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn2));
    const OpArgs* dops = ops_buf.as<OpArgs>();
    const double* const* drhs = rhs_buf.as<const double*>();
    const LsqrVectors* dvecs = vecs_buf.as<LsqrVectors>();
    void* args[] = {(void*)&dops, (void*)&drhs, &prm, (void*)&dvecs, &C, &zero_below};
    cudaLaunchAttribute at;
    const cudaLaunchConfig_t cfg = cluster_config((unsigned)(B * C), (unsigned)C, dyn2, ctx->stream, at);
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    DO_CUDA(ctx, cudaLaunchKernelExC(&cfg, kern, args));
    ctx->launches++;
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    return 0;
}

// Many right-hand sides against the operator of the current conic_setup (lsqr_multi_kernel), G groups of KB directions.
// Operators up to CL_CLUSTER_WORK without PSD cones: one thread-block cluster per group, every group in one launch
// (clusters beyond those the GPU holds at once start as earlier groups retire).  Larger operators and problems with PSD
// cones: one cooperative grid per group, the groups one after another.
int32_t lsqr_run_conic_multi(diffopt_b200_ctx* ctx, int KB, int64_t G, const double* rhs, const double* rhs_norm2,
                             double zero_below, LsqrParams prm, double* x, double* stats) {
    ConicState& s = ctx->conic;
    const int64_t n = s.n, m = s.m, N = n + m + 1;
    MultiArgs a{};
    a.op = conic_view(ctx, true);  // the blk / t_blk row blocks
    a.rhs = rhs;
    a.rhs_norm2 = rhs_norm2;
    a.zero_below = zero_below;
    a.x = x;
    a.stats = stats;
    a.sumd2 = s.psd_sumd2;
    const int64_t work = s.A.nnz * 2 + n + 2 * m + s.psd_sumd2 * 8;
    bool cluster = work <= CL_CLUSTER_WORK && s.npsd == 0;
    const void* k_cluster = KB == 4 ? (const void*)lsqr_multi_kernel<4, true> : (const void*)lsqr_multi_kernel<8, true>;
    const void* k_grid = KB == 4 ? (const void*)lsqr_multi_kernel<4, false> : (const void*)lsqr_multi_kernel<8, false>;
    const size_t dyn = sizeof(double) * (size_t)KB * MR_PLD;
    int cs = 0;
    if (cluster) {
        DO_CUDA(ctx, cudaFuncSetAttribute(k_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        if (cudaFuncSetAttribute(k_cluster, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) cudaGetLastError();
        for (int c : {16, 8}) {
            cudaLaunchAttribute at;
            cudaLaunchConfig_t cfg = cluster_config((unsigned)c, (unsigned)c, dyn, nullptr, at);
            cfg.blockDim = dim3(MR_THREADS);
            int resident = 0;
            if (cudaOccupancyMaxActiveClusters(&resident, k_cluster, &cfg) == cudaSuccess && resident >= 1) {
                cs = c;
                break;
            }
            cudaGetLastError();
        }
        cluster = cs > 0;
    }
    int grid = cs;
    if (!cluster) {
        DO_CUDA(ctx, cudaFuncSetAttribute(k_grid, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        grid = coop_grid(ctx, k_grid, dyn, work);
    }
    a.ctas = grid;
    a.work_stride = (size_t)KB * (size_t)(3 * N + 2 * m + 2 * s.psd_sumd2 + (int64_t)LSQR_NSLOTS * grid);
    const int64_t regions = cluster ? G : 1;
    DO_CUDA(ctx, ctx->lsqr.m_work.reserve(sizeof(double) * a.work_stride * (size_t)regions));
    a.work = ctx->lsqr.m_work.as<double>();
    DO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (cluster) {
        a.group0 = 0;
        void* args[] = {&a, &prm};
        cudaLaunchAttribute at;
        cudaLaunchConfig_t cfg = cluster_config((unsigned)(G * cs), (unsigned)cs, dyn, ctx->stream, at);
        cfg.blockDim = dim3(MR_THREADS);
        DO_CUDA(ctx, cudaLaunchKernelExC(&cfg, k_cluster, args));
        ctx->launches++;
    } else {
        for (int64_t g = 0; g < G; ++g) {
            a.group0 = (int)g;
            void* args[] = {&a, &prm};
            DO_CUDA(ctx, cudaLaunchCooperativeKernel(k_grid, dim3(grid), dim3(MR_THREADS), args, dyn, ctx->stream));
            ctx->launches++;
        }
    }
    DO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    return 0;
}

// Host: Julia CSC (1-based int64) -> device CSR of the matrix and of its transpose (0-based int32).
int32_t csr_from_csc_host(diffopt_b200_ctx* ctx, int64_t nrows, int64_t ncols, const int64_t* colptr,
                          const int64_t* rowval, const double* nzval, CsrDev& out) {
    if (nrows < 0 || ncols < 0 || !colptr) BAD_ARG(ctx, "csc: bad dimensions");
    const int64_t nnz = colptr[ncols] - colptr[0];
    if (colptr[0] != 1) BAD_ARG(ctx, "csc: colptr must be 1-based (Julia SparseMatrixCSC)");
    if (nnz < 0 || nnz > 2000000000LL || nrows > 2000000000LL || ncols > 2000000000LL)
        BAD_ARG(ctx, "csc: too large for int32 indices");
    // transpose view = CSC arrays reinterpreted: rows of A' are the columns of A
    std::vector<int> t_rowptr((size_t)ncols + 1), t_colind((size_t)nnz);
    for (int64_t j = 0; j <= ncols; ++j) t_rowptr[(size_t)j] = (int)(colptr[j] - 1);
    for (int64_t k = 0; k < nnz; ++k) {
        int64_t r = rowval[k] - 1;
        if (r < 0 || r >= nrows) BAD_ARG(ctx, "csc: row index out of range");
        t_colind[(size_t)k] = (int)r;
    }
    // CSR of A by counting sort over rows
    std::vector<int> rowptr((size_t)nrows + 1, 0), colind((size_t)nnz);
    std::vector<double> val((size_t)nnz);
    for (int64_t k = 0; k < nnz; ++k) rowptr[(size_t)t_colind[(size_t)k] + 1]++;
    for (int64_t i = 0; i < nrows; ++i) rowptr[(size_t)i + 1] += rowptr[(size_t)i];
    std::vector<int> next(rowptr.begin(), rowptr.end() - 1);
    for (int64_t j = 0; j < ncols; ++j)
        for (int k = t_rowptr[(size_t)j]; k < t_rowptr[(size_t)j + 1]; ++k) {
            int r = t_colind[(size_t)k];
            int dst = next[(size_t)r]++;
            colind[(size_t)dst] = (int)j;
            val[(size_t)dst] = nzval[k];
        }
    // row blocks of the streaming SpMV: <= ST_CHUNK nonzeros and <= SP_THREADS rows each, or one longer row
    auto row_blocks = [](const std::vector<int>& rp, int64_t nr, std::vector<int>& blk) {
        blk.clear();
        blk.push_back(0);
        int64_t r = 0;
        while (r < nr) {
            const int s0 = rp[(size_t)r];
            int64_t e = r;
            while (e < nr && rp[(size_t)e + 1] - s0 <= ST_CHUNK && e - r < SP_THREADS) ++e;
            if (e == r) e = r + 1;
            blk.push_back((int)e);
            r = e;
        }
        // interleave (first row, first nonzero) per block: one 8-byte load per block end for the issuing thread
        std::vector<int> d2(blk.size() * 2);
        for (size_t k = 0; k < blk.size(); ++k) {
            d2[2 * k] = blk[k];
            d2[2 * k + 1] = rp[(size_t)blk[k]];
        }
        blk.swap(d2);
    };
    // the same for the cluster-synchronised kernel: about one block per CTA and round, <= CL_CHUNK nonzeros each
    auto cluster_blocks = [](const std::vector<int>& rp, int64_t nr, int64_t CTAS, std::vector<int>& blk) {
        const int64_t nz = nr > 0 ? rp[(size_t)nr] : 0;
        const int64_t rounds = std::max<int64_t>(1, (nz + CTAS * CL_CHUNK - 1) / (CTAS * CL_CHUNK));
        const int64_t rows_round = std::max<int64_t>(1, (nr + CTAS * CL_THREADS - 1) / (CTAS * CL_THREADS));
        const int64_t want = CTAS * std::max(rounds, rows_round);
        double target = (double)std::max<int64_t>(nz / want + 1, 1);
        for (int attempt = 0; attempt < 24; ++attempt) {
            const int cap = (int)std::min<double>(target, (double)CL_CHUNK);
            blk.clear();
            blk.push_back(0);
            int64_t r = 0;
            while (r < nr) {
                const int s0 = rp[(size_t)r];
                int64_t e = r;
                while (e < nr && rp[(size_t)e + 1] - s0 <= cap && e - r < CL_THREADS) ++e;
                if (e == r) e = r + 1;
                blk.push_back((int)e);
                r = e;
            }
            if ((int64_t)blk.size() - 1 <= want || cap >= CL_CHUNK) break;
            target *= 1.03;
        }
        std::vector<int> d2(blk.size() * 2);
        for (size_t k = 0; k < blk.size(); ++k) {
            d2[2 * k] = blk[k];
            d2[2 * k + 1] = rp[(size_t)blk[k]];
        }
        blk.swap(d2);
    };
    std::vector<int> blk, t_blk, cblk, t_cblk, gblk, t_gblk;
    row_blocks(rowptr, nrows, blk);
    row_blocks(t_rowptr, ncols, t_blk);
    const int64_t cl_ctas = ctx->csr_cluster_ctas > 0 ? ctx->csr_cluster_ctas : CL_MAX_CTAS;
    cluster_blocks(rowptr, nrows, cl_ctas, cblk);
    cluster_blocks(t_rowptr, ncols, cl_ctas, t_cblk);
    cluster_blocks(rowptr, nrows, ctx->sm_count, gblk);
    cluster_blocks(t_rowptr, ncols, ctx->sm_count, t_gblk);
    out.ncblk = (int64_t)cblk.size() / 2 - 1;
    out.t_ncblk = (int64_t)t_cblk.size() / 2 - 1;
    out.ngblk = (int64_t)gblk.size() / 2 - 1;
    out.t_ngblk = (int64_t)t_gblk.size() / 2 - 1;
    out.nblk = (int64_t)blk.size() / 2 - 1;
    out.t_nblk = (int64_t)t_blk.size() / 2 - 1;
    // Large operators (the streaming driver): a second copy of (val, colind) with the nonzeros of every row block
    // ordered by column, plus each nonzero's position inside its block.  The gathers of a warp then fall into few
    // 128-byte lines when the operator has any locality (the L1TEX takes ~one line request per clock per SM, which is
    // what bounds the row-block SpMV), the products are scattered back to their CSR positions in shared memory, and the
    // row sums are unchanged bit for bit.
    std::vector<double> sval, t_sval;
    std::vector<int> scol, t_scol;
    std::vector<unsigned short> spos, t_spos;
    const char* sort_env = getenv("DIFFOPT_B200_SPMV_SORT");
    const bool want_sort = sort_env ? atoi(sort_env) != 0 : nnz >= ((int64_t)1 << 21);
    auto sort_blocks = [](const std::vector<int>& blk2, const std::vector<int>& ci, const double* va,
                          std::vector<double>& sv, std::vector<int>& sc, std::vector<unsigned short>& sp) {
        const size_t nb = blk2.size() / 2 - 1;
        const size_t nz = ci.size();
        sv.resize(nz); sc.resize(nz); sp.resize(nz);
        auto work = [&](size_t b0, size_t b1) {
            std::vector<int> idx;
            for (size_t b = b0; b < b1; ++b) {
                const int s0 = blk2[2 * b + 1], s1 = blk2[2 * b + 3], cnt = s1 - s0;
                if (cnt > ST_CHUNK) {  // one long row: streamed in place
                    for (int k = s0; k < s1; ++k) { sv[(size_t)k] = va[k]; sc[(size_t)k] = ci[(size_t)k]; sp[(size_t)k] = 0; }
                    continue;
                }
                idx.resize((size_t)cnt);
                for (int j = 0; j < cnt; ++j) idx[(size_t)j] = j;
                std::stable_sort(idx.begin(), idx.end(), [&](int a, int c) { return ci[(size_t)(s0 + a)] < ci[(size_t)(s0 + c)]; });
                for (int j = 0; j < cnt; ++j) {
                    const int k = s0 + idx[(size_t)j];
                    sv[(size_t)(s0 + j)] = va[k];
                    sc[(size_t)(s0 + j)] = ci[(size_t)k];
                    sp[(size_t)(s0 + j)] = (unsigned short)idx[(size_t)j];
                }
            }
        };
        const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < hw; ++t) pool.emplace_back(work, nb * t / hw, nb * (t + 1) / hw);
        for (auto& th : pool) th.join();
    };
    if (want_sort && nnz > 0) {
        sort_blocks(blk, colind, val.data(), sval, scol, spos);
        sort_blocks(t_blk, t_colind, nzval, t_sval, t_scol, t_spos);
    }
    out.sorted = want_sort && nnz > 0;
    out.nrows = nrows;
    out.ncols = ncols;
    out.nnz = nnz;
    auto up = [&](DevBuf& b, const void* src, size_t bytes) -> cudaError_t {
        cudaError_t e = b.reserve(bytes ? bytes : 8);
        if (e != cudaSuccess) return e;
        return bytes ? cudaMemcpyAsync(b.ptr, src, bytes, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
    };
    DO_CUDA(ctx, up(out.rowptr, rowptr.data(), sizeof(int) * rowptr.size()));
    DO_CUDA(ctx, up(out.colind, colind.data(), sizeof(int) * colind.size()));
    DO_CUDA(ctx, up(out.val, val.data(), sizeof(double) * val.size()));
    DO_CUDA(ctx, up(out.t_rowptr, t_rowptr.data(), sizeof(int) * t_rowptr.size()));
    DO_CUDA(ctx, up(out.t_colind, t_colind.data(), sizeof(int) * t_colind.size()));
    DO_CUDA(ctx, up(out.t_val, nzval, sizeof(double) * (size_t)nnz));
    if (out.sorted) {
        DO_CUDA(ctx, up(out.sval, sval.data(), sizeof(double) * sval.size()));
        DO_CUDA(ctx, up(out.scol, scol.data(), sizeof(int) * scol.size()));
        DO_CUDA(ctx, up(out.spos, spos.data(), sizeof(unsigned short) * spos.size()));
        DO_CUDA(ctx, up(out.t_sval, t_sval.data(), sizeof(double) * t_sval.size()));
        DO_CUDA(ctx, up(out.t_scol, t_scol.data(), sizeof(int) * t_scol.size()));
        DO_CUDA(ctx, up(out.t_spos, t_spos.data(), sizeof(unsigned short) * t_spos.size()));
    }
    DO_CUDA(ctx, up(out.blk, blk.data(), sizeof(int) * blk.size()));
    DO_CUDA(ctx, up(out.t_blk, t_blk.data(), sizeof(int) * t_blk.size()));
    DO_CUDA(ctx, up(out.cblk, cblk.data(), sizeof(int) * cblk.size()));
    DO_CUDA(ctx, up(out.t_cblk, t_cblk.data(), sizeof(int) * t_cblk.size()));
    DO_CUDA(ctx, up(out.gblk, gblk.data(), sizeof(int) * gblk.size()));
    DO_CUDA(ctx, up(out.t_gblk, t_gblk.data(), sizeof(int) * t_gblk.size()));
    DO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // host vectors die at return
    return 0;
}
