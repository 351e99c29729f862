// Device-side building blocks of the pivot-free LDL' fast path of the batched KKT sensitivity solve, shared by the
// kernel tuned for the headline shape (qp_batch_sqd.cu) and the kernel for any (n, m, p) (qp_batch_sqd_any.cu):
// the 8 x 8 tile layout, the diagonal-block elimination, the panel-row solve, the blocked factorisation with both
// right-hand sides riding along and the paired backward substitution.  Algorithm: see qp_batch_sqd.cu.
#pragma once
#include "common.cuh"

#ifndef QP_ABLATE
#define QP_ABLATE 0
#endif

namespace sqd {

constexpr int THREADS = 128, NWARP = THREADS / 32;
constexpr unsigned FULL = 0xffffffffu;
constexpr double PIV_RTOL = 1e-12;

__device__ __forceinline__ int tix(int I, int J) { return ((I * (I + 1)) >> 1) + J; }

// One instance's stored LDL' factor (qp_batch_factorize; written by the store mode of qp_kkt_sqd_any_kernel, read by
// qp_batch_factored.cu), `stride` doubles per instance, every segment 16-byte aligned:
//   ints  [0] = ma, the active-set size (-1: the instance is served by the pivoted LU), [1 .. m] = apos (reduced row of
//         inequality i minus n8, -1 when inactive)
//   dvec  D = G z - h (m)
//   rd    1 / d of every reduced row (8 nt_cap)
//   tiles the lower-triangular tile grid (tix order) exactly as factor<>() leaves it: strict lower triangles of the
//         diagonal tiles hold L_jj, the tiles below the diagonal W(I, j) = L(I, j) D_j, in-tile swizzle of el()
struct FactorLayout {
    int ints, dvec, rd, tiles, stride;
    __host__ __device__ FactorLayout(int m, int nt_cap) {
        ints = 0;
        dvec = (((m + 2) >> 1) + 1) & ~1;
        rd = dvec + ((m + 1) & ~1);
        tiles = rd + 8 * nt_cap;
        stride = (tiles + (nt_cap * (nt_cap + 1) / 2) * 64 + 15) & ~15;
    }
};

// Offset of element (r, c) inside an 8 x 8 tile.  Rows are 64 B; the four 16-byte chunks of row r are stored at
// chunk ^ ((r >> 1) & 3).  DMMA fragment accesses (lane (g, t) -> chunk t of row g) and whole-row accesses (one lane
// per row, chunk q of rows 0..7) are then both free of shared-memory bank conflicts.
__device__ __forceinline__ int el(int r, int c) { return r * 8 + ((((c >> 1) ^ (r >> 1)) & 3) << 1) + (c & 1); }
__device__ __forceinline__ int swz(int r) { return (r >> 1) & 3; }

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

// m16n8k8: two vertically adjacent 8 x 8 tiles (rows g and g+8 of the 16-row A / C operands) against one B tile.
// With the k-slot convention used throughout (slot t <-> tile column 2t, slot t+4 <-> column 2t+1) the operands
// are exactly the double2 fragments at offset `fo` of the two A tiles, the B tile and the two C tiles.
__device__ __forceinline__ void dmma16(double2& c_top, double2& c_bot, const double2 a_top, const double2 a_bot, const double2 b) {
    asm("mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+d"(c_top.x), "+d"(c_top.y), "+d"(c_bot.x), "+d"(c_bot.y)
        : "d"(a_top.x), "d"(a_bot.x), "d"(a_top.y), "d"(a_bot.y), "d"(b.x), "d"(b.y));
}

__device__ __forceinline__ double2 ldg2(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }

// 1/x: hardware estimate (rel. error <= 2^-20) + one cubic Newton step r0 (1 + e + e^2), e = 1 - x r0:
// rel. error e^3 < 2^-60, three dependent FMAs on the pivot chain instead of four.
__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    const double t = fma(e, e, e);
    return fma(r, t, r);
}

// named barrier of the warp pair that owns right-hand side r (ids 4, 5)
__device__ __forceinline__ void pair_barrier(const int r) {
    if (r) asm volatile("bar.sync 5, 64;" ::: "memory");
    else asm volatile("bar.sync 4, 64;" ::: "memory");
}

__device__ __forceinline__ double sum_over_g(double v) {  // lanes sharing t = lane & 3
    v += __shfl_xor_sync(FULL, v, 4);
    v += __shfl_xor_sync(FULL, v, 8);
    v += __shfl_xor_sync(FULL, v, 16);
    return v;
}
__device__ __forceinline__ double sum_over_t(double v) {  // lanes sharing g = lane >> 2
    v += __shfl_xor_sync(FULL, v, 1);
    v += __shfl_xor_sync(FULL, v, 2);
    return v;
}

// LDL' of the 8 x 8 diagonal block by ONE thread, in registers.  The pivot chain is software pipelined: the next
// pivot (one FMA behind r) and its reciprocal are started before the bulk of the rank-1 update is issued.
// On exit the strict lower triangle of the tile holds the unit-lower factor L11, rd[] = 1/d.  Pivots are
// checked after the chain (expected sign, |d_k| > PIV_RTOL x reference; NaN fails).  selfref: the reference is
// the block's own starting diagonal (first block of the Schur complement), recorded into ref[].
static __device__ __noinline__ void elim8(double* D, double* ref, double* rd, const bool positive, const bool selfref, int* fail) {
    double a[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            if (c <= i) {
                const double2 v = *reinterpret_cast<const double2*>(&D[el(i, c)]);
                a[i][c] = v.x;
                a[i][c + 1] = v.y;
            }
        }
    }
    double thr[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double rf = selfref ? fabs(a[k][k]) : ref[k];
        if (selfref) ref[k] = rf;
        thr[k] = PIV_RTOL * rf;
    }
    double r = fast_rcp(a[0][0]);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        rd[k] = r;
        double rn = 0.0;
        if (k < 7) {
            const double dn = fma(-(a[k + 1][k] * a[k + 1][k]), r, a[k + 1][k + 1]);
            a[k + 1][k + 1] = dn;
            rn = fast_rcp(dn);
        }
        double lk[8];
#pragma unroll
        for (int i = k + 1; i < 8; ++i) lk[i] = a[i][k] * r;
#pragma unroll
        for (int i = k + 2; i < 8; ++i) a[i][k + 1] = fma(-lk[i], a[k + 1][k], a[i][k + 1]);
#pragma unroll
        for (int c = k + 2; c < 8; ++c) {
#pragma unroll
            for (int i = c; i < 8; ++i) a[i][c] = fma(-lk[i], a[c][k], a[i][c]);
        }
#pragma unroll
        for (int i = k + 1; i < 8; ++i) D[el(i, k)] = lk[i];
        r = rn;
    }
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 8; ++k) ok = ok && ((positive ? a[k][k] : -a[k][k]) > thr[k]);
    if (!ok) *fail = 1;
}

// One row w (8 doubles at p) of a panel tile: w <- w L11^-T, i.e. solve x L11' = w with the unit-lower L11 stored
// in the strict lower triangle of tile Ld.  sw = swz(row) for a tile row, 0 for a plain vector.
// scale != nullptr: the result is also multiplied by scale[0..7] (right-hand side rows: v = D^-1 L^-1 r).
__device__ __forceinline__ void panel_row(double* p, const int sw, const double* Ld, const double* scale) {
    double w[8];
    {
        const double2* pp = reinterpret_cast<const double2*>(p);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double2 v = pp[q ^ sw];
            w[2 * q] = v.x;
            w[2 * q + 1] = v.y;
        }
    }
#pragma unroll
    for (int c = 1; c < 8; ++c) {  // row c of L11: entries 0..c-1
        double l[8];
#pragma unroll
        for (int k = 0; k < c; k += 2) {
            const double2 v = *reinterpret_cast<const double2*>(&Ld[el(c, k)]);
            l[k] = v.x;
            l[k + 1] = v.y;
        }
        double acc = w[c], acc2 = 0.0;
#pragma unroll
        for (int k = 0; k < c; ++k) {
            if (k & 1) acc2 = fma(-w[k], l[k], acc2);
            else acc = fma(-w[k], l[k], acc);
        }
        w[c] = acc + acc2;
    }
    if (scale) {
#pragma unroll
        for (int c = 0; c < 8; ++c) w[c] *= scale[c];
    }
    double2* pp = reinterpret_cast<double2*>(p);
#pragma unroll
    for (int q = 0; q < 4; ++q) pp[q ^ sw] = make_double2(w[2 * q], w[2 * q + 1]);
}

// named barriers (id 0 is __syncthreads)
__device__ __forceinline__ void bar_sync(const int id, const int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(const int id, const int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// Work vectors of one instance (shared memory), all indexed in the reduced ordering and at least 8 * nt long.
struct Vecs {
    double *yf, *yb;    // right-hand sides -> v = D^-1 L^-1 r -> solutions (0: forward mode, 1: reverse mode)
    double *sf, *sb;    // backward-substitution accumulators of the critical warps (zero on entry)
    double *sf2, *sb2;  // ... and of their helper warps (zero on entry)
    double *ref;        // starting magnitude of every diagonal entry of the z block (pivot test); the rest is recorded here
    double *rd;         // 1 / d_k
    int* fail;          // set when a pivot fails its test
};

#ifdef QP_PROFILE
#define SQD_SUB_PARAM , long long (&sub)[6]
#define SQD_SUB_ARG , sub
#define SUB0() tsub = clock64()
#define SUB(i)                    \
    do {                          \
        long long _n = clock64(); \
        sub[i] += _n - tsub;      \
        tsub = _n;                \
    } while (0)
#else
#define SQD_SUB_PARAM
#define SQD_SUB_ARG
#define SUB0()
#define SUB(i)
#endif

// Blocked LDL' (block 8) of the nt x nt tile grid T (lower triangle, tix order); tile rows < ntz belong to the z block
// (pivots expected positive), the rest to the constraint block (negative).  Called by all 128 threads after a
// __syncthreads(); the caller synchronises again before it reads the result.  NTZC > 0: ntz known at compile time.
template <int NTZC>
__device__ __forceinline__ void factor(double* const T, const Vecs& V, const int nt, const int np, const int ntz_rt, const int tid,
                                       const int lane, const int warp, const int g, const int t, const int fo SQD_SUB_PARAM) {
    const int ntz = NTZC > 0 ? NTZC : ntz_rt;
#ifdef QP_PROFILE
    long long tsub = 0;
#endif
    // ---- blocked LDL' (block 8), both right-hand sides riding along as two extra panel rows.
    // Warp 0 runs the critical path on its own: eliminate the diagonal block j (one thread, registers), form
    // W(j+1,j), apply it to tile (j+1,j+1), eliminate that ... and only exchanges named-barrier arrivals with
    // the bulk warps 1-3, which per step j solve the remaining panel rows W(I,j) = A(I,j) L11^-T (one thread
    // per row, FMA pipe) and apply the trailing update C(I,K) -= W(I,j) D^-1 W(K,j)' on the DMMA pipe
    // (A fragment reused along a tile row, rows dealt to the warps in snake order).
    //   BAR_E: warp 0 arrives when L_jj, 1/d_j and W(j+1,j) are in place -> bulk warps may run step j
    //   BAR_F: bulk warps arrive when step j is applied               -> warp 0 may touch tiles (j+1, .)
    //   BAR_B: bulk-internal, between the panel rows and the trailing update
    constexpr int BAR_E = 1, BAR_F = 2, BAR_B = 3;
    if (warp == 0) {
        if (lane == 0) elim8(T, &V.ref[0], &V.rd[0], true, false, V.fail);
        __syncwarp();
        for (int j = 0; j < nt; ++j) {
            const int c0 = j << 3;
            SUB0();
            if (j > 0) bar_sync(BAR_F, THREADS);
            SUB(0);
            if (j < nt - 1) {
                double* Wt = T + tix(j + 1, j) * 64;
#if QP_ABLATE != 1
                if (lane < 8) panel_row(Wt + lane * 8, swz(lane), T + tix(j, j) * 64, nullptr);
#endif
                __syncwarp();
            }
            SUB(4);
            __threadfence_block();
            SUB(5);
            bar_arrive(BAR_E, THREADS);
            SUB(1);
            if (j < nt - 1) {
                const double2 wf = *reinterpret_cast<const double2*>(T + tix(j + 1, j) * 64 + fo);
                double* Dn = T + tix(j + 1, j + 1) * 64;
                double2 c = *reinterpret_cast<double2*>(Dn + fo);
                dmma(c.x, c.y, wf.x * -V.rd[c0 + 2 * t], wf.x);
                dmma(c.x, c.y, wf.y * -V.rd[c0 + 2 * t + 1], wf.y);
                *reinterpret_cast<double2*>(Dn + fo) = c;
                __syncwarp();
                SUB(2);
#if QP_ABLATE != 2
                if (lane == 0) elim8(Dn, &V.ref[c0 + 8], &V.rd[c0 + 8], j + 1 < ntz, j + 1 == ntz, V.fail);
#endif
                __syncwarp();
                SUB(3);
            }
        }
    } else {
        const int bt = tid - 32, bw = warp - 1;  // bulk thread / warp index
        for (int j = 0; j < nt; ++j) {
            const int c0 = j << 3;
            SUB0();
            bar_sync(BAR_E, THREADS);
            SUB(0);
            const double* Ld = T + tix(j, j) * 64;
            {   // panel rows 8(j+2) .. np-1 and the two right-hand sides (threads 94, 95)
#if QP_ABLATE != 3
                if (bt < 94) {
                    for (int rr = c0 + 16 + bt; rr < np; rr += 94) panel_row(T + tix(rr >> 3, j) * 64 + (rr & 7) * 8, swz(rr & 7), Ld, nullptr);
                } else {
                    panel_row((bt == 94 ? V.yf : V.yb) + c0, 0, Ld, &V.rd[c0]);
                }
#endif
            }
            if (j == nt - 1) break;
            SUB(1);
            bar_sync(BAR_B, THREADS - 32);
            SUB(2);
            const double nr0 = -V.rd[c0 + 2 * t], nr1 = -V.rd[c0 + 2 * t + 1];
            for (int rr = c0 + 8 + bt; rr < np; rr += THREADS - 32) {
                const double2* wrow = reinterpret_cast<const double2*>(T + tix(rr >> 3, j) * 64 + (rr & 7) * 8);
                double uf = V.yf[rr], ub = V.yb[rr], uf2 = 0.0, ub2 = 0.0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const double2 w2 = wrow[q ^ swz(rr & 7)];
                    const double2 vf = *reinterpret_cast<const double2*>(&V.yf[c0 + 2 * q]);
                    const double2 vb2 = *reinterpret_cast<const double2*>(&V.yb[c0 + 2 * q]);
                    uf = fma(-w2.x, vf.x, uf);
                    uf2 = fma(-w2.y, vf.y, uf2);
                    ub = fma(-w2.x, vb2.x, ub);
                    ub2 = fma(-w2.y, vb2.y, ub2);
                }
                V.yf[rr] = uf + uf2;
                V.yb[rr] = ub + ub2;
            }
            SUB(3);
            // tile rows I = nt-1 .. j+2 (row j+1 is warp 0's single tile) taken in PAIRS (I1-1, I1): one m16n8k8 DMMA
            // updates the two vertically adjacent tiles of a column with a shared B fragment; pairs are dealt to the
            // warps in snake order
            const int nrows = nt - 2 - j, nitems = (nrows + 1) >> 1;
            const double* const b0p = T + tix(j + 1, j) * 64 + fo;
            for (int rnd = 0; 3 * rnd < nitems; ++rnd) {
                const int idx = 3 * rnd + ((rnd & 1) ? 2 - bw : bw);
#if QP_ABLATE == 4
                continue;
#endif
                if (idx >= nitems) continue;
                const int I1 = nt - 1 - 2 * idx, I0 = I1 - 1;
                const double2 w1 = *reinterpret_cast<const double2*>(T + tix(I1, j) * 64 + fo);
                const double2 a1 = make_double2(w1.x * nr0, w1.y * nr1);
                const double* bp = b0p;
                double* c1p = T + tix(I1, j + 1) * 64 + fo;
                int K = j + 1;
                if (I0 >= j + 2) {
                    double2 a0 = *reinterpret_cast<const double2*>(T + tix(I0, j) * 64 + fo);
                    a0.x *= nr0;
                    a0.y *= nr1;
                    double* c0p = T + tix(I0, j + 1) * 64 + fo;
                    for (; K + 3 <= I0; K += 4) {  // four columns per iteration: four independent DMMAs in flight
                        const double2 b0 = *reinterpret_cast<const double2*>(bp);
                        const double2 b1 = *reinterpret_cast<const double2*>(bp + (K + 1) * 64);
                        const double2 b2 = *reinterpret_cast<const double2*>(bp + (2 * K + 3) * 64);
                        const double2 b3 = *reinterpret_cast<const double2*>(bp + (3 * K + 6) * 64);
                        bp += (4 * K + 10) * 64;
                        double2 c00 = *reinterpret_cast<double2*>(c0p), c10 = *reinterpret_cast<double2*>(c1p);
                        double2 c01 = *reinterpret_cast<double2*>(c0p + 64), c11 = *reinterpret_cast<double2*>(c1p + 64);
                        double2 c02 = *reinterpret_cast<double2*>(c0p + 128), c12 = *reinterpret_cast<double2*>(c1p + 128);
                        double2 c03 = *reinterpret_cast<double2*>(c0p + 192), c13 = *reinterpret_cast<double2*>(c1p + 192);
                        dmma16(c00, c10, a0, a1, b0);
                        dmma16(c01, c11, a0, a1, b1);
                        dmma16(c02, c12, a0, a1, b2);
                        dmma16(c03, c13, a0, a1, b3);
                        *reinterpret_cast<double2*>(c0p) = c00;
                        *reinterpret_cast<double2*>(c1p) = c10;
                        *reinterpret_cast<double2*>(c0p + 64) = c01;
                        *reinterpret_cast<double2*>(c1p + 64) = c11;
                        *reinterpret_cast<double2*>(c0p + 128) = c02;
                        *reinterpret_cast<double2*>(c1p + 128) = c12;
                        *reinterpret_cast<double2*>(c0p + 192) = c03;
                        *reinterpret_cast<double2*>(c1p + 192) = c13;
                        c0p += 256;
                        c1p += 256;
                    }
                    for (; K < I0; K += 2) {  // two columns per iteration
                        const double2 b0 = *reinterpret_cast<const double2*>(bp);
                        const double2 b1 = *reinterpret_cast<const double2*>(bp + (K + 1) * 64);
                        bp += (2 * K + 3) * 64;
                        double2 c00 = *reinterpret_cast<double2*>(c0p), c10 = *reinterpret_cast<double2*>(c1p);
                        double2 c01 = *reinterpret_cast<double2*>(c0p + 64), c11 = *reinterpret_cast<double2*>(c1p + 64);
                        dmma16(c00, c10, a0, a1, b0);
                        dmma16(c01, c11, a0, a1, b1);
                        *reinterpret_cast<double2*>(c0p) = c00;
                        *reinterpret_cast<double2*>(c1p) = c10;
                        *reinterpret_cast<double2*>(c0p + 64) = c01;
                        *reinterpret_cast<double2*>(c1p + 64) = c11;
                        c0p += 128;
                        c1p += 128;
                    }
                    if (K == I0) {  // column I0: diagonal tile of row I0 and tile (I1, I0)
                        const double2 b0 = *reinterpret_cast<const double2*>(bp);
                        double2 c00 = *reinterpret_cast<double2*>(c0p), c10 = *reinterpret_cast<double2*>(c1p);
                        dmma16(c00, c10, a0, a1, b0);
                        *reinterpret_cast<double2*>(c0p) = c00;
                        *reinterpret_cast<double2*>(c1p) = c10;
                        c1p += 64;
                        ++K;
                    }
                } else {  // odd row count: row j+2 alone, column j+1 first
                    const double2 b0 = *reinterpret_cast<const double2*>(bp);
                    double2 ca = *reinterpret_cast<double2*>(c1p);
                    dmma(ca.x, ca.y, a1.x, b0.x);
                    dmma(ca.x, ca.y, a1.y, b0.y);
                    *reinterpret_cast<double2*>(c1p) = ca;
                    c1p += 64;
                    ++K;
                }
                {   // diagonal tile (I1, I1): B = W(I1, j) itself
                    double2 ca = *reinterpret_cast<double2*>(c1p);
                    dmma(ca.x, ca.y, a1.x, w1.x);
                    dmma(ca.x, ca.y, a1.y, w1.y);
                    *reinterpret_cast<double2*>(c1p) = ca;
                }
                if (j == ntz - 1) {  // Schur complement of the z block complete: record the diagonals of tiles (I,I)
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int I = q ? I1 : I0;
                        if (I >= j + 2) {
                            const double2 dg = *reinterpret_cast<const double2*>(T + tix(I, I) * 64 + fo);
                            if (g == 2 * t) V.ref[8 * I + g] = fabs(dg.x);
                            if (g == 2 * t + 1) V.ref[8 * I + g] = fabs(dg.y);
                        }
                    }
                }
            }
            __threadfence_block();
            bar_arrive(BAR_F, THREADS);
            SUB(4);
        }
    }
}

// Backward substitution L' x = v for both right-hand sides (called by all 128 threads between two __syncthreads()).
// pf / pf_lines: optional global-memory range (128-byte lines) prefetched into L2 by an otherwise idle warp.
__device__ __forceinline__ void backward(const double* const T, const Vecs& V, const int nt, const int lane, const int warp, const char* pf,
                                         const int pf_lines) {
    // ---- backward substitution L' x = v.  Right-hand side r (0: forward mode, 1: reverse mode) is owned by the
    // warp pair (r, r+2): the critical warp r computes x_j = L11^-T (v_j - D^-1 (s + s2)_j) and folds
    // W(j, .)' x_j into s for the 32 columns next to the diagonal; its helper warp r+2 folds the remaining
    // columns into s2 one step behind.  The pair meets at a named barrier once per step.
    {
        const int rhs = warp & 1;
        double* y = rhs ? V.yb : V.yf;
        double* s1 = rhs ? V.sb : V.sf;
        double* s2 = rhs ? V.sb2 : V.sf2;
        if (warp < 2) {
            for (int j = nt - 1; j >= 0; --j) {
                const int c0 = j << 3;
                const double* Dt = T + tix(j, j) * 64;
                pair_barrier(rhs);
                // every lane redundantly: x_j = L11^-T (v_j - D^-1 (s + s2)_j), unit-lower L11 in the diagonal tile
                double x8[8];
#pragma unroll
                for (int k = 0; k < 8; k += 2) {
                    const double2 yy = *reinterpret_cast<const double2*>(&y[c0 + k]);
                    const double2 sa = *reinterpret_cast<const double2*>(&s1[c0 + k]);
                    const double2 sc = *reinterpret_cast<const double2*>(&s2[c0 + k]);
                    const double2 rr = *reinterpret_cast<const double2*>(&V.rd[c0 + k]);
                    x8[k] = fma(-rr.x, sa.x + sc.x, yy.x);
                    x8[k + 1] = fma(-rr.y, sa.y + sc.y, yy.y);
                }
#pragma unroll
                for (int k = 7; k >= 1; --k) {
#pragma unroll
                    for (int c = 0; c < k; c += 2) {
                        const double2 l2 = *reinterpret_cast<const double2*>(&Dt[el(k, c)]);
                        x8[c] = fma(-l2.x, x8[k], x8[c]);
                        if (c + 1 < k) x8[c + 1] = fma(-l2.y, x8[k], x8[c + 1]);
                    }
                }
                if (lane == 0) {
#pragma unroll
                    for (int k = 0; k < 8; k += 2) *reinterpret_cast<double2*>(&y[c0 + k]) = make_double2(x8[k], x8[k + 1]);
                }
                const int c = c0 - 1 - lane;
                if (c >= 0) {
                    const double* wt = T + tix(j, c >> 3) * 64;
                    const int cc = c & 7;
                    double v = s1[c], v2 = 0.0;
#pragma unroll
                    for (int k = 0; k < 8; k += 2) {
                        v = fma(wt[el(k, cc)], x8[k], v);
                        v2 = fma(wt[el(k + 1, cc)], x8[k + 1], v2);
                    }
                    s1[c] = v + v2;
                }
                __syncwarp();
            }
        } else {
            if (warp == 2 && pf) {  // the caller's output phase reads this next (G of the instance): pull it into L2
                for (int l = lane; l < pf_lines; l += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf + (size_t)l * 128));
            }
            for (int j = nt - 1; j >= 0; --j) {
                pair_barrier(rhs);
                const int jj = j + 1, c1 = jj << 3;  // x_jj is published
                if (jj < nt && c1 > 32) {
                    double x8[8];
#pragma unroll
                    for (int k = 0; k < 8; k += 2) {
                        const double2 xx = *reinterpret_cast<const double2*>(&y[c1 + k]);
                        x8[k] = xx.x;
                        x8[k + 1] = xx.y;
                    }
                    for (int c = c1 - 33 - lane; c >= 0; c -= 32) {
                        const double* wt = T + tix(jj, c >> 3) * 64;
                        const int cc = c & 7;
                        double v = s2[c], v2 = 0.0;
#pragma unroll
                        for (int k = 0; k < 8; k += 2) {
                            v = fma(wt[el(k, cc)], x8[k], v);
                            v2 = fma(wt[el(k + 1, cc)], x8[k + 1], v2);
                        }
                        s2[c] = v + v2;
                    }
                }
            }
        }
    }
}

}  // namespace sqd
