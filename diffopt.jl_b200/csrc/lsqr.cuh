// Persistent cooperative LSQR (Paige-Saunders) over two kinds of linear operator:
//   OP_CSR   : explicit sparse matrix (the QP backend's `lsqr(LHS, RHS)` branch, QuadraticProgram.jl:488)
//   OP_CONIC : matrix-free M = [0 A'Dpi c; -A I-Dpi b; -c' -b'Dpi 0]  (ConicProgram.jl:243-247), used by
//              `lsqr(M, g)` at ConicProgram.jl:323,372 -- the dense Dpi blocks are never formed.
// One kernel runs the whole iteration: vectors stay in L2/HBM, Golub-Kahan scalars live replicated in
// registers, norms are reduced deterministically (per-CTA partials + fixed-order sum), grid.sync()
// separates the phases; there is no host round-trip per iteration.  Large conic operators run the same
// iteration as one kernel per phase (the streaming driver).  Every driver shares one copy of the arithmetic
// in lsqr.cu: the scalar recurrences and stop tests (LsqrScalars), the vector initialisation and deferred
// x / w update, and the row-block phases of M and M'.
#pragma once
#include "common.cuh"

struct CsrView {
    int nrows, ncols;
    const int* rowptr;
    const int* colind;
    const double* val;
    const int* blk;  // row blocks of the streaming SpMV (nblk + 1 entries), see CsrDev
    int nblk;
    // column-ordered copy of every streaming block and each nonzero's CSR slot inside its block (or null)
    const double* sval;
    const int* scol;
    const unsigned short* spos;
};

struct ConicOpView {
    int n, m;
    CsrView A;   // m x n
    CsrView At;  // n x m
    const double *b, *c;
    const double* diag;       // per row: 1 (zero cone -> dual is free), (sign(v)+1)/2 (nonneg); unused on SOC/PSD rows
    const signed char* kind;  // per row: 0 diag row, 2 SOC row, 3 PSD row, 4 + j row j of a 3 x 3 block cone
    const double* blk3;       // rows of 3 x 3 block cones: out[i] = blk3[3i .. 3i+2] . y[first row .. first row + 2]
    int nsoc;
    const int* soc_off;   // first row of each SOC cone
    const int* soc_dim;
    const int* soc_case;  // 0: identity (|x| <= t), 1: zero (|x| <= -t), 2: general
    const double* soc_nx; // |x|
    const double* v;      // y - s (length m)
    // PSD cones (operator form: U (B o (U' X U)) U')
    int npsd;
    const int* psd_off;        // first row
    const int* psd_d;          // side
    const long long* psd_uoff; // offset (in doubles) into U / Bm / work
    const double* psd_U;       // eigenvectors, column-major d x d per cone
    const double* psd_Bm;      // B matrix, d x d per cone
    const int* psd_ident;      // 1 if all eigenvalues >= 0 (Dpi = I)
    const int* psd_toff;       // first 32 x 32 output tile of each cone in the flattened tile list (npsd + 1 entries)
    int psd_ntiles;
    double* psd_w0;            // 3 scratch matrices per cone (d x d each)
    double* psd_w1;
    double* psd_w2;
    double* wc;   // scratch, length m : Dpi * t2   (forward)  /  r = A u1 - u2 - b u3 (transpose)
};

struct LsqrParams {
    double atol, btol, conlim;
    long long maxiter;
};

// Scalars of LSQR (Paige-Saunders, damp = 0): the Golub-Kahan bidiagonalisation with true vectors u = su * u_mem and
// v = sv * v_mem, the plane rotations, the norm and condition estimates and the stop code.  Every driver advances them
// with these methods in the same order: start, first_alpha, then per iteration the stop tests of the previous one,
// next_beta, next_alpha (when beta > 0) and rotate.
struct LsqrScalars {
    double alpha, beta, su, sv, rhobar, phibar, rho, t1, t2, tau;
    double anorm, acond, ddnorm, res2, xnorm, xxnorm, z, sn2, cs2, rnorm, arnorm, bnorm;
    long long itn;
    int istop;

    // beta = ||b|| from ||b||^2; right-hand sides of norm <= zero_below count as zero.  True when v = A'u is to be formed.
    __device__ __forceinline__ bool start(double b2, double zero_below) {
        *this = LsqrScalars{};
        beta = sqrt(b2);
        if (beta <= zero_below) beta = 0.0;
        su = sv = rho = 1.0;
        cs2 = -1.0;
        rnorm = beta;
        if (beta > 0) su = 1.0 / beta;
        return beta > 0;
    }
    // alpha = ||A'u|| from its square (0 when beta = 0) and the start-up values of the recurrences
    __device__ __forceinline__ void first_alpha(double a2) {
        alpha = sqrt(a2);
        if (alpha > 0) sv = 1.0 / alpha;
        arnorm = alpha * beta;
        bnorm = beta;
        rhobar = alpha;
        phibar = beta;
    }
    // stop tests of the iteration rotated last; dd: its share of ddnorm (sum of ||w / rho||^2)
    __device__ __forceinline__ void stop_tests(double dd, const LsqrParams& prm) {
        ddnorm += dd;
        acond = anorm * sqrt(ddnorm);
        const double test1 = rnorm / bnorm;
        const double test2 = arnorm / (anorm * rnorm);
        const double test3 = 1.0 / acond;
        const double t1_ = test1 / (1.0 + anorm * xnorm / bnorm);
        const double rtol = prm.btol + prm.atol * anorm * xnorm / bnorm;
        const double ctol = prm.conlim > 0 ? 1.0 / prm.conlim : 0.0;
        if (itn >= prm.maxiter) istop = 7;
        if (1.0 + test3 <= 1.0) istop = 6;
        if (1.0 + test2 <= 1.0) istop = 5;
        if (1.0 + t1_ <= 1.0) istop = 4;
        if (test3 <= ctol) istop = 3;
        if (test2 <= prm.atol) istop = 2;
        if (test1 <= rtol) istop = 1;
    }
    // next iteration: beta = ||A v - alpha u|| from its square.  True when the next alpha is to be formed.
    __device__ __forceinline__ bool next_beta(double u2) {
        itn += 1;
        beta = sqrt(u2);
        if (beta > 0) {
            su = 1.0 / beta;
            anorm = sqrt(anorm * anorm + alpha * alpha + beta * beta);
        } else {
            su = 1.0;  // u_mem is exactly zero
        }
        return beta > 0;
    }
    // alpha = ||A'u - beta v|| from its square
    __device__ __forceinline__ void next_alpha(double v2) {
        alpha = sqrt(v2);
        sv = alpha > 0 ? 1.0 / alpha : 1.0;
    }
    __device__ __forceinline__ void rotate() {
        const double rhobar1 = rhobar;
        rho = hypot(rhobar1, beta);
        const double cs = rhobar1 / rho, sn = beta / rho;
        const double theta = sn * alpha;
        rhobar = -cs * alpha;
        const double phi = cs * phibar;
        phibar = sn * phibar;
        tau = sn * phi;
        t1 = phi / rho;
        t2 = -theta / rho;
        const double delta = sn2 * rho, gambar = -cs2 * rho, rhs_ = phi - delta * z;
        const double zbar = rhs_ / gambar;
        xnorm = sqrt(xxnorm + zbar * zbar);
        const double gamma = hypot(gambar, theta);
        cs2 = gambar / gamma;
        sn2 = theta / gamma;
        z = rhs_ / gamma;
        xxnorm += z * z;
        rnorm = sqrt(phibar * phibar + res2);
        arnorm = alpha * fabs(tau);
    }
    __device__ __forceinline__ void write_stats(double* stats) const {
        stats[0] = (double)istop;
        stats[1] = (double)itn;
        stats[2] = rnorm;
        stats[3] = arnorm;
        stats[4] = anorm;
        stats[5] = acond;
        stats[6] = xnorm;
    }
};

constexpr int LSQR_NSLOTS = 8;  // partial-sum slots per CTA

struct LsqrVectors {
    double *u, *v, *w, *x;  // lengths nrows, ncols, ncols, ncols
    double* partials;       // [LSQR_NSLOTS][gridDim.x]
    double* stats;          // out: istop, itn, rnorm, arnorm, anorm, acond, xnorm
};

// Work region of one problem of the lock-step batch, offsets in doubles for an operator of order N solved by C CTAs:
// rhs (N + 1) | x, u, v, w (N each) | partial sums (LSQR_NSLOTS * C) | statistics (8).  `stride` (even: every region
// stays 16-byte aligned) separates consecutive problems.
struct LsqrBatchLayout {
    size_t x, u, v, w, partials, stats, stride;
    LsqrBatchLayout(int64_t N, int C)
        : x((size_t)N + 1), u(x + (size_t)N), v(u + (size_t)N), w(v + (size_t)N), partials(w + (size_t)N),
          stats(partials + (size_t)LSQR_NSLOTS * C), stride((stats + 8 + 1) & ~(size_t)1) {}
};

int32_t lsqr_run_csr(diffopt_b200_ctx* ctx, const CsrDev& M, bool trans, const double* rhs_dev, LsqrParams prm,
                     double* x_dev, double* stats_host7);
int32_t lsqr_run_conic(diffopt_b200_ctx* ctx, const double* rhs_dev, LsqrParams prm, double* x_dev,
                       double* stats_host7);
int32_t conic_apply_M(diffopt_b200_ctx* ctx, const double* t_dev, bool transpose, double* out_dev);
int32_t conic_apply_dpi(diffopt_b200_ctx* ctx, const double* t_dev, bool transpose, double* out_dev);
int32_t lsqr_run_conic_batch(diffopt_b200_ctx* ctx, std::vector<ConicState>& states, int C, bool stage, double* work,
                             const LsqrBatchLayout& L, LsqrParams prm, double zero_below, DevBuf& ops_buf, DevBuf& vecs_buf,
                             DevBuf& rhs_buf);
// KB (4 or 8) right-hand sides per group, G groups, against the operator of the current conic_setup (lsqr_multi_kernel):
// rhs, x [G][N][KB] (interleaved), rhs_norm2 [G][KB] (a right-hand side of norm <= zero_below gives x = 0 and zero
// statistics), stats [G][KB][4] = istop, itn, rnorm, arnorm.  Enqueued on ctx->stream between ctx->ev0 and ctx->ev1.
int32_t lsqr_run_conic_multi(diffopt_b200_ctx* ctx, int KB, int64_t G, const double* rhs, const double* rhs_norm2,
                             double zero_below, LsqrParams prm, double* x, double* stats);
int32_t csr_from_csc_host(diffopt_b200_ctx* ctx, int64_t nrows, int64_t ncols, const int64_t* colptr,
                          const int64_t* rowval, const double* nzval, CsrDev& out);
