// Power cone K_a = {(x, y, z) : x >= 0, y >= 0, x^a y^(1-a) >= |z|}, 0 < a < 1: projection Pi_K(v), the polar part
// Pi_K°(v) = v - Pi_K(v) and the symmetric 3 x 3 Jacobian DPi_K(v), one thread per cone (cone_pow_kernel).
// The dual cone is K* = {(u, v, w) : u >= 0, v >= 0, (u/a)^a (v/(1-a))^(1-a) >= |w|}, the polar cone K° = -K*.
//
// v = (x0, y0, z0); cases in this order (the order fixes the value at ties):
//   1. v in K                                     -> p = v,                     D = I
//   2. v in K° (x0 <= 0, y0 <= 0,                 -> p = 0,                     D = 0
//      (-x0/a)^a (-y0/(1-a))^(1-a) >= |z0|)
//   3. z0 = 0                                     -> p = (x0+, y0+, 0),         D = diag([x0 > 0], [y0 > 0], 0)
//   4. otherwise p lies on the curved boundary (N. T. V. Hien, "Differential properties of Euclidean projection onto
//      power cone", 2015): p = (X(r), Y(r), sign(z0) r), v - p = mu (-a r / X, -(1-a) r / Y, sign(z0)), mu = |z0| - r,
//      X(r) = (x0 + sqrt(x0^2 + 4 a r mu)) / 2, Y(r) = (y0 + sqrt(y0^2 + 4 (1-a) r mu)) / 2 and r in (0, |z0|) the root
//      of the decreasing psi(r) = a log X + (1-a) log Y - log r.  For every r of that interval <p, v - p> = 0 exactly
//      and only the membership of p in K (and of v - p in K°) needs the root.  The root is found in t = log(r / |z0|)
//      (r may lie hundreds of decades below |v| when |z0| is tiny and a is close to 0 or 1) by Newton's method
//      safeguarded by a bracket; X, Y and psi are evaluated through their logarithms, with X = 2 a r mu / (s - x0)
//      where x0 <= 0 (no cancellation next to an axis, no underflow of X).
//   Jacobian of case 4: implicit differentiation of p - v + mu grad f(p) = 0, f(p) = |z| - x^a y^(1-a):
//   DPi_K = M^-1 - M^-1 g g' M^-1 / (g' M^-1 g), g = (-a r / X, -(1-a) r / Y, sign z0), M = I + c b b',
//   b = (1/X, -1/Y, 0), c = mu r a (1-a).  M^-1 = I - w h h' with h = (Y, -X, 0) / |(X, Y)| and
//   w = 1 / (1 + (X Y / |(X, Y)|)^2 / c); g is scaled by its largest magnitude (D does not depend on the scale of g).
#pragma once
#include <math.h>

#include "exp_cone.cuh"

// One side (x with exponent a, or y with exponent 1 - a) of the case-4 boundary point at r = e^lr, mu = e^lmu:
// X, log X, log of s = sqrt(x0^2 + 4 a r mu), and the polar component x0 - X.
__host__ __device__ inline void pow_cone_side(double x0, double a, double lr, double lmu, double& X, double& lX,
                                              double& ls, double& qx) {
    const double lphi = log(4.0 * a) + lr + lmu;            // log(4 a r mu)
    const double sphi = exp(0.5 * lphi);
    if (x0 > 0.0) {
        const double s = hypot(x0, sphi);
        X = 0.5 * (x0 + s);
        lX = log(X);
        ls = log(s);
        qx = -exp(lphi - log(2.0 * (s + x0)));              // x0 - X = -4 a r mu / (2 (s + x0))
    } else if (x0 < 0.0) {
        const double s = hypot(x0, sphi);
        lX = lphi - log(2.0 * (s - x0));                    // X = 4 a r mu / (2 (s - x0))
        X = exp(lX);
        ls = log(s);
        qx = 0.5 * (x0 - s);
    } else {
        lX = 0.5 * (lphi - log(4.0));                       // X = sqrt(a r mu)
        X = exp(lX);
        ls = log(2.0) + lX;
        qx = -X;
    }
}

// psi at t = log(r / |z0|) and d psi / dt, with the boundary point's pieces
struct PowConeEval {
    double psi, dpsi, X, Y, lX, lY, qx, qy;
};

__host__ __device__ inline PowConeEval pow_cone_psi(double t, double x0, double y0, double lz, double az, double alpha) {
    PowConeEval e;
    const double lr = lz + t;
    const double lmu = lz + log(-expm1(t));
    double lsx, lsy;
    pow_cone_side(x0, alpha, lr, lmu, e.X, e.lX, lsx, e.qx);
    pow_cone_side(y0, 1.0 - alpha, lr, lmu, e.Y, e.lY, lsy, e.qy);
    e.psi = alpha * e.lX + (1.0 - alpha) * e.lY - lr;
    // r dX/dr / X = a^2 r (mu - r) / (s X), the same for Y
    const double mr = -az * (expm1(t) + exp(t));            // mu - r
    e.dpsi = alpha * alpha * mr * exp(lr - e.lX - lsx) + (1.0 - alpha) * (1.0 - alpha) * mr * exp(lr - e.lY - lsy) - 1.0;
    return e;
}

// p = Pi_K(v), q = v - Pi_K(v) (the polar part, in K°), D = DPi_K(v) row-major (symmetric).  Returns the number of
// evaluations of psi (0 in cases 1-3).
__host__ __device__ inline int pow_cone_project(double x0, double y0, double z0, double alpha, double* p, double* q,
                                                double* D) {
    for (int k = 0; k < 9; ++k) D[k] = 0.0;
    const double az = fabs(z0);
    // case 1: v in K
    if (x0 >= 0.0 && y0 >= 0.0 && pow(x0, alpha) * pow(y0, 1.0 - alpha) >= az) {
        p[0] = x0; p[1] = y0; p[2] = z0;
        q[0] = q[1] = q[2] = 0.0;
        D[0] = D[4] = D[8] = 1.0;
        return 0;
    }
    // case 2: v in the polar cone
    if (x0 <= 0.0 && y0 <= 0.0 && pow(-x0 / alpha, alpha) * pow(-y0 / (1.0 - alpha), 1.0 - alpha) >= az) {
        p[0] = p[1] = p[2] = 0.0;
        q[0] = x0; q[1] = y0; q[2] = z0;
        return 0;
    }
    // case 3
    if (z0 == 0.0) {
        p[0] = fmax(x0, 0.0); p[1] = fmax(y0, 0.0); p[2] = 0.0;
        q[0] = fmin(x0, 0.0); q[1] = fmin(y0, 0.0); q[2] = 0.0;
        D[0] = x0 > 0.0 ? 1.0 : 0.0;
        D[4] = y0 > 0.0 ? 1.0 : 0.0;
        return 0;
    }
    // case 4.  psi(t) falls from psi(-inf) > 0 (not case 2) to psi(0-) < 0 (not case 1).  hi starts at the negative
    // number closest to 0 (mu = -|z0| expm1(t) carries its relative accuracy only while t does: next to K the root is
    // at t ~ -mu / |z0|, hundreds of decades below 1), lo is found by doubling the step downwards
    const double lz = log(az);
    double lo = -INFINITY, hi = -4.9406564584124654e-324;
    int evals = 0;
    PowConeEval e;
    for (double b = -1.0; b >= -4096.0; b *= 2.0) {
        e = pow_cone_psi(b, x0, y0, lz, az, alpha);
        ++evals;
        if (e.psi >= 0.0) { lo = b; break; }
        hi = b;
    }
    // (psi < 0 down to t = -4096: r and the X, Y it ties to z are far below the rounding level of |v|)
    if (lo == -INFINITY) lo = hi;
    // safeguarded Newton (rtsafe) on G = -psi, increasing in t; its bisection steps are geometric while the bracket
    // spans more than a factor of 4 (the root may be anywhere in [-1, -5e-324]), and the stop test is relative
    auto bisect = [](double a, double b) { return a < 4.0 * b ? -sqrt(-a) * sqrt(-b) : 0.5 * (a + b); };
    double t = bisect(lo, hi), dx = hi - lo;
    for (int it = 0; it < 200 && lo < hi; ++it) {
        e = pow_cone_psi(t, x0, y0, lz, az, alpha);
        ++evals;
        const double G = -e.psi, Gp = -e.dpsi;
        if (G == 0.0) break;
        if (G < 0.0) lo = t; else hi = t;
        const double nt = t - G / Gp, dxo = dx;
        if (!(Gp > 0.0) || !(nt > lo && nt < hi) || fabs(2.0 * G) > fabs(dxo * Gp)) {
            const double tb = bisect(lo, hi);
            dx = tb - t;
            t = tb;
        } else {
            dx = G / Gp;
            t = nt;
        }
        if (fabs(dx) <= 2e-16 * fabs(t)) break;
    }
    e = pow_cone_psi(t, x0, y0, lz, az, alpha);
    const double sg = z0 > 0.0 ? 1.0 : -1.0;
    const double lr = lz + t, lmu = lz + log(-expm1(t));
    p[0] = e.X; p[1] = e.Y; p[2] = sg * az * exp(t);
    q[0] = e.qx; q[1] = e.qy; q[2] = -sg * az * expm1(t);
    // Jacobian.  (hx, hy) = (X, Y) / max(X, Y) and beta = (X Y / |(X, Y)|)^2 / c from logarithms (X or Y may
    // underflow); M^-1 = I - w h h' written as (I - h h') + (1 - w) h h' so that nothing cancels where beta << 1
    const double lm = fmax(e.lX, e.lY);
    const double hx = exp(e.lX - lm), hy = exp(e.lY - lm), hn2 = hx * hx + hy * hy;
    const double lxy = e.lX + e.lY - lm - 0.5 * log(hn2);   // log(X Y / |(X, Y)|)
    // 1 / beta, at most 1e300: where beta underflows (X or Y hundreds of decades below |v|) g collapses onto that axis
    // too, and a floor of 1e-300 keeps g' M^-1 g > 0 with the limit D = I - e e' of that axis
    const double ib = fmin(exp(lmu + lr + log(alpha * (1.0 - alpha)) - 2.0 * lxy), 1e300);
    const double w = 1.0 / (1.0 + 1.0 / ib), wb = 1.0 / (1.0 + ib);
    const double Mi[9] = {(hx * hx + wb * hy * hy) / hn2, w * hx * hy / hn2, 0.0,
                          w * hx * hy / hn2, (hy * hy + wb * hx * hx) / hn2, 0.0,
                          0.0, 0.0, 1.0};
    const double l0 = log(alpha) + lr - e.lX, l1 = log(1.0 - alpha) + lr - e.lY, lg = fmax(fmax(l0, l1), 0.0);
    const double g[3] = {-exp(l0 - lg), -exp(l1 - lg), sg * exp(-lg)};
    sym3_bordered_block(Mi, g, D);
    return evals;
}

#ifdef __CUDACC__
// One thread per power cone: vp of the cone's three rows and its Dpi block in the layout of cone_exp_kernel (row i of
// the cone holds blk[3 i .. 3 i + 2]).  neg[c] != 0 (PowerCone listed, pi onto K*): Pi_K*(v) = -Pi_K°(-v),
// DPi_K*(v) = I - DPi_K(-v).  alpha[c] is the cone's exponent; `iters` (optional) receives the evaluations of psi.
__global__ void cone_pow_kernel(int ncones, const int* __restrict__ off, const signed char* __restrict__ neg,
                                const double* __restrict__ alpha, const double* __restrict__ v, double* vp, double* blk,
                                int* iters) {
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < ncones; c += gridDim.x * blockDim.x) {
        const int o = off[c];
        const bool ng = neg[c] != 0;
        const double sg = ng ? -1.0 : 1.0;
        double p[3], q[3], D[9];
        const int ev = pow_cone_project(sg * v[o], sg * v[o + 1], sg * v[o + 2], alpha[c], p, q, D);
        for (int k = 0; k < 3; ++k) vp[o + k] = ng ? -q[k] : p[k];
        for (int k = 0; k < 9; ++k) blk[3 * (long long)o + k] = ng ? (k % 4 == 0 ? 1.0 : 0.0) - D[k] : D[k];
        if (iters) iters[c] = ev;
    }
}
#endif
