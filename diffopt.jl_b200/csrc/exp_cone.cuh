// Exponential cone K = cl{(x, y, z) : y > 0, y e^(x/y) <= z}: projection Pi_K(v), the polar part Pi_K°(v) = v - Pi_K(v)
// and the symmetric 3 x 3 Jacobian DPi_K(v), one thread per cone (cone_exp_kernel).
//
// v = (r, s, t); cases in this order (the order fixes the value at ties):
//   1. v in K                                    -> p = v,                 D = I
//   2. v in K° = -K* (r > 0, r e^(s/r) <= -e t;  -> p = 0,                 D = 0
//      or r = 0, s <= 0, t <= 0)
//   3. r <= 0, s <= 0                            -> p = (r, 0, max(t, 0)), D = diag(1, 0, [t > 0])
//   4. otherwise p lies on the curved boundary: p = y (rho, 1, e^rho), v - p = w (1, 1 - rho, -e^-rho), with
//      y = ((rho-1) r + s) / (rho^2 - rho + 1), w = (r - rho s) / (rho^2 - rho + 1) and rho the root of the increasing
//      h(rho) = ((rho-1) r + s) e^rho - (r - rho s) e^-rho - (rho^2 - rho + 1) t on the interval where y > 0 and w > 0
//      (H. A. Friberg, "Projection onto the exponential cone: a univariate root-finding problem").  For every rho of
//      that interval p is in K, v - p in K° and <p, v - p> = 0 exactly; only the z-components of p + (v - p) = v need
//      the root.  h is evaluated scaled by e^-|rho| (no overflow for any rho), the root found by Newton's method
//      safeguarded by a bracket, and the root's pair (p, v - p) competes with Friberg's
//      heuristic pairs by their Moreau error -- those win where y (or w) is so small that the root's formula has lost
//      its digits (projection next to the ray y = 0, large |rho|).
//   Jacobian of case 4: implicit differentiation of p - v + mu grad f(p) = 0, f(p) = y e^(x/y) - z = 0, mu = z - t:
//   DPi_K = leading 3 x 3 block of [[I + mu H, g], [g', 0]]^-1, g = (e^rho, e^rho (1 - rho), -1),
//   mu H = (w / y) a a', a = (1, -rho, 0); closed form M^-1 - M^-1 g g' M^-1 / (g' M^-1 g), M = I + mu H
//   (Sherman-Morrison), with g scaled by 1 / max(e^rho, 1) (D does not depend on the scale of g).
#pragma once
#include <math.h>

#ifndef __CUDACC__
#define __host__
#define __device__
#endif

// Leading 3 x 3 block of [[M, g], [g', 0]]^-1 from Mi = M^-1 (symmetric): D = Mi - Mi g g' Mi / (g' Mi g).  The
// projection Jacobian of every cone with one curved boundary surface f = 0 (exponential, power).
__host__ __device__ inline void sym3_bordered_block(const double* Mi, const double* g, double* D) {
    double u[3];
    for (int i = 0; i < 3; ++i) u[i] = Mi[3 * i] * g[0] + Mi[3 * i + 1] * g[1] + Mi[3 * i + 2] * g[2];
    const double gu = g[0] * u[0] + g[1] * u[1] + g[2] * u[2];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) D[3 * i + j] = Mi[3 * i + j] - u[i] * u[j] / gu;
}

// scaled h and h' at rho: both times e^-|rho|, so G / Gp is the Newton step of h
__host__ __device__ inline void exp_cone_h(double rho, double r, double s, double t, double& G, double& Gp) {
    const double a = (rho - 1.0) * r + s, b = r - rho * s, q = rho * rho - rho + 1.0;
    const double ap = rho * r + s, bp = b + s, qp = 2.0 * rho - 1.0;
    if (rho >= 0.0) {
        const double e = exp(-rho);
        G = a - b * e * e - q * t * e;
        Gp = ap + bp * e * e - qp * t * e;
    } else {
        const double e = exp(rho);
        G = a * e * e - b - q * t * e;
        Gp = ap * e * e + bp - qp * t * e;
    }
}

// p = Pi_K(v), q = v - Pi_K(v) (the polar part, in K°), D = DPi_K(v) row-major (symmetric).  Returns the number of
// evaluations of h (0 in cases 1-3).
__host__ __device__ inline int exp_cone_project(double r, double s, double t, double* p, double* q, double* D) {
    for (int k = 0; k < 9; ++k) D[k] = 0.0;
    // case 1: v in K
    if ((s > 0.0 && s * exp(r / s) <= t) || (s == 0.0 && r <= 0.0 && t >= 0.0)) {
        p[0] = r; p[1] = s; p[2] = t;
        q[0] = q[1] = q[2] = 0.0;
        D[0] = D[4] = D[8] = 1.0;
        return 0;
    }
    // case 2: v in the polar cone
    if ((r > 0.0 && r * exp(s / r) <= -2.718281828459045 * t) || (r == 0.0 && s <= 0.0 && t <= 0.0)) {
        p[0] = p[1] = p[2] = 0.0;
        q[0] = r; q[1] = s; q[2] = t;
        return 0;
    }
    // case 3
    if (r <= 0.0 && s <= 0.0) {
        p[0] = r; p[1] = 0.0; p[2] = t > 0.0 ? t : 0.0;
        q[0] = 0.0; q[1] = s; q[2] = t > 0.0 ? 0.0 : t;
        D[0] = 1.0;
        D[8] = t > 0.0 ? 1.0 : 0.0;
        return 0;
    }
    // case 4: bracket [lo, hi] of the interval where y > 0 and w > 0 (one end may be infinite)
    double lo = -INFINITY, hi = INFINITY;
    if (r > 0.0) lo = 1.0 - s / r;
    else if (r < 0.0) hi = 1.0 - s / r;
    if (s > 0.0) hi = fmin(hi, r / s);
    else if (s < 0.0) lo = fmax(lo, r / s);
    int evals = 0;
    double G, Gp;
    if (hi == INFINITY) {  // grow the bracket upwards: h(hi) >= 0 ends it
        const double base = fmax(lo, 0.0);
        for (double step = 1.0; evals < 64; step *= 2.0) {
            const double b = base + step;
            exp_cone_h(b, r, s, t, G, Gp);
            ++evals;
            if (G >= 0.0) { hi = b; break; }
            lo = b;
        }
        if (hi == INFINITY) hi = lo;  // (not reached for finite v)
    } else if (lo == -INFINITY) {
        const double base = fmin(hi, 0.0);
        for (double step = 1.0; evals < 64; step *= 2.0) {
            const double b = base - step;
            exp_cone_h(b, r, s, t, G, Gp);
            ++evals;
            if (G <= 0.0) { lo = b; break; }
            hi = b;
        }
        if (lo == -INFINITY) lo = hi;
    }
    // safeguarded Newton (rtsafe): the bracket shrinks at every evaluation; a step that leaves it, or that would not
    // halve the step before last, is replaced by bisection
    double rho = 0.5 * (lo + hi), dxo = hi - lo, dx = dxo;
    for (int it = 0; it < 100 && lo < hi; ++it) {
        exp_cone_h(rho, r, s, t, G, Gp);
        ++evals;
        if (G == 0.0) break;
        if (G < 0.0) lo = rho; else hi = rho;
        const double nr = rho - G / Gp;
        dxo = dx;
        if (!(Gp > 0.0) || !(nr > lo && nr < hi) || fabs(2.0 * G) > fabs(dxo * Gp)) {
            dx = 0.5 * (hi - lo);
            rho = lo + dx;
        } else {
            dx = G / Gp;
            rho = nr;
        }
        if (fabs(dx) <= 2e-16 * fmax(1.0, fabs(rho))) break;
    }
    const double den = rho * rho - rho + 1.0;
    const double y = fmax(((rho - 1.0) * r + s) / den, 0.0);
    const double w = fmax((r - rho * s) / den, 0.0);
    // pairs (p in K, q in K°), exact members of their sets; the one with the smallest Moreau error
    // max(|p + q - v|, |<p, q>| / |v|) is kept.  The root's pairs are exactly orthogonal; Friberg's heuristic pairs are
    // ((r-, 0, t+), (0, s-, t-)), ((r, s, max(t, s e^(r/s))), (0, 0, <= 0)) for s > 0 and
    // ((0, 0, >= 0), (r, s, min(t, -r e^(s/r - 1)))) for r > 0.
    const double nv = sqrt(r * r + s * s + t * t);
    double best = INFINITY;
    // (a heuristic pair carries a handicap of 1e-15 |v|, the rounding level of the root's pairs: it replaces them only
    // where they have lost digits, so the projection stays smooth wherever the root's formula is accurate)
    auto take = [&](double p0, double p1, double p2, double q0, double q1, double q2, double handicap) {
        const double e0 = p0 + q0 - r, e1 = p1 + q1 - s, e2 = p2 + q2 - t;
        const double err = fmax(sqrt(e0 * e0 + e1 * e1 + e2 * e2), fabs(p0 * q0 + p1 * q1 + p2 * q2) / nv) + handicap;
        if (err < best) {
            best = err;
            p[0] = p0; p[1] = p1; p[2] = p2;
            q[0] = q0; q[1] = q1; q[2] = q2;
        }
        return err;
    };
    // y (or w) from its formula cancels where it is tiny; the z-equation y e^rho - w e^-rho = t then gives it from the
    // other one.  The Jacobian takes (y, w) of the most accurate of these pairs.
    double yb = y, wb = w, eb = INFINITY;
    auto root_pair = [&](double yy, double ww) {
        if (!(yy >= 0.0 && ww >= 0.0)) return;
        // (y e^rho as a product while e^rho is finite: exp(rho + log y) rounds rho + log y absolutely)
        const double pz = yy > 0.0 ? (rho < 700.0 ? yy * exp(rho) : exp(rho + log(yy))) : 0.0;
        const double qz = ww > 0.0 ? (rho > -700.0 ? -ww * exp(-rho) : -exp(log(ww) - rho)) : 0.0;
        const double e = take(rho * yy, yy, pz, ww, (1.0 - rho) * ww, qz, 0.0);
        if (e < eb) { eb = e; yb = yy; wb = ww; }
    };
    root_pair(y, w);
    root_pair((t + w * exp(-rho)) * exp(-rho), w);
    root_pair(y, (y * exp(rho) - t) * exp(rho));
    const double hc = 1e-15 * nv;
    take(fmin(r, 0.0), 0.0, fmax(t, 0.0), 0.0, fmin(s, 0.0), fmin(t, 0.0), hc);
    if (s > 0.0) {
        const double z = fmax(t, s * exp(r / s));
        take(r, s, z, 0.0, 0.0, fmin(t - z, 0.0), hc);
    }
    if (r > 0.0) {
        const double z = fmin(t, -r * exp(s / r - 1.0));
        take(0.0, 0.0, fmax(t - z, 0.0), r, s, z, hc);
    }
    // Jacobian.  M^-1 = I - a a' / kappa with kappa = y / w + 1 + rho^2, written without cancellation
    const double kappa = (wb > 0.0 ? yb / wb : INFINITY) + 1.0 + rho * rho;
    double Mi[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0};
    if (kappa < INFINITY) {   // (w == 0: mu H = 0, M = I)
        const double yw = yb / wb;
        Mi[0] = (yw + rho * rho) / kappa;
        Mi[1] = Mi[3] = rho / kappa;
        Mi[4] = (yw + 1.0) / kappa;
    } else {
        Mi[0] = Mi[4] = 1.0;
    }
    const double sc = rho > 0.0 ? exp(-rho) : 1.0, er = rho > 0.0 ? 1.0 : exp(rho);
    const double g[3] = {er, er * (1.0 - rho), -sc};
    sym3_bordered_block(Mi, g, D);
    return evals;
}

#ifdef __CUDACC__
// One thread per cone of a 3 x 3 block kind (exponential / dual exponential): vp of the cone's three rows and its
// Dpi block, stored by row -- row i of the cone holds blk[3 i .. 3 i + 2], so the 9 coefficients of a cone whose first
// row is o sit at blk[3 o .. 3 o + 8], row-major.  neg[c] != 0 (DualExponentialCone listed, pi onto K*):
// Pi_K*(v) = -Pi_K°(-v), DPi_K*(v) = I - DPi_K(-v).  `iters` (optional) receives the evaluations of h per cone.
__global__ void cone_exp_kernel(int ncones, const int* __restrict__ off, const signed char* __restrict__ neg,
                                const double* __restrict__ v, double* vp, double* blk, int* iters) {
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < ncones; c += gridDim.x * blockDim.x) {
        const int o = off[c];
        const bool ng = neg[c] != 0;
        const double sg = ng ? -1.0 : 1.0;
        double p[3], q[3], D[9];
        const int ev = exp_cone_project(sg * v[o], sg * v[o + 1], sg * v[o + 2], p, q, D);
        for (int k = 0; k < 3; ++k) vp[o + k] = ng ? -q[k] : p[k];
        for (int k = 0; k < 9; ++k) blk[3 * (long long)o + k] = ng ? (k % 4 == 0 ? 1.0 : 0.0) - D[k] : D[k];
        if (iters) iters[c] = ev;
    }
}
#endif
