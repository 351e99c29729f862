"""Hard sample points and projection certificates for the power cone K_a = {(x, y, z): x >= 0, y >= 0,
x^a y^(1-a) >= |z|}, shared by the CPU (oracle, host-compiled device header) and GPU (device) tests."""
import math

import numpy as np

ALPHAS = (0.01, 0.1, 0.5, 0.9, 0.99)


def hard_sample(N, alpha, seed=0):
    """N points v with |v| log-uniform in [1e-6, 1e3] and their exponents (``alpha`` a number, or None for exponents
    uniform in [0.02, 0.98]).  Returns (V, a, P): P[i] is the known Pi_K(V[i]) where it is known (NaN elsewhere).

    * a quarter are exact case-4 points v = p + mu g(p), p = (X, Y, +-X^a Y^(1-a)) on the curved boundary with X or Y
      down to 1e-12 |v| and mu > 0 (g = (-a r / X, -(1-a) r / Y, sign z));
    * an eighth have |z0| tiny (1e-14 .. 1e-3) next to a negative x0 or y0;
    * the rest are uniform in direction."""
    rng = np.random.default_rng(seed)
    a = np.full(N, float(alpha)) if alpha is not None else rng.uniform(0.02, 0.98, N)
    V = rng.normal(size=(N, 3))
    P = np.full((N, 3), np.nan)
    k = N // 4
    X = 10.0 ** rng.uniform(-12, 0, k)
    Y = 10.0 ** rng.uniform(-12, 0, k)
    big = rng.integers(0, 2, k) == 0               # one of X, Y at scale 1, the other anywhere down to 1e-12
    X[big] = 10.0 ** rng.uniform(-1, 0, big.sum())
    Y[~big] = 10.0 ** rng.uniform(-1, 0, (~big).sum())
    ak = a[:k]
    r = np.exp(ak * np.log(X) + (1 - ak) * np.log(Y))
    mu = 10.0 ** rng.uniform(-6, 1, k)
    sg = np.where(rng.integers(0, 2, k) == 0, -1.0, 1.0)
    P[:k] = np.stack([X, Y, sg * r], 1)
    V[:k] = np.stack([X - mu * ak * r / X, Y - mu * (1 - ak) * r / Y, sg * (r + mu)], 1)
    k2 = N // 8
    sl = slice(k, k + k2)
    neg_x = rng.integers(0, 2, k2) == 0
    V[sl, 0] = np.where(neg_x, -np.abs(V[sl, 0]), V[sl, 0])
    V[sl, 1] = np.where(neg_x, V[sl, 1], -np.abs(V[sl, 1]))
    V[sl, 2] = 10.0 ** rng.uniform(-14, -3, k2) * np.abs(np.where(neg_x, V[sl, 0], V[sl, 1])) * \
        np.where(rng.integers(0, 2, k2) == 0, -1.0, 1.0)
    scale = 10.0 ** rng.uniform(-6, 3, N) / np.linalg.norm(V, axis=1)
    return V * scale[:, None], a, P * scale[:, None]


def _violation(x, y, z, a, sx, sy):
    """Upper bound on the distance from (x, y, z) to {(x/sx)^a (y/sy)^(1-a) >= |z|, x, y >= 0}: the move onto x, y >= 0
    plus the smallest of the moves along x, along y and along z that enter the set."""
    d = max(-x, 0.0) + max(-y, 0.0)
    x, y, az = max(x, 0.0), max(y, 0.0), abs(z)
    if az == 0.0:
        return d
    lx = math.log(x / sx) if x > 0 else -math.inf
    ly = math.log(y / sy) if y > 0 else -math.inf
    lg = a * lx + (1 - a) * ly
    lz = math.log(az)
    if lg >= lz:
        return d
    along_z = az - math.exp(lg)
    along_x = sx * math.exp(min((lz - (1 - a) * ly) / a, 700.0)) - x if y > 0 else math.inf
    along_y = sy * math.exp(min((lz - a * lx) / (1 - a), 700.0)) - y if x > 0 else math.inf
    return d + min(along_z, along_x, along_y)


def violation_K(p, a):
    return _violation(float(p[0]), float(p[1]), float(p[2]), a, 1.0, 1.0)


def violation_Kdual(u, a):
    return _violation(float(u[0]), float(u[1]), float(u[2]), a, a, 1.0 - a)


def certificate_errors(v, p, a, dual=False):
    """Relative errors of the optimality certificate of p = Pi_K(v) (dual: p = Pi_K*(v)): p in the cone, p - v in
    its dual, <p, p - v> = 0 -- each over |v| (|v|^2 for the inner product)."""
    nv = float(np.linalg.norm(v))
    d = np.asarray(p) - np.asarray(v)
    if dual:
        return violation_Kdual(p, a) / nv, violation_K(d, a) / nv, abs(float(np.dot(p, d))) / nv ** 2
    return violation_K(p, a) / nv, violation_Kdual(d, a) / nv, abs(float(np.dot(p, d))) / nv ** 2
