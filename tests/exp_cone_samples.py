"""Hard sample points and projection certificates for the exponential cone K = cl{(x, y, z): y > 0, y e^(x/y) <= z},
shared by the CPU (oracle) and GPU (device) tests."""
import math

import numpy as np


def hard_sample(N, seed=0):
    """N points v with |v| log-uniform in [1e-6, 1e3]: a quarter built so that Pi_K(v) is on the curved boundary with
    |rho| = |x / y| up to 500 and y down to 1e-12 |v| (next to the ray y = 0), an eighth next to the boundary between
    case 3 (r <= 0, s <= 0) and case 4 (s a tiny positive multiple of |r|), the rest uniform in direction."""
    rng = np.random.default_rng(seed)
    V = rng.normal(size=(N, 3))
    k = N // 4
    rho = rng.uniform(-500, 500, k)
    y = 10.0 ** rng.uniform(-12, 0, k)
    w = 10.0 ** rng.uniform(-6, 1, k)
    P = np.stack([rho * y, y, np.exp(np.minimum(rho + np.log(y), 700.0))], 1)          # on the boundary of K
    Q = w[:, None] * np.stack([np.ones(k), 1 - rho, -np.exp(np.minimum(-rho, 700.0))], 1)  # orthogonal, in the polar
    V[:k] = P + Q
    k2 = N // 8
    V[k:k + k2, 0] = -np.abs(V[k:k + k2, 0])
    V[k:k + k2, 1] = 10.0 ** rng.uniform(-14, -3, k2) * np.abs(V[k:k + k2, 0])
    V = V[np.all(np.isfinite(V), 1) & (np.abs(V).max(axis=1) > 0)]
    V /= np.abs(V).max(axis=1)[:, None]
    V /= np.linalg.norm(V, axis=1)[:, None]
    return V * (10.0 ** rng.uniform(-6, 3, len(V)))[:, None]


def violation_K(p):
    """Upper bound on the distance from p to K: the smaller of the moves along x and along z that enter K."""
    x, y, z = (float(a) for a in p)
    if y < 0:
        return -y + violation_K((x, 0.0, z))
    if y == 0:
        return max(x, 0.0) + max(-z, 0.0)
    along_z = max(0.0, y * math.exp(min(x / y, 700.0)) - z)
    along_x = max(0.0, x - y * math.log(z / y)) if z > 0 else math.inf
    return min(along_z, along_x)


def violation_Kdual(u):
    """K* = {(u, v, w): (u - v, -u, w) in K}."""
    return violation_K((u[0] - u[1], -u[0], u[2]))


def certificate_errors(v, p, dual=False):
    """Relative errors of the optimality certificate of p = Pi_K(v) (dual: p = Pi_K*(v)): p in the cone, p - v in
    its dual, <p, p - v> = 0 -- each over |v| (|v|^2 for the inner product)."""
    nv = float(np.linalg.norm(v))
    d = np.asarray(p) - np.asarray(v)
    if dual:
        return violation_Kdual(p) / nv, violation_K(d) / nv, abs(float(np.dot(p, d))) / nv ** 2
    return violation_K(p) / nv, violation_Kdual(d) / nv, abs(float(np.dot(p, d))) / nv ** 2
