"""Oracle (test infrastructure, CPU): the exponential cone K = cl{(x, y, z): y > 0, y e^(x/y) <= z} and its dual
K* = cl{(u, v, w): u < 0, -u e^(v/u) <= e w}, and the product-of-cones helpers of ``oracle.cones`` / the conic
gradient cache of ``oracle.conic`` extended to them (every other cone is delegated to ``oracle.cones`` unchanged).

As for every cone, pi projects onto the DUAL of the listed MOI set (``diff_opt.jl:496,515``):

* ``ExponentialCone`` (``EXP``) -> pi onto K* by Moreau, Pi_K*(v) = v + Pi_K(-v) (= -Pi_K°(-v)),
  DPi_K*(v) = I - DPi_K(-v);
* ``DualExponentialCone`` (``DUAL_EXP``) -> pi onto K.

Pi_K(v), v = (r, s, t), cases checked in this order (the order is the tie rule; no reference test reaches a tie):
1. v in K: v, I.  2. v in K° = -K* (r > 0 and r e^(s/r) <= -e t, or r = 0, s <= 0, t <= 0): 0, 0.
3. r <= 0, s <= 0: (r, 0, max(t, 0)), diag(1, 0, [t > 0]).  4. the curved boundary, p = y (rho, 1, e^rho) with rho the
root of Friberg's increasing h (``_exp_project``); DPi_K = leading 3 x 3 block of the inverse of the bordered KKT
matrix of the projection.  MathOptSetDistances implements the same sets; its values at the ties are not pinned here.

Independent of the CUDA arithmetic (``csrc/exp_cone.cuh``): the root by scipy ``brentq`` on the scaled h, the Jacobian
by a 4 x 4 ``numpy.linalg.solve``.  Cone type codes are shared with ``include/diffopt_b200.h``.
"""
from __future__ import annotations

import math

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp
from scipy.optimize import brentq

from oracle import cones
from oracle.cones import NONNEG, PSD, SOC, ZERO, cone_offsets  # noqa: F401  (one module for every cone code)
from oracle.conic import ConicCache

EXP, DUAL_EXP = 4, 5   # DIFFOPT_CONE_EXP / DIFFOPT_CONE_DUAL_EXP in include/diffopt_b200.h


def _xexp(a):
    return math.exp(min(a, 709.0))


def _exp_h_scaled(rho, r, s, t):
    """Friberg's h(rho) = ((rho-1) r + s) e^rho - (r - rho s) e^-rho - (rho^2 - rho + 1) t, times e^-|rho|."""
    e = math.exp(-abs(rho))
    if rho >= 0:
        return ((rho - 1) * r + s) - (r - rho * s) * e * e - (rho * rho - rho + 1) * t * e
    return ((rho - 1) * r + s) * e * e - (r - rho * s) - (rho * rho - rho + 1) * t * e


def exp_case(r, s, t):
    if (s > 0 and s * _xexp(r / s) <= t) or (s == 0 and r <= 0 and t >= 0):
        return 1
    if (r > 0 and r * _xexp(s / r) <= -math.e * t) or (r == 0 and s <= 0 and t <= 0):
        return 2
    if r <= 0 and s <= 0:
        return 3
    return 4


def _exp_root(r, s, t):
    """Root rho of h on the interval where (rho-1) r + s > 0 and r - rho s > 0 (case 4)."""
    lo, hi = -math.inf, math.inf
    if r > 0:
        lo = 1 - s / r
    elif r < 0:
        hi = 1 - s / r
    if s > 0:
        hi = min(hi, r / s)
    elif s < 0:
        lo = max(lo, r / s)
    f = lambda x: _exp_h_scaled(x, r, s, t)  # noqa: E731
    if hi == math.inf:          # one end is open: grow a bracket from the other one
        base, step = max(lo, 0.0), 1.0
        while f(base + step) < 0:
            lo, step = base + step, 2 * step
        hi = base + step
    elif lo == -math.inf:
        base, step = min(hi, 0.0), 1.0
        while f(base - step) > 0:
            hi, step = base - step, 2 * step
        lo = base - step
    flo, fhi = f(lo), f(hi)
    if flo >= 0:
        return lo
    if fhi <= 0:
        return hi
    return brentq(f, lo, hi, xtol=1e-300, rtol=4 * np.finfo(float).eps, maxiter=1000)


def _exp_project(v):
    """(Pi_K(v), Pi_K°(v), (rho, y, w) or None, case) for the exponential cone K.  Case 4: for any rho of the root's interval,
    p = y (rho, 1, e^rho) is in K and q = w (1, 1 - rho, -e^-rho) in K°, orthogonal, and p + q = v but for the
    z-component, which the root settles.  Where y (or w) is tiny that formula has lost its digits, so the pair competes
    with Friberg's heuristic pairs (exact members of K x K°) by the Moreau error max(|p + q - v|, |<p, q>| / |v|)."""
    r, s, t = (float(a) for a in v)
    case = exp_case(r, s, t)
    if case == 1:
        return np.array([r, s, t]), np.zeros(3), None, 1
    if case == 2:
        return np.zeros(3), np.array([r, s, t]), None, 2
    if case == 3:
        return np.array([r, 0.0, max(t, 0.0)]), np.array([0.0, s, min(t, 0.0)]), None, 3
    rho = _exp_root(r, s, t)
    den = rho * rho - rho + 1
    y = max(((rho - 1) * r + s) / den, 0.0)
    w = max((r - rho * s) / den, 0.0)
    pairs = [((min(r, 0.0), 0.0, max(t, 0.0)), (0.0, min(s, 0.0), min(t, 0.0)), None)]
    # y (or w) from its formula cancels where it is tiny: the z-equation y e^rho - w e^-rho = t gives it from the other
    for yy, ww in ((y, w), ((t + w * _xexp(-rho)) * _xexp(-rho), w), (y, (y * _xexp(rho) - t) * _xexp(rho))):
        if yy >= 0 and ww >= 0:
            pz = (yy * math.exp(rho) if rho < 700 else _xexp(rho + math.log(yy))) if yy > 0 else 0.0
            qz = (-ww * math.exp(-rho) if rho > -700 else -_xexp(math.log(ww) - rho)) if ww > 0 else 0.0
            pairs.append(((rho * yy, yy, pz), (ww, (1 - rho) * ww, qz), (yy, ww)))
    if s > 0:
        z = max(t, s * _xexp(r / s))
        pairs.append(((r, s, z), (0.0, 0.0, min(t - z, 0.0)), None))
    if r > 0:
        z = min(t, -r * _xexp(s / r - 1))
        pairs.append(((0.0, 0.0, max(t - z, 0.0)), (r, s, z), None))
    vv = np.array([r, s, t])
    nv = np.linalg.norm(vv)

    def err(pq):   # heuristic pairs (no (y, w)) carry a handicap of 1e-15 |v|: they win only where the root's lost digits
        p, q = np.array(pq[0]), np.array(pq[1])
        with np.errstate(over="ignore", invalid="ignore"):
            e = max(np.linalg.norm(p + q - vv), abs(p @ q) / nv) + (1e-15 * nv if pq[2] is None else 0.0)
        return e if np.isfinite(e) else math.inf
    p, q, _ = min(pairs, key=err)
    yw = min((pq for pq in pairs if pq[2] is not None), key=err, default=(None, None, (y, w)))[2]
    return np.array(p), np.array(q), (rho, *yw), 4


def _exp_jacobian(v):
    """DPi_K(v) for the exponential cone: cases 1-3 in closed form, case 4 by the bordered KKT system of the projection
    p - v + mu grad f(p) = 0, f(p) = y e^(x/y) - z, mu = z - t:  leading 3 x 3 block of [[I + mu Hf, g], [g', 0]]^-1."""
    r, s, t = (float(a) for a in v)
    p, q, root, case = _exp_project(v)
    if case == 1:
        return np.eye(3)
    if case == 2:
        return np.zeros((3, 3))
    if case == 3:
        return np.diag([1.0, 0.0, 1.0 if t > 0 else 0.0])
    rho, y, w = root                            # w = mu e^rho
    a = np.array([1.0, -rho, 0.0])
    # g = (e^rho, e^rho (1 - rho), -1) divided by max(e^rho, 1): the block does not depend on the scale of g
    g = np.array([1.0, 1 - rho, -math.exp(-rho)]) if rho > 0 else np.array([math.exp(rho), math.exp(rho) * (1 - rho), -1.0])
    K = np.zeros((4, 4))
    K[:3, :3] = np.eye(3) + ((w / y) if y > 0 else 1e300) * np.outer(a, a)
    K[:3, 3] = g
    K[3, :3] = g
    rhs = np.zeros((4, 3))
    rhs[:3, :3] = np.eye(3)
    return np.linalg.solve(K, rhs)[:3, :3]



def project(v, ctype):
    """pi of one cone: exponential cones here, every other code through ``oracle.cones.project``."""
    v = np.asarray(v, float)
    if ctype == EXP:        # dual: K*, Pi_K*(v) = -Pi_K°(-v)  (= v + Pi_K(-v))
        return -_exp_project(-v)[1]
    if ctype == DUAL_EXP:   # dual: K
        return _exp_project(v)[0]
    return cones.project(v, ctype)


def project_gradient(v, ctype):
    """Dense Dpi of one cone."""
    v = np.asarray(v, float)
    if ctype == EXP:
        return np.eye(3) - _exp_jacobian(-v)
    if ctype == DUAL_EXP:
        return _exp_jacobian(v)
    return cones.project_gradient(v, ctype)


def apply_gradient(v, ctype, y, transpose=False):
    """Dpi (or Dpi') of one cone applied to y; the exponential blocks are symmetric."""
    if ctype in (EXP, DUAL_EXP):
        return project_gradient(v, ctype) @ np.asarray(y, float)
    return cones.apply_gradient(v, ctype, y, transpose)


def pi(v, cone_types, cone_dims):
    """``DiffOpt.π`` (diff_opt.jl:491-499) over a product of cones."""
    off = cones.cone_offsets(cone_dims)
    out = np.empty(off[-1])
    for c, t in enumerate(cone_types):
        out[off[c]:off[c + 1]] = project(v[off[c]:off[c + 1]], t)
    return out


def Dpi_blocks(v, cone_types, cone_dims):
    """``DiffOpt.Dπ`` (diff_opt.jl:509-519): list of dense blocks."""
    off = cones.cone_offsets(cone_dims)
    return [project_gradient(v[off[c]:off[c + 1]], t) for c, t in enumerate(cone_types)]


def Dpi_dense(v, cone_types, cone_dims):
    return sla.block_diag(*Dpi_blocks(v, cone_types, cone_dims))


def gradient_cache(A, b, c, x, s, y, cone_types, cone_dims):
    """``oracle.conic.gradient_cache`` with exponential cones among the cones; the result feeds ``oracle.conic.forward``,
    ``reverse`` and ``reverse_param_grads`` as is."""
    v = np.asarray(y, float) - np.asarray(s, float)                 # ConicProgram.jl:222
    return assemble_cache(A, b, c, x, s, y, Dpi_blocks(v, cone_types, cone_dims), pi(v, cone_types, cone_dims))


def assemble_cache(A, b, c, x, s, y, blocks, vp):
    """The gradient cache of ``oracle.conic`` from the dense Dpi blocks of every cone and vp = pi(y - s)."""
    A = sp.csc_matrix(A, dtype=np.float64)
    m, n = A.shape
    b = np.asarray(b, float)
    c = np.asarray(c, float)
    x, s, y = (np.asarray(t, float) for t in (x, s, y))
    Dpi = sp.block_diag([sp.csc_matrix(B) for B in blocks], format="csc")
    cc = sp.csc_matrix(c.reshape(n, 1))
    bb = sp.csc_matrix(b.reshape(m, 1))
    M = sp.bmat([                                                    # :243-247
        [sp.csc_matrix((n, n)), A.T @ Dpi, cc],
        [-A, sp.identity(m, format="csc") - Dpi, bb],
        [-cc.T, -(bb.T @ Dpi), sp.csc_matrix((1, 1))],
    ], format="csc")
    return ConicCache(M, vp, Dpi, A, b, c, x, s, y)
