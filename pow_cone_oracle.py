"""Oracle (test infrastructure, CPU): the power cone K_a = {(x, y, z): x >= 0, y >= 0, x^a y^(1-a) >= |z|}, 0 < a < 1,
and its dual K_a* = {(u, v, w): u >= 0, v >= 0, (u/a)^a (v/(1-a))^(1-a) >= |w|}, with the product-of-cones helpers and
the conic gradient cache extended to them (exponential cones go to ``exp_cone_oracle``, every other cone to
``oracle.cones``).  Power cones carry their exponent a in ``cone_params`` (one entry per cone, read for codes 6 and 7).

As for every cone, pi projects onto the DUAL of the listed MOI set (``diff_opt.jl:496,515``):

* ``PowerCone(a)`` (``POW``) -> pi onto K* by Moreau, Pi_K*(v) = v + Pi_K(-v), DPi_K*(v) = I - DPi_K(-v);
* ``DualPowerCone(a)`` (``DUAL_POW``) -> pi onto K.

Pi_K(v), v = (x0, y0, z0), cases checked in this order (the order is the tie rule; no reference test reaches a tie):
1. v in K: v, I.  2. v in K° = -K*: 0, 0.  3. z0 = 0: (x0+, y0+, 0), diag([x0 > 0], [y0 > 0], 0).
4. the curved boundary, p = (X(r), Y(r), sign(z0) r), X(r) = (x0 + sqrt(x0^2 + 4 a r (|z0| - r))) / 2 (Y with 1 - a),
r the root in (0, |z0|) of psi(r) = a log X + (1-a) log Y - log r (Hien 2015); DPi_K = leading 3 x 3 block of the inverse
of the bordered KKT matrix of the projection.  MathOptSetDistances implements the same sets; its values at the ties
are not pinned here.

Independent of the CUDA arithmetic (``csrc/pow_cone.cuh``, which runs Newton's method in log r): the root by scipy
``brentq`` on psi in r, the Jacobian by a 4 x 4 ``numpy.linalg.solve``.  Cone type codes are shared with
``include/diffopt_b200.h``.
"""
from __future__ import annotations

import math

import numpy as np
import scipy.linalg as sla
from scipy.optimize import brentq

import exp_cone_oracle as oexp
from oracle import cones
from oracle.cones import NONNEG, PSD, SOC, ZERO, cone_offsets  # noqa: F401  (one module for every cone code)

EXP, DUAL_EXP = oexp.EXP, oexp.DUAL_EXP
POW, DUAL_POW = 6, 7   # DIFFOPT_CONE_POW / DIFFOPT_CONE_DUAL_POW in include/diffopt_b200.h


def _log(a):
    return math.log(a) if a > 0 else -math.inf


def pow_case(x0, y0, z0, a):
    az = abs(z0)
    if x0 >= 0 and y0 >= 0 and a * _log(x0) + (1 - a) * _log(y0) >= _log(az):
        return 1
    if x0 <= 0 and y0 <= 0 and a * _log(-x0 / a) + (1 - a) * _log(-y0 / (1 - a)) >= _log(az):
        return 2
    if z0 == 0:
        return 3
    return 4


def _side(x0, a, r, mu):
    """X and x0 - X at r, mu = |z0| - r (no cancellation: X = phi / (2 (s - x0)) where x0 <= 0), and log X."""
    phi = 4 * a * r * mu
    s = math.hypot(x0, math.sqrt(phi))
    if x0 > 0:
        X = 0.5 * (x0 + s)
        return X, -phi / (2 * (s + x0)), math.log(X)
    if s - x0 > 0 and r > 0 and mu > 0:
        lX = math.log(4 * a) + math.log(r) + math.log(mu) - math.log(2 * (s - x0))
        return math.exp(lX), 0.5 * (x0 - s), lX
    return 0.0, 0.5 * (x0 - s), -math.inf


def _psi(r, x0, y0, az, a):
    mu = az - r
    lX = _side(x0, a, r, mu)[2]
    lY = _side(y0, 1 - a, r, mu)[2]
    return a * lX + (1 - a) * lY - math.log(r)


def _pow_root(x0, y0, z0, a):
    """r in (0, |z0|) with psi(r) = 0 (case 4); psi falls from > 0 at 0+ to < 0 at |z0|-.  0.0 where the root is below
    the smallest double."""
    az = abs(z0)
    f = lambda r: max(min(_psi(r, x0, y0, az, a), 1e300), -1e300)  # noqa: E731
    hi, k = az, 1
    while True:                 # lo = |z0| / 2^k, k = 1, 2, 4, ...: the first with psi(lo) >= 0
        lo = math.ldexp(az, -k)
        if lo == 0.0:
            return 0.0
        if f(lo) >= 0:
            break
        hi, k = lo, 2 * k
    if f(lo) == 0:
        return lo
    return brentq(f, lo, hi, xtol=1e-320, rtol=4 * np.finfo(float).eps, maxiter=2000)


def _pow_project(v, a):
    """(Pi_K(v), Pi_K°(v), r, case) for the power cone K_a."""
    x0, y0, z0 = (float(t) for t in v)
    case = pow_case(x0, y0, z0, a)
    if case == 1:
        return np.array([x0, y0, z0]), np.zeros(3), None, 1
    if case == 2:
        return np.zeros(3), np.array([x0, y0, z0]), None, 2
    if case == 3:
        return np.array([max(x0, 0.0), max(y0, 0.0), 0.0]), np.array([min(x0, 0.0), min(y0, 0.0), 0.0]), None, 3
    r = _pow_root(x0, y0, z0, a)
    az = abs(z0)
    mu = az - r
    X, qx, _ = _side(x0, a, r, mu)
    Y, qy, _ = _side(y0, 1 - a, r, mu)
    sg = math.copysign(1.0, z0)
    return np.array([X, Y, sg * r]), np.array([qx, qy, sg * mu]), r, 4


def _pow_jacobian(v, a):
    """DPi_K(v): cases 1-3 in closed form, case 4 by the bordered KKT system of p - v + mu grad f(p) = 0,
    f = |z| - x^a y^(1-a), mu = |z0| - r: leading 3 x 3 block of [[I + mu Hf, g], [g', 0]]^-1."""
    x0, y0, z0 = (float(t) for t in v)
    p, q, r, case = _pow_project(v, a)
    if case == 1:
        return np.eye(3)
    if case == 2:
        return np.zeros((3, 3))
    if case == 3:
        return np.diag([1.0 if x0 > 0 else 0.0, 1.0 if y0 > 0 else 0.0, 0.0])
    X, Y = p[0], p[1]
    mu = abs(z0) - r
    g = np.array([-a * r / X, -(1 - a) * r / Y, math.copysign(1.0, z0)])
    g /= np.abs(g).max()                      # the block does not depend on the scale of g
    bvec = np.array([1.0 / X, -1.0 / Y, 0.0])
    K = np.zeros((4, 4))
    K[:3, :3] = np.eye(3) + mu * r * a * (1 - a) * np.outer(bvec, bvec)
    K[:3, 3] = g
    K[3, :3] = g
    rhs = np.zeros((4, 3))
    rhs[:3, :3] = np.eye(3)
    return np.linalg.solve(K, rhs)[:3, :3]


def _param(cone_params, c):
    return None if cone_params is None else float(cone_params[c])


def project(v, ctype, param=None):
    """pi of one cone: power cones here (param = the exponent), every other code through ``exp_cone_oracle``."""
    v = np.asarray(v, float)
    if ctype == POW:        # dual: K*, Pi_K*(v) = -Pi_K°(-v)
        return -_pow_project(-v, param)[1]
    if ctype == DUAL_POW:   # dual: K
        return _pow_project(v, param)[0]
    return oexp.project(v, ctype)


def project_gradient(v, ctype, param=None):
    """Dense Dpi of one cone."""
    v = np.asarray(v, float)
    if ctype == POW:
        return np.eye(3) - _pow_jacobian(-v, param)
    if ctype == DUAL_POW:
        return _pow_jacobian(v, param)
    return oexp.project_gradient(v, ctype)


def pi(v, cone_types, cone_dims, cone_params=None):
    """``DiffOpt.π`` (diff_opt.jl:491-499) over a product of cones."""
    off = cones.cone_offsets(cone_dims)
    out = np.empty(off[-1])
    for c, t in enumerate(cone_types):
        out[off[c]:off[c + 1]] = project(v[off[c]:off[c + 1]], t, _param(cone_params, c))
    return out


def Dpi_blocks(v, cone_types, cone_dims, cone_params=None):
    """``DiffOpt.Dπ`` (diff_opt.jl:509-519): list of dense blocks."""
    off = cones.cone_offsets(cone_dims)
    return [project_gradient(v[off[c]:off[c + 1]], t, _param(cone_params, c)) for c, t in enumerate(cone_types)]


def Dpi_dense(v, cone_types, cone_dims, cone_params=None):
    return sla.block_diag(*Dpi_blocks(v, cone_types, cone_dims, cone_params))


def gradient_cache(A, b, c, x, s, y, cone_types, cone_dims, cone_params=None):
    """``oracle.conic.gradient_cache`` with exponential and power cones among the cones; the result feeds
    ``oracle.conic.forward``, ``reverse`` and ``reverse_param_grads`` as is."""
    v = np.asarray(y, float) - np.asarray(s, float)                 # ConicProgram.jl:222
    return oexp.assemble_cache(A, b, c, x, s, y, Dpi_blocks(v, cone_types, cone_dims, cone_params),
                               pi(v, cone_types, cone_dims, cone_params))
