"""Exponential and dual exponential cones on the CPU: the oracle's projection (optimality certificates on a hard sample),
its Jacobian (central differences, symmetry), a closed-form known answer through the oracle's conic pipeline, and the
``bench_data.conic_exp_problem`` generator (exact KKT points)."""
import math

import numpy as np
import pytest

import bench_data
import exp_cone_oracle as oc
from exp_cone_samples import certificate_errors, hard_sample, violation_K, violation_Kdual
from oracle import conic as oconic

CERT_TOL = 1e-12


def test_header_and_python_cone_codes_agree():
    import diffopt_b200
    capi = diffopt_b200.submodule("_capi")
    assert (capi.CONE_EXP, capi.CONE_DUAL_EXP) == (oc.EXP, oc.DUAL_EXP) == (4, 5)
    import os
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "diffopt_b200.h")).read()
    assert "#define DIFFOPT_CONE_EXP 4" in hdr and "#define DIFFOPT_CONE_DUAL_EXP 5" in hdr


@pytest.mark.parametrize("ctype", [oc.DUAL_EXP, oc.EXP])
def test_oracle_projection_certificates(ctype):
    """p = Pi_K(v) (DualExponentialCone rows) and p = Pi_K*(v) (ExponentialCone rows, through Moreau) on 10^5 points:
    p in the cone, p - v in its dual, <p, p - v> = 0, each to 1e-12 relative."""
    V = hard_sample(100_000, seed=1 + ctype)
    assert len(V) >= 100_000 - 10
    worst = np.zeros(3)
    for v in V:
        p = oc.project(v, ctype)
        worst = np.maximum(worst, certificate_errors(v, p, dual=ctype == oc.EXP))
    assert (worst <= CERT_TOL).all(), worst


def test_oracle_moreau_and_cases():
    rng = np.random.default_rng(3)
    for v in rng.normal(size=(2000, 3)) * 10.0 ** rng.uniform(-3, 2, (2000, 1)):
        p, q = oc.project(v, oc.DUAL_EXP), -oc.project(-v, oc.EXP)     # Pi_K(v) and Pi_K°(v) = -Pi_K*(-v)
        assert np.linalg.norm(p + q - v) <= 1e-12 * np.linalg.norm(v)
    # the closed-form cases and their tie rules
    assert np.array_equal(oc.project([-1.0, 2.0, 5.0], oc.DUAL_EXP), [-1.0, 2.0, 5.0])          # in K
    assert np.array_equal(oc.project_gradient([-1.0, 2.0, 5.0], oc.DUAL_EXP), np.eye(3))
    assert np.array_equal(oc.project([1.0, -1.0, -3.0], oc.DUAL_EXP), np.zeros(3))               # in K° = -K*
    assert np.array_equal(oc.project([-2.0, -1.0, 3.0], oc.DUAL_EXP), [-2.0, 0.0, 3.0])          # case 3
    assert np.array_equal(oc.project_gradient([-2.0, -1.0, 3.0], oc.DUAL_EXP), np.diag([1.0, 0.0, 1.0]))
    assert np.array_equal(oc.project_gradient([-2.0, -1.0, -3.0], oc.DUAL_EXP), np.diag([1.0, 0.0, 0.0]))
    assert np.array_equal(oc.project_gradient(np.zeros(3), oc.DUAL_EXP), np.eye(3))              # v = 0 is in K
    assert np.array_equal(oc.project_gradient(np.zeros(3), oc.EXP), np.zeros((3, 3)))            # I - DPi_K(0)


def _case(v):
    return oc.exp_case(*(float(a) for a in v))


@pytest.mark.parametrize("ctype", [oc.DUAL_EXP, oc.EXP])
def test_oracle_jacobian_central_differences(ctype):
    """Dpi against central differences of pi (relative 1e-6) at points at least 1e-3 |v| away from a case boundary;
    every block symmetric."""
    rng = np.random.default_rng(11 + ctype)
    V = rng.normal(size=(3000, 3)) * 10.0 ** rng.uniform(-2, 2, (3000, 1))
    probes = rng.normal(size=(24, 3))
    probes /= np.linalg.norm(probes, axis=1)[:, None]
    seen, checked = set(), 0
    for v in V:
        sv = -v if ctype == oc.EXP else v
        nv = np.linalg.norm(v)
        c = _case(sv)
        if any(_case(sv + 1e-3 * nv * d) != c for d in probes):
            continue
        seen.add(c)
        D = oc.project_gradient(v, ctype)
        assert np.abs(D - D.T).max() <= 1e-12 * max(1.0, np.abs(D).max())
        h = 1e-6 * nv
        J = np.empty((3, 3))
        for k in range(3):
            e = np.zeros(3)
            e[k] = h
            J[:, k] = (oc.project(v + e, ctype) - oc.project(v - e, ctype)) / (2 * h)
        assert np.abs(J - D).max() <= 1e-6 * max(1.0, np.abs(D).max()), (v, D, J)
        checked += 1
    assert seen == {1, 2, 3, 4} and checked >= 2000


@pytest.mark.parametrize("b0", [0.3, 2.0, 5.0])
def test_closed_form_known_answer_oracle(b0):
    """min -x s.t. (x, 1, b0) in ExponentialCone: x = log b0, s = (log b0, 1, b0), y = (-1, log b0 - 1, 1/b0);
    forward with db = e3 gives dx = 1/b0."""
    import scipy.sparse as sp
    A = sp.csc_matrix(-np.array([[1.0], [0.0], [0.0]]))
    b, c = np.array([0.0, 1.0, b0]), np.array([-1.0])
    x = np.array([math.log(b0)])
    s = np.array([math.log(b0), 1.0, b0])
    y = np.array([-1.0, math.log(b0) - 1.0, 1.0 / b0])
    assert np.allclose(c + A.T @ y, 0.0, atol=1e-15) and abs(s @ y) <= 1e-15
    cache = oc.gradient_cache(A, b, c, x, s, y, [oc.EXP], [3])
    assert np.allclose(cache.vp, oc.project(y - s, oc.EXP), atol=0)
    dx, _ = oconic.forward(cache, sp.csc_matrix((3, 1)), np.array([0.0, 0.0, 1.0]), np.zeros(1),
                           atol=1e-14, btol=1e-14, conlim=1e14)
    assert dx[0] == pytest.approx(1.0 / b0, rel=1e-9)


def test_generator_yields_kkt_points():
    d = bench_data.conic_exp_problem(n=300, n_zero=20, n_nonneg=150, n_soc=8, soc_dim=5, n_exp=60, n_dual_exp=50,
                                     nnz_per_row=5, seed=3)
    A, s, y = d["A"], d["s"], d["y"]
    assert np.allclose(d["c"] + A.T @ y, 0.0, atol=1e-12)
    assert np.allclose(A @ d["x"] + s, d["b"], atol=1e-12)
    assert abs(s @ y) <= 1e-10 * np.linalg.norm(s) * np.linalg.norm(y)
    off = oc.cone_offsets(d["cone_dims"])
    cases = set()
    for k, t in enumerate(d["cone_types"]):
        ss, yy = s[off[k]:off[k + 1]], y[off[k]:off[k + 1]]
        nn = max(np.linalg.norm(ss) + np.linalg.norm(yy), 1e-300)
        if t == oc.ZERO:
            assert not ss.any()
        elif t == oc.NONNEG:
            assert (ss >= 0).all() and (yy >= 0).all()
        elif t == oc.SOC:
            assert np.linalg.norm(ss[1:]) <= ss[0] * (1 + 1e-12) and np.linalg.norm(yy[1:]) <= yy[0] * (1 + 1e-12)
        elif t == oc.EXP:             # s in K, y in K*
            assert violation_K(ss) <= 1e-12 * nn and violation_Kdual(yy) <= 1e-12 * nn
            cases.add(_case(-(yy - ss)))
        else:                         # DualExponentialCone: s in K*, y in K
            assert violation_Kdual(ss) <= 1e-12 * nn and violation_K(yy) <= 1e-12 * nn
            cases.add(_case(yy - ss))
        assert abs(ss @ yy) <= 1e-12 * nn ** 2
    assert cases == {1, 2, 3, 4}
