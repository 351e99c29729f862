"""Power and dual power cones on the CPU: the oracle's projection (optimality certificates on a hard sample, exact
boundary points, Moreau, the case order), its Jacobian (central differences, symmetry), a closed-form known answer
through the oracle's conic pipeline, the generator's KKT points, and the device header ``csrc/pow_cone.cuh`` compiled
for the host against the oracle."""
import math
import os
import subprocess

import numpy as np
import pytest

import bench_data
import pow_cone_oracle as oc
from oracle import conic as oconic
from pow_cone_samples import ALPHAS, certificate_errors, hard_sample, violation_K, violation_Kdual

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CERT_TOL = 1e-12
SAMPLE = 20_000


def test_header_and_python_cone_codes_agree():
    import diffopt_b200
    capi = diffopt_b200.submodule("_capi")
    assert (capi.CONE_POW, capi.CONE_DUAL_POW) == (oc.POW, oc.DUAL_POW) == (6, 7)
    hdr = open(os.path.join(ROOT, "include", "diffopt_b200.h")).read()
    assert "#define DIFFOPT_CONE_POW 6" in hdr and "#define DIFFOPT_CONE_DUAL_POW 7" in hdr


@pytest.mark.parametrize("alpha", ALPHAS + (None,))
@pytest.mark.parametrize("ctype", [oc.DUAL_POW, oc.POW])
def test_oracle_projection_certificates(ctype, alpha):
    """p = Pi_K(v) (DualPowerCone rows) and p = Pi_K*(v) (PowerCone rows, through Moreau): p in the cone, p - v in its
    dual, <p, p - v> = 0, each to 1e-12 relative; the exact boundary points of the sample recovered to 1e-12 |v|."""
    V, A, P = hard_sample(SAMPLE, alpha, seed=1 + ctype)
    worst, rec = np.zeros(3), 0.0
    for v, a, pk in zip(V, A, P):
        p = oc.project(v, ctype, a)
        worst = np.maximum(worst, certificate_errors(v, p, a, dual=ctype == oc.POW))
        if ctype == oc.DUAL_POW and not np.isnan(pk[0]):
            rec = max(rec, np.linalg.norm(p - pk) / np.linalg.norm(v))
    assert (worst <= CERT_TOL).all(), worst
    assert rec <= 1e-12, rec


def test_oracle_moreau_and_cases():
    rng = np.random.default_rng(3)
    for v, a in zip(rng.normal(size=(2000, 3)) * 10.0 ** rng.uniform(-3, 2, (2000, 1)), rng.uniform(0.02, 0.98, 2000)):
        p, q = oc.project(v, oc.DUAL_POW, a), -oc.project(-v, oc.POW, a)     # Pi_K(v) and Pi_K°(v) = -Pi_K*(-v)
        assert np.linalg.norm(p + q - v) <= 1e-12 * np.linalg.norm(v)
    a = 0.3
    assert oc.pow_case(2.0, 3.0, 1.0, a) == 1                                  # in K
    assert np.array_equal(oc.project([2.0, 3.0, 1.0], oc.DUAL_POW, a), [2.0, 3.0, 1.0])
    assert np.array_equal(oc.project_gradient([2.0, 3.0, 1.0], oc.DUAL_POW, a), np.eye(3))
    assert oc.pow_case(-2.0, -3.0, 1.0, a) == 2                                # in K° = -K*
    assert np.array_equal(oc.project([-2.0, -3.0, 1.0], oc.DUAL_POW, a), np.zeros(3))
    assert np.array_equal(oc.project_gradient([-2.0, -3.0, 1.0], oc.DUAL_POW, a), np.zeros((3, 3)))
    assert oc.pow_case(-2.0, 3.0, 0.0, a) == 3                                 # z0 = 0, mixed signs
    assert np.array_equal(oc.project([-2.0, 3.0, 0.0], oc.DUAL_POW, a), [0.0, 3.0, 0.0])
    assert np.array_equal(oc.project_gradient([-2.0, 3.0, 0.0], oc.DUAL_POW, a), np.diag([0.0, 1.0, 0.0]))
    # ties go to the first case that holds: v = 0 is in K (and in K°), (0, 0, 0) -> I; (0, -1, 0) is in K°
    assert np.array_equal(oc.project_gradient(np.zeros(3), oc.DUAL_POW, a), np.eye(3))
    assert np.array_equal(oc.project_gradient(np.zeros(3), oc.POW, a), np.zeros((3, 3)))       # I - DPi_K(0)
    assert oc.pow_case(0.0, -1.0, 0.0, a) == 2 and oc.pow_case(1.0, -1.0, 1e-300, a) == 4


@pytest.mark.parametrize("ctype", [oc.DUAL_POW, oc.POW])
def test_oracle_jacobian_central_differences(ctype):
    """Dpi against central differences of pi (1e-6) at points at least 1e-3 |v| away from a case boundary; every
    block symmetric."""
    rng = np.random.default_rng(11 + ctype)
    V = rng.normal(size=(3000, 3)) * 10.0 ** rng.uniform(-2, 2, (3000, 1))
    A = rng.uniform(0.05, 0.95, 3000)
    probes = rng.normal(size=(24, 3))
    probes /= np.linalg.norm(probes, axis=1)[:, None]
    seen, checked = set(), 0
    for v, a in zip(V, A):
        sv = -v if ctype == oc.POW else v
        nv = np.linalg.norm(v)
        c = oc.pow_case(*sv, a)
        if any(oc.pow_case(*(sv + 1e-3 * nv * d), a) != c for d in probes):
            continue
        seen.add(c)
        D = oc.project_gradient(v, ctype, a)
        assert np.abs(D - D.T).max() <= 1e-12 * max(1.0, np.abs(D).max())
        h = 1e-6 * nv
        J = np.empty((3, 3))
        for k in range(3):
            e = np.zeros(3)
            e[k] = h
            J[:, k] = (oc.project(v + e, ctype, a) - oc.project(v - e, ctype, a)) / (2 * h)
        assert np.abs(J - D).max() <= 1e-6 * max(1.0, np.abs(D).max()), (v, a, D, J)
        checked += 1
    assert seen == {1, 2, 4} and checked >= 2000


def known_answer(alpha, a, b):
    """min -t s.t. (a, b, t) in PowerCone(alpha): one variable, A = -e3, b = (a, b, 0), c = (-1);
    x = t* = a^alpha b^(1-alpha), s = (a, b, t*), y = (alpha t*/a, (1-alpha) t*/b, -1)."""
    import scipy.sparse as sp
    t = a ** alpha * b ** (1 - alpha)
    return (sp.csc_matrix(-np.array([[0.0], [0.0], [1.0]])), np.array([a, b, 0.0]), np.array([-1.0]), np.array([t]),
            np.array([a, b, t]), np.array([alpha * t / a, (1 - alpha) * t / b, -1.0]))


@pytest.mark.parametrize("alpha,a,b", [(0.3, 2.0, 0.5), (0.5, 1.0, 4.0), (0.8, 3.0, 1.5)])
def test_closed_form_known_answer_oracle(alpha, a, b):
    """Forward with db = e1 gives dx = alpha t*/a, with db = e2 dx = (1-alpha) t*/b."""
    import scipy.sparse as sp
    A, bb, c, x, s, y = known_answer(alpha, a, b)
    assert np.allclose(c + A.T @ y, 0.0, atol=1e-15) and abs(s @ y) <= 1e-14
    cache = oc.gradient_cache(A, bb, c, x, s, y, [oc.POW], [3], [alpha])
    assert np.allclose(cache.vp, oc.project(y - s, oc.POW, alpha), atol=0)
    t = x[0]
    for k, want in ((0, alpha * t / a), (1, (1 - alpha) * t / b)):
        db = np.zeros(3)
        db[k] = 1.0
        dx, _ = oconic.forward(cache, sp.csc_matrix((3, 1)), db, np.zeros(1), atol=1e-14, btol=1e-14, conlim=1e14)
        assert dx[0] == pytest.approx(want, rel=1e-12)


def test_generator_yields_kkt_points():
    d = bench_data.conic_exp_problem(n=300, n_zero=20, n_nonneg=150, n_soc=8, soc_dim=5, n_exp=20, n_dual_exp=20,
                                     nnz_per_row=5, seed=3, n_pow=60, n_dual_pow=50)
    A, s, y, params = d["A"], d["s"], d["y"], d["cone_params"]
    assert np.allclose(d["c"] + A.T @ y, 0.0, atol=1e-12)
    assert np.allclose(A @ d["x"] + s, d["b"], atol=1e-12)
    assert abs(s @ y) <= 1e-10 * np.linalg.norm(s) * np.linalg.norm(y)
    off = oc.cone_offsets(d["cone_dims"])
    cases = set()
    for k, t in enumerate(d["cone_types"]):
        if t not in (oc.POW, oc.DUAL_POW):
            assert params[k] == 0.0
            continue
        a = params[k]
        assert 0.05 <= a <= 0.95
        ss, yy = s[off[k]:off[k + 1]], y[off[k]:off[k + 1]]
        nn = max(np.linalg.norm(ss) + np.linalg.norm(yy), 1e-300)
        if t == oc.POW:               # s in K, y in K*
            assert violation_K(ss, a) <= 1e-12 * nn and violation_Kdual(yy, a) <= 1e-12 * nn
            cases.add(oc.pow_case(*-(yy - ss), a))
        else:                         # DualPowerCone: s in K*, y in K
            assert violation_Kdual(ss, a) <= 1e-12 * nn and violation_K(yy, a) <= 1e-12 * nn
            cases.add(oc.pow_case(*(yy - ss), a))
        assert abs(ss @ yy) <= 1e-12 * nn ** 2
    assert cases == {1, 2, 4}


_HOST_DRIVER = r"""
#include <cstdio>
#include "pow_cone.cuh"
// stdin: records (x0, y0, z0, alpha); stdout: p[3], q[3], D[9], evaluations of psi -- 16 doubles per record
int main() {
    double rec[4], out[16];
    while (fread(rec, sizeof(double), 4, stdin) == 4) {
        out[15] = pow_cone_project(rec[0], rec[1], rec[2], rec[3], out, out + 3, out + 6);
        fwrite(out, sizeof(double), 16, stdout);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def host_pow_cone(tmp_path_factory):
    """``pow_cone_project`` of the device header built for the host with g++."""
    d = tmp_path_factory.mktemp("pow_cone_host")
    src, exe = d / "drv.cpp", d / "drv"
    src.write_text(_HOST_DRIVER)
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "diffopt.jl_b200", "csrc"), str(src), "-o",
                        str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

    def run(V, A):
        inp = np.ascontiguousarray(np.concatenate([V, np.asarray(A)[:, None]], 1), dtype=np.float64).tobytes()
        out = subprocess.run([str(exe)], input=inp, capture_output=True, check=True).stdout
        return np.frombuffer(out).reshape(-1, 16)
    return run


@pytest.mark.parametrize("alpha", ALPHAS + (None,))
def test_device_header_on_the_host_matches_the_oracle(host_pow_cone, alpha):
    """The CUDA arithmetic before any GPU run: projection within 1e-10 |v| of the oracle's, certificates to 1e-12,
    Moreau p + q = v, symmetric Jacobian; the Jacobian equals the oracle's at points of normal scale."""
    V, A, _ = hard_sample(SAMPLE, alpha, seed=40)
    R = host_pow_cone(V, A)
    worst, dev = np.zeros(3), 0.0
    for v, a, out in zip(V, A, R):
        nv = np.linalg.norm(v)
        worst = np.maximum(worst, certificate_errors(v, out[:3], a))
        dev = max(dev, np.linalg.norm(out[:3] - oc.project(v, oc.DUAL_POW, a)) / nv)
        assert np.linalg.norm(out[:3] + out[3:6] - v) <= 1e-15 * nv * 4
        D = out[6:15].reshape(3, 3)
        assert np.array_equal(D, D.T)
    assert (worst <= CERT_TOL).all(), worst
    assert dev <= 1e-10, dev
    rng = np.random.default_rng(7)
    W = rng.normal(size=(2000, 3)) * 10.0 ** rng.uniform(-2, 2, (2000, 1))
    Aw = rng.uniform(0.05, 0.95, 2000) if alpha is None else np.full(2000, alpha)
    R = host_pow_cone(W, Aw)
    assert max(np.abs(out[6:15].reshape(3, 3) - oc.project_gradient(v, oc.DUAL_POW, a)).max()
               for v, a, out in zip(W, Aw, R)) <= 1e-9
    assert (R[:, 15] <= 200).all()
