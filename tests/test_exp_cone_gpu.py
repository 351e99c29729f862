"""Exponential and dual exponential cones on the device (cone_exp_kernel, the 3 x 3 block rows of dpi_apply) against the
CPU oracle: pi, Dpi and M, the projection certificates on a hard sample, forward / reverse through every LSQR driver,
a closed-form known answer, the lock-step batch and bad input."""
import math

import numpy as np
import pytest
import scipy.sparse as sp

import bench_data
import diffopt_b200
import exp_cone_oracle as ocones
from exp_cone_samples import certificate_errors, hard_sample
from oracle import conic as oconic
from oracle import lsqr as olsqr

pytestmark = pytest.mark.gpu
RTOL_LSQR = 1e-6
TIGHT = dict(atol=1e-12, btol=1e-12, conlim=1e12)


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


def _model(ctx, d):
    cm = diffopt_b200.submodule("conic")
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    return model


def _cache(d):
    return ocones.gradient_cache(d["A"], d["b"], d["c"], d["x"], d["s"], d["y"], d["cone_types"], d["cone_dims"])


@pytest.mark.parametrize("psd_sides", [(), (5,)])
def test_exp_pi_dpi_and_M_operator(ctx, psd_sides):
    d = bench_data.conic_exp_problem(n=80, n_zero=7, n_nonneg=30, n_soc=5, soc_dim=5, n_exp=14, n_dual_exp=11,
                                     nnz_per_row=4, seed=12, psd_sides=psd_sides)
    model = _model(ctx, d)
    v = d["y"] - d["s"]
    assert rel(model.vp(), ocones.pi(v, d["cone_types"], d["cone_dims"])) <= 1e-11
    D = ocones.Dpi_dense(v, d["cone_types"], d["cone_dims"])
    Md = _cache(d).M.toarray()
    rng = np.random.default_rng(0)
    for _ in range(2):
        t = rng.normal(size=D.shape[0])
        assert rel(model.dpi_apply(t), D @ t) <= 1e-11
        assert rel(model.dpi_apply(t, transpose=True), D.T @ t) <= 1e-11
        T = rng.normal(size=Md.shape[0])
        assert rel(model.M_apply(T), Md @ T) <= 1e-11
        assert rel(model.M_apply(T, transpose=True), Md.T @ T) <= 1e-11


@pytest.mark.parametrize("ctype", [ocones.DUAL_EXP, ocones.EXP])
def test_device_projection_certificates(ctx, ctype):
    """The hard sample of the CPU test packed as 3-row cones of one setup (v = y - s with s = 0): the device's vp
    satisfies the certificates to 1e-12 and agrees with the oracle."""
    cm = diffopt_b200.submodule("conic")
    V = hard_sample(30_000, seed=20 + ctype)
    k = len(V)
    m = 3 * k
    A = sp.csc_matrix((np.ones(m), (np.arange(m), np.zeros(m, dtype=np.int64))), shape=(m, 1))
    model = cm.ConicModel(ctx, A, np.zeros(m), np.zeros(1), [ctype] * k, [3] * k)
    model.set_variable_primal(np.zeros(1)); model.set_constraint_primal(np.zeros(m)); model.set_constraint_dual(V.ravel())
    P = model.vp().reshape(k, 3)
    worst = np.zeros(3)
    dev = 0.0
    for v, p in zip(V, P):
        worst = np.maximum(worst, certificate_errors(v, p, dual=ctype == ocones.EXP))
    for i in range(0, k, 7):
        dev = max(dev, np.linalg.norm(P[i] - ocones.project(V[i], ctype)) / np.linalg.norm(V[i]))
    assert (worst <= 1e-12).all(), worst
    assert dev <= 1e-10, dev


def _exp_problem(**kw):
    return bench_data.conic_exp_problem(n=200, n_zero=20, n_nonneg=120, n_soc=6, soc_dim=5, n_exp=16, n_dual_exp=14,
                                        nnz_per_row=6, seed=21, **kw)


@pytest.mark.parametrize("mode,psd_sides", [("cluster", ()), ("gstream", ()), ("grid", ()), ("stream", ()), ("grid", (6,))])
def test_exp_forward_reverse_every_driver(ctx, monkeypatch, mode, psd_sides):
    """Forward / reverse against the oracle at matched tight tolerances through each LSQR driver (`grid` is the
    256-thread build of problems with PSD cones, run here without and with one); at fixed small iteration counts the
    iterates match the oracle's."""
    monkeypatch.setenv("DIFFOPT_B200_LSQR", mode)
    d = _exp_problem(psd_sides=psd_sides)
    model = _model(ctx, d)
    cache = _cache(d)
    for iters in (1, 2, 3):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        assert model.last_stats["itn"] == iters
        assert rel(model.back_grad_cache["g"], oconic.reverse(cache, d["seed"], **tol)) <= 1e-9
    kw = dict(TIGHT, maxiter=20000)
    model.tolerances = kw
    model.reverse_differentiate(d["seed"])
    g = oconic.reverse(cache, d["seed"], **kw)
    _, db, dc = oconic.reverse_param_grads(cache, g, dense_dA=False)
    assert rel(model.back_grad_cache["g"], g) <= RTOL_LSQR
    assert rel(model.reverse_objective_function(), dc) <= RTOL_LSQR
    assert rel(model.get_db(), db) <= RTOL_LSQR
    rng = np.random.default_rng(5)
    dA = sp.random(*d["A"].shape, density=0.01, random_state=2).tocsc()
    dbv, dcv = rng.normal(size=d["A"].shape[0]), rng.normal(size=200)
    model.forward_differentiate(dA, dbv, dcv)
    dx, _ = oconic.forward(cache, dA, dbv, dcv, **kw)
    assert rel(model.forward_variable_primal(), dx) <= RTOL_LSQR


@pytest.mark.parametrize("b0", [0.3, 2.0, 5.0])
def test_exp_closed_form_known_answer(ctx, b0):
    """min -x s.t. (x, 1, b0) in ExponentialCone through the C ABI: forward with db = e3 gives dx = 1/b0; the reverse
    result is pinned against the oracle (the reference's reverse solves with M, not M')."""
    cm = diffopt_b200.submodule("conic")
    A = sp.csc_matrix(-np.array([[1.0], [0.0], [0.0]]))
    b, c = np.array([0.0, 1.0, b0]), np.array([-1.0])
    x = np.array([math.log(b0)])
    s = np.array([math.log(b0), 1.0, b0])
    y = np.array([-1.0, math.log(b0) - 1.0, 1.0 / b0])
    model = cm.ConicModel(ctx, A, b, c, [cm.CONE_EXP], [3])
    model.set_variable_primal(x); model.set_constraint_primal(s); model.set_constraint_dual(y)
    kw = dict(atol=1e-14, btol=1e-14, conlim=1e14, maxiter=200)
    model.tolerances = kw
    model.forward_differentiate(db=np.array([0.0, 0.0, 1.0]))
    assert model.forward_variable_primal()[0] == pytest.approx(1.0 / b0, rel=1e-9)
    cache = ocones.gradient_cache(A, b, c, x, s, y, [ocones.EXP], [3])
    model.reverse_differentiate(np.array([1.0]))
    assert rel(model.back_grad_cache["g"], oconic.reverse(cache, np.array([1.0]), **kw)) <= 1e-9


@pytest.mark.parametrize("ctas", [1, 4])
def test_exp_lockstep_batch_matches_single_problem_solves(ctx, ctas):
    cm = diffopt_b200.submodule("conic")
    kw = dict(TIGHT, maxiter=20000)
    ds, models = [], []
    for k in range(4):
        d = bench_data.conic_exp_problem(n=150, n_zero=15, n_nonneg=90, n_soc=4, soc_dim=6, n_exp=10 + k, n_dual_exp=12 - k,
                                         nnz_per_row=5 + k % 2, seed=300 + k, solution_scale=0.2)
        ds.append(d)
        models.append(_model(ctx, d))
    seeds = np.stack([d["seed"] for d in ds])
    batch = cm.ConicBatch(ctx, models, ctas_per_problem=ctas)
    batch.tolerances = kw
    out = batch.reverse_differentiate(seeds)
    for k, (d, mdl) in enumerate(zip(ds, models)):
        cache = _cache(d)
        dz = np.concatenate([seeds[k], np.zeros(d["A"].shape[0]), [-(d["x"] @ seeds[k])]])
        g, info = olsqr.lsqr(cache.M, dz, return_info=True, **kw)
        assert int(out["stats"][k][0]) == info.istop
        assert abs(int(out["stats"][k][1]) - info.itn) <= max(3, info.itn // 50)
        assert rel(out["g"][k], g) <= RTOL_LSQR
        mdl.tolerances = kw
        mdl.reverse_differentiate(seeds[k])
        assert rel(out["g"][k], mdl.back_grad_cache["g"]) <= RTOL_LSQR
        assert rel(out["db"][k], mdl.get_db()) <= RTOL_LSQR


def test_exp_cone_bad_dimension(ctx):
    cm = diffopt_b200.submodule("conic")
    for ct in (cm.CONE_EXP, cm.CONE_DUAL_EXP):
        A = sp.csc_matrix(np.ones((4, 1)))
        model = cm.ConicModel(ctx, A, np.zeros(4), np.zeros(1), [ct], [4])
        model.set_variable_primal(np.zeros(1)); model.set_constraint_primal(np.zeros(4)); model.set_constraint_dual(np.zeros(4))
        with pytest.raises(Exception, match="exponential cone dimension must be 3"):
            model.vp()
