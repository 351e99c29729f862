"""Power and dual power cones on the device (cone_pow_kernel, the 3 x 3 block rows of dpi_apply) against the CPU
oracle: pi, Dpi and M on mixed problems, the projection certificates on a hard sample, forward / reverse through every
LSQR driver, a closed-form known answer through the C ABI, the lock-step batch, bad input, and the old entry point."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

import bench_data
import diffopt_b200
import pow_cone_oracle as ocones
from oracle import conic as oconic
from oracle import lsqr as olsqr
from pow_cone_samples import certificate_errors, hard_sample
from test_pow_cone_cpu import known_answer

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
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"], d["cone_params"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    return model


def _cache(d):
    return ocones.gradient_cache(d["A"], d["b"], d["c"], d["x"], d["s"], d["y"], d["cone_types"], d["cone_dims"],
                                 d["cone_params"])


@pytest.mark.parametrize("psd_sides", [(), (5,)])
def test_pow_pi_dpi_and_M_operator(ctx, psd_sides):
    d = bench_data.conic_exp_problem(n=80, n_zero=7, n_nonneg=30, n_soc=5, soc_dim=5, n_exp=6, n_dual_exp=5,
                                     nnz_per_row=4, seed=12, psd_sides=psd_sides, n_pow=14, n_dual_pow=11)
    model = _model(ctx, d)
    v = d["y"] - d["s"]
    args = (v, d["cone_types"], d["cone_dims"], d["cone_params"])
    assert rel(model.vp(), ocones.pi(*args)) <= 1e-11
    D = ocones.Dpi_dense(*args)
    Md = _cache(d).M.toarray()
    rng = np.random.default_rng(0)
    for _ in range(2):
        t = rng.normal(size=D.shape[0])
        assert rel(model.dpi_apply(t), D @ t) <= 1e-11
        assert rel(model.dpi_apply(t, transpose=True), D.T @ t) <= 1e-11
        T = rng.normal(size=Md.shape[0])
        assert rel(model.M_apply(T), Md @ T) <= 1e-11
        assert rel(model.M_apply(T, transpose=True), Md.T @ T) <= 1e-11


@pytest.mark.parametrize("alpha", [0.01, 0.5, 0.99, None])
@pytest.mark.parametrize("ctype", [ocones.DUAL_POW, ocones.POW])
def test_device_projection_certificates(ctx, ctype, alpha):
    """The hard sample of the CPU test packed as 3-row cones of one setup (v = y - s with s = 0): the device's vp
    satisfies the certificates to 1e-12 and agrees with the oracle."""
    cm = diffopt_b200.submodule("conic")
    V, A, _ = hard_sample(20_000, alpha, seed=20 + ctype)
    k = len(V)
    m = 3 * k
    Am = sp.csc_matrix((np.ones(m), (np.arange(m), np.zeros(m, dtype=np.int64))), shape=(m, 1))
    model = cm.ConicModel(ctx, Am, np.zeros(m), np.zeros(1), [ctype] * k, [3] * k, A)
    model.set_variable_primal(np.zeros(1)); model.set_constraint_primal(np.zeros(m)); model.set_constraint_dual(V.ravel())
    P = model.vp().reshape(k, 3)
    worst = np.zeros(3)
    dev = 0.0
    for v, a, p in zip(V, A, P):
        worst = np.maximum(worst, certificate_errors(v, p, a, dual=ctype == ocones.POW))
    for i in range(0, k, 7):
        dev = max(dev, np.linalg.norm(P[i] - ocones.project(V[i], ctype, A[i])) / np.linalg.norm(V[i]))
    assert (worst <= 1e-12).all(), worst
    assert dev <= 1e-10, dev


# Converged solves of two drivers (different reduction orders) agree to 1e-6 only where M is well conditioned; power
# cones with exponents near 0.05 / 0.95 make many draws of this generator ill-conditioned (cond(M) up to 1e11), so the
# seeds are ones whose M is conditioned like the exponential-cone tests' problems, and the tests check that premise.
ACOND_MAX = 1e6


def _pow_problem(psd_sides=()):
    return bench_data.conic_exp_problem(n=200, n_zero=20, n_nonneg=120, n_soc=6, soc_dim=5, n_exp=6, n_dual_exp=4,
                                        nnz_per_row=6, seed=35 if psd_sides else 34, n_pow=16, n_dual_pow=14,
                                        psd_sides=psd_sides)


def _reverse_rhs(d, seed):
    return np.concatenate([seed, np.zeros(d["A"].shape[0]), [-(d["x"] @ seed)]])


@pytest.mark.parametrize("mode,psd_sides", [("cluster", ()), ("gstream", ()), ("grid", ()), ("stream", ()), ("grid", (6,))])
def test_pow_forward_reverse_every_driver(ctx, monkeypatch, mode, psd_sides):
    """Forward / reverse against the oracle at matched tight tolerances through each LSQR driver; at fixed small
    iteration counts the iterates match the oracle's."""
    monkeypatch.setenv("DIFFOPT_B200_LSQR", mode)
    d = _pow_problem(psd_sides=psd_sides)
    model = _model(ctx, d)
    cache = _cache(d)
    for iters in (1, 2, 3):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        assert model.last_stats["itn"] == iters
        assert rel(model.back_grad_cache["g"], oconic.reverse(cache, d["seed"], **tol)) <= 1e-9
    kw = dict(TIGHT, maxiter=20000)
    assert olsqr.lsqr(cache.M, _reverse_rhs(d, d["seed"]), return_info=True, **kw)[1].acond <= ACOND_MAX
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


@pytest.mark.parametrize("alpha,a,b", [(0.3, 2.0, 0.5), (0.5, 1.0, 4.0), (0.8, 3.0, 1.5)])
def test_pow_closed_form_known_answer(ctx, alpha, a, b):
    """min -t s.t. (a, b, t) in PowerCone(alpha) through the C ABI: forward with db = e1 gives dx = alpha t*/a, with
    db = e2 dx = (1-alpha) t*/b; the reverse result is pinned against the oracle."""
    cm = diffopt_b200.submodule("conic")
    A, bb, c, x, s, y = known_answer(alpha, a, b)
    model = cm.ConicModel(ctx, A, bb, c, [cm.CONE_POW], [3], [alpha])
    model.set_variable_primal(x); model.set_constraint_primal(s); model.set_constraint_dual(y)
    kw = dict(atol=1e-14, btol=1e-14, conlim=1e14, maxiter=200)
    model.tolerances = kw
    t = x[0]
    for k, want in ((0, alpha * t / a), (1, (1 - alpha) * t / b)):
        db = np.zeros(3)
        db[k] = 1.0
        model.forward_differentiate(db=db)
        assert model.forward_variable_primal()[0] == pytest.approx(want, rel=1e-9)
    cache = ocones.gradient_cache(A, bb, c, x, s, y, [ocones.POW], [3], [alpha])
    model.reverse_differentiate(np.array([1.0]))
    assert rel(model.back_grad_cache["g"], oconic.reverse(cache, np.array([1.0]), **kw)) <= 1e-9


@pytest.mark.parametrize("ctas", [1, 4])
def test_pow_lockstep_batch_matches_single_problem_solves(ctx, ctas):
    cm = diffopt_b200.submodule("conic")
    kw = dict(TIGHT, maxiter=20000)
    ds, models = [], []
    for k, seed in enumerate((320, 321, 322, 343)):
        d = bench_data.conic_exp_problem(n=150, n_zero=15, n_nonneg=90, n_soc=4, soc_dim=6, n_exp=4, n_dual_exp=4,
                                         nnz_per_row=5 + k % 2, seed=seed, solution_scale=0.2, n_pow=8 + k,
                                         n_dual_pow=10 - k)
        ds.append(d)
        models.append(_model(ctx, d))
    seeds = np.stack([d["seed"] for d in ds])
    batch = cm.ConicBatch(ctx, models, ctas_per_problem=ctas)
    batch.tolerances = kw
    out = batch.reverse_differentiate(seeds)
    for k, (d, mdl) in enumerate(zip(ds, models)):
        cache = _cache(d)
        g, info = olsqr.lsqr(cache.M, _reverse_rhs(d, seeds[k]), return_info=True, **kw)
        assert info.acond <= ACOND_MAX
        assert int(out["stats"][k][0]) == info.istop
        assert abs(int(out["stats"][k][1]) - info.itn) <= max(3, info.itn // 50)
        assert rel(out["g"][k], g) <= RTOL_LSQR
        mdl.tolerances = kw
        mdl.reverse_differentiate(seeds[k])
        assert rel(out["g"][k], mdl.back_grad_cache["g"]) <= RTOL_LSQR
        assert rel(out["db"][k], mdl.get_db()) <= RTOL_LSQR


def _setup_rc(ctx, ct, dim, params, entry="diffopt_b200_conic_setup_ex"):
    """Return code and message of a setup of one cone of type ct (dimension dim) through the C ABI."""
    capi = diffopt_b200.submodule("_capi")
    lsq = diffopt_b200.submodule("lsqr")
    colptr, rowval, nzval = lsq.julia_csc(sp.csc_matrix(np.ones((dim, 1))))
    z, x = np.zeros(dim), np.zeros(1)
    types, dims = np.array([ct], dtype=np.int32), np.array([dim], dtype=np.int64)
    args = [ctx.h, 1, dim, capi.ptr(colptr), capi.ptr(rowval), capi.ptr(nzval), capi.ptr(z), capi.ptr(x), capi.ptr(x),
            capi.ptr(z), capi.ptr(z), 1, capi.ptr(types), capi.ptr(dims)]
    if entry.endswith("_ex"):
        args.append(capi.ptr(None if params is None else np.asarray(params, dtype=np.float64)))
    rc = getattr(ctx.lib, entry)(*args, capi.HOST)
    return rc, ctx.lib.diffopt_b200_last_error(ctx.h).decode() if rc else ""


def test_pow_cone_bad_input(ctx):
    cm = diffopt_b200.submodule("conic")
    for ct in (cm.CONE_POW, cm.CONE_DUAL_POW):
        rc, msg = _setup_rc(ctx, ct, 4, [0.5])
        assert rc == -1 and "power cone dimension must be 3" in msg
        for a in (0.0, 1.0, -0.5, float("nan"), float("inf")):
            rc, msg = _setup_rc(ctx, ct, 3, [a])
            assert rc == -1 and "exponent must be finite and in (0, 1)" in msg, (a, msg)
        rc, msg = _setup_rc(ctx, ct, 3, None)
        assert rc == -1 and "conic_setup_ex" in msg
        rc, msg = _setup_rc(ctx, ct, 3, None, entry="diffopt_b200_conic_setup")
        assert rc == -1 and "conic_setup_ex" in msg
        rc, msg = _setup_rc(ctx, ct, 3, [0.5])
        assert rc == 0, msg
    # the lock-step batch takes the same checks
    capi = diffopt_b200.submodule("_capi")
    ctx.check(ctx.lib.diffopt_b200_conic_batch_begin(ctx.h, 1, 1))
    lsq = diffopt_b200.submodule("lsqr")
    colptr, rowval, nzval = lsq.julia_csc(sp.csc_matrix(np.ones((3, 1))))
    z, x = np.zeros(3), np.zeros(1)
    rc = ctx.lib.diffopt_b200_conic_batch_add(
        ctx.h, 1, 3, capi.ptr(colptr), capi.ptr(rowval), capi.ptr(nzval), capi.ptr(z), capi.ptr(x), capi.ptr(x),
        capi.ptr(z), capi.ptr(z), 1, capi.ptr(np.array([cm.CONE_POW], dtype=np.int32)),
        capi.ptr(np.array([3], dtype=np.int64)), capi.HOST)
    assert rc == -1 and "conic_setup_ex" in ctx.lib.diffopt_b200_last_error(ctx.h).decode()


def test_old_and_new_setup_entry_points_agree_bitwise(ctx):
    """conic_setup and conic_setup_ex(cone_param = NULL) on an existing exponential-cone problem: the same vp."""
    capi = diffopt_b200.submodule("_capi")
    lsq = diffopt_b200.submodule("lsqr")
    d = bench_data.conic_exp_problem(n=300, n_zero=20, n_nonneg=150, n_soc=8, soc_dim=5, n_exp=60, n_dual_exp=50,
                                     nnz_per_row=5, seed=3)
    colptr, rowval, nzval = lsq.julia_csc(d["A"])
    m, n = d["A"].shape
    types = np.ascontiguousarray(d["cone_types"], dtype=np.int32)
    dims = np.ascontiguousarray(d["cone_dims"], dtype=np.int64)
    args = [ctx.h, n, m, capi.ptr(colptr), capi.ptr(rowval), capi.ptr(nzval)] + \
        [capi.ptr(np.ascontiguousarray(d[k], dtype=np.float64)) for k in ("b", "c", "x", "s", "y")] + \
        [len(types), capi.ptr(types), capi.ptr(dims)]
    out = []
    for ex in (False, True):
        ctx.check(ctx.lib.diffopt_b200_conic_setup_ex(*args, None, capi.HOST) if ex else
                  ctx.lib.diffopt_b200_conic_setup(*args, capi.HOST))
        vp = np.empty(m)
        ctx.check(ctx.lib.diffopt_b200_conic_get_vp(ctx.h, capi.ptr(vp), capi.HOST))
        out.append(vp)
    assert np.array_equal(out[0], out[1])
    assert ctypes.sizeof(ctypes.c_double) == 8
