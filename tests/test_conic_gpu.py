"""GPU parity tests for the LSQR and ConicProgram hot path (through the C ABI) vs the CPU oracle.

Tolerance (BASELINE.json north_star): relative error <= 1e-6 for LSQR-based sensitivities, both sides
run with the same explicit tolerances (``matched residual tolerance``)."""
import numpy as np
import pytest
import scipy.sparse as sp

import bench_data
import diffopt_b200
from oracle import cones as ocones
from oracle import conic as oconic
from oracle import lsqr as olsqr
from oracle import qp as oqp

pytestmark = pytest.mark.gpu
RTOL_LSQR = 1e-6
TIGHT = dict(atol=1e-12, btol=1e-12, conlim=1e12)


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


def test_lsqr_csc_matches_oracle(ctx):
    lsqr = diffopt_b200.submodule("lsqr")
    rng = np.random.default_rng(3)
    A = (sp.random(400, 250, density=0.04, random_state=1) + sp.eye(400, 250)).tocsc()
    b = rng.normal(size=400)
    x, st = lsqr.lsqr_csc(ctx, A, b)
    xo, info = olsqr.lsqr(A, b, return_info=True)
    # near convergence the ||A'r|| estimate is rounding-sensitive (reduction order), so the stop may
    # land one iteration apart; the iterates themselves agree far below the 1e-6 parity bar
    assert abs(st["itn"] - info.itn) <= 2 and st["istop"] == info.istop
    assert rel(x, xo) <= RTOL_LSQR
    for mi in (5, 40):   # same iteration count -> same iterate to rounding
        xg, sg = lsqr.lsqr_csc(ctx, A, b, maxiter=mi)
        xc, ic = olsqr.lsqr(A, b, maxiter=mi, return_info=True)
        assert sg["itn"] == ic.itn == mi and sg["istop"] == ic.istop == 7
        assert rel(xg, xc) <= 1e-8
    bt = rng.normal(size=250)
    xt, _ = lsqr.lsqr_csc(ctx, A, bt, trans=True)
    assert rel(xt, olsqr.lsqr(A.T.tocsc(), bt)) <= RTOL_LSQR


@pytest.mark.parametrize("mode", ["cluster", "gstream", "grid"])
def test_persistent_lsqr_variants_match_oracle(ctx, monkeypatch, mode):
    """The three persistent LSQR drivers (single cluster with hardware barriers / one CTA per SM / the 256-thread build
    of problems with PSD cones, all with the row-block SpMV) on explicit CSC matrices and on the conic operator: same
    iterates as the oracle at matched iteration counts, same answer at convergence."""
    monkeypatch.setenv("DIFFOPT_B200_LSQR", mode)
    lsqr = diffopt_b200.submodule("lsqr")
    cm = diffopt_b200.submodule("conic")
    rng = np.random.default_rng(8)
    A = (sp.random(700, 450, density=0.03, random_state=3) + sp.eye(700, 450)).tocsc()
    A = sp.vstack([A, sp.csc_matrix((3, 450))]).tocsc()          # empty rows
    A[5, :] = rng.normal(size=450)                                # one dense row
    A = A.tocsc()
    b = rng.normal(size=703)
    bt = rng.normal(size=450)
    # a row of 5000 nonzeros, longer than the row blocks of every driver (<= 4096): the one-row, whole-CTA branch of the
    # row-block SpMV (scaled so that it does not dominate the spectrum: at full scale the iterates of this matrix move by
    # 1e-9 under 1e-16 perturbations of A after 6 iterations, at 0.1 by 3e-14)
    rng = np.random.default_rng(9)
    L = (sp.random(400, 5000, density=0.03, random_state=4) + sp.eye(400, 5000)).tolil()
    L[7, :] = 0.1 * rng.normal(size=5000)
    for A, b, bt in ((A, b, bt), (L.tocsc(), rng.normal(size=400), rng.normal(size=5000))):
        for mi in (1, 3, 6):
            xg, sg = lsqr.lsqr_csc(ctx, A, b, maxiter=mi)
            xc, ic = olsqr.lsqr(A, b, maxiter=mi, return_info=True)
            assert sg["itn"] == ic.itn == mi
            # the dense rows make these matrices ill conditioned: rounding differences (summation order) grow quickly
            # with the iteration count (1e-7 .. 3e-4 at 30 iterations depending on the build), so iterates are compared
            # at small counts and the answer at convergence
            assert rel(xg, xc) <= 1e-10, (A.shape, mi, rel(xg, xc))
        x, st = lsqr.lsqr_csc(ctx, A, b)
        assert rel(x, olsqr.lsqr(A, b)) <= RTOL_LSQR
        xt, _ = lsqr.lsqr_csc(ctx, A, bt, trans=True, maxiter=4)
        assert rel(xt, olsqr.lsqr(A.T.tocsc(), bt, maxiter=4)) <= 1e-10
    d = bench_data.conic_config4(n=300, n_zero=30, n_nonneg=200, n_soc=20, soc_dim=6, nnz_per_row=5, seed=31)
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    cache = _oracle_cache(d)
    for iters in (1, 2, 3):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        assert model.last_stats["itn"] == iters
        assert rel(model.back_grad_cache["g"], oconic.reverse(cache, d["seed"], **tol)) <= 1e-9


def test_lp_config1_lsqr_on_kkt(ctx):
    """BASELINE config 1: LP n=200, m=100 -> rank-deficient KKT, minimum-norm LSQR limit."""
    qpm = diffopt_b200.submodule("qp")
    d = bench_data.lp_config1()
    model = qpm.QPModel(ctx, d["Q"], d["q"], d["G"], d["h"], d["A"], d["b"])
    model.set_variable_primal(d["z"]); model.set_constraint_dual_le(-d["lam"]); model.set_constraint_dual_eq(-d["nu"])
    model.iterative_tolerances = dict(atol=1e-13, btol=1e-13, conlim=1e14, maxiter=5000)
    model.reverse_differentiate(d["seed"])
    got = np.concatenate(model.back_grad_cache)
    want = np.concatenate(oqp.reverse(d["Q"], d["G"], d["h"], d["A"], d["z"], d["lam"], d["nu"], d["seed"],
                                      atol=1e-13, btol=1e-13, conlim=1e14, maxiter=5000))
    assert rel(got, want) <= RTOL_LSQR
    K = oqp.create_lhs(d["z"], d["lam"], d["Q"], d["G"], d["h"], d["A"])
    rhs = np.zeros(300); rhs[:200] = d["seed"]
    assert rel(got, -np.linalg.pinv(K) @ rhs) <= 1e-5      # min-norm solution
    # default tolerances as the reference would run it
    model.iterative_tolerances = dict(atol=None, btol=None, conlim=None, maxiter=None)
    model.reverse_differentiate(d["seed"])
    want = np.concatenate(oqp.reverse(d["Q"], d["G"], d["h"], d["A"], d["z"], d["lam"], d["nu"], d["seed"]))
    assert rel(np.concatenate(model.back_grad_cache), want) <= RTOL_LSQR


def test_lp_known_answers(ctx, kat):
    qpm = diffopt_b200.submodule("qp")
    for name in ["lp_simplex_example", "lp_fixed_variable", "lp_nonactive"]:
        c = kat[name]
        n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
        a = lambda k, shape: np.array(c[k], float).reshape(shape)
        model = qpm.QPModel(ctx, a("Q", (n, n)), a("q", n), a("G", (m, n)), a("h", m), a("A", (p, n)), a("b", p))
        model.set_variable_primal(c["z"]); model.set_constraint_dual_le(-a("lam", m)); model.set_constraint_dual_eq(-a("nu", p))
        model.reverse_differentiate(c["seed"])
        dq, _ = model.reverse_objective_function()
        got = dict(dq=dq, grad_z=dq, grad_lam=model.back_grad_cache[1],
                   dh=-np.array([model.get_db_le(i) for i in range(m)]),
                   db=-np.array([model.get_db_eq(i) for i in range(p)]),
                   dG=np.array([model.get_dA_le(i) for i in range(m)]).reshape(m, n),
                   dA=np.array([model.get_dA_eq(i) for i in range(p)]).reshape(p, n))
        for k, e in c["exp"].items():
            e = np.array(e, float).ravel(); g = np.asarray(got[k]).ravel()
            assert np.linalg.norm(g - e) <= max(c["tol"], c["tol"] * max(np.linalg.norm(g), np.linalg.norm(e))), (name, k)
        if "fwd" in c:
            f = c["fwd"]
            fa = lambda k, shape: np.array(f[k], float).reshape(shape)
            model.forward_differentiate(fa("dQ", (n, n)), fa("dq", n), fa("dG", (m, n)), fa("dh", m), fa("dA", (p, n)), fa("db", p))
            assert np.allclose(model.forward_variable_primal(), c["exp_fwd"]["dz"], atol=c["tol"])


def _model_from_kat(ctx, c):
    cm = diffopt_b200.submodule("conic")
    model = cm.ConicModel.from_moi(ctx, np.array(c["coefficients"], float), c["constants"], c["c"],
                                   c["cone_types"], c["cone_dims"])
    model.set_variable_primal(c["x"]); model.set_constraint_primal(c["s"]); model.set_constraint_dual(c["y"])
    return model


@pytest.mark.parametrize("name", ["conic_socp", "conic_psd2", "conic_psd3"])
def test_conic_reference_known_answers(ctx, kat, name):
    c = kat[name]
    model = _model_from_kat(ctx, c)
    for f in c.get("fwd", []):
        model.forward_differentiate(np.array(f["dA"], float), f["db"], f["dc"])
        assert np.allclose(model.forward_variable_primal(), f["exp_dx"], atol=c["tol"])
    for r in c.get("rev", []):
        model.reverse_differentiate(r["seed"])
        assert np.allclose(model.get_db(r["exp_db_rows"]), r["exp_db"], atol=c["tol"])


def _oracle_cache(d):
    return oconic.gradient_cache(d["A"], d["b"], d["c"], d["x"], d["s"], d["y"], d["cone_types"], d["cone_dims"])


@pytest.mark.parametrize("psd_sides", [(), (4, 7), (12,)])
def test_pi_dpi_and_M_operator(ctx, psd_sides):
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4(n=60, n_zero=7, n_nonneg=30, n_soc=9, soc_dim=5, nnz_per_row=4, seed=11,
                                 psd_sides=psd_sides)
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    v = d["y"] - d["s"]
    assert np.allclose(model.vp(), ocones.pi(v, d["cone_types"], d["cone_dims"]), rtol=1e-11, atol=1e-12)
    D = ocones.Dpi_dense(v, d["cone_types"], d["cone_dims"])      # the reference's dense blocks
    cache = _oracle_cache(d)
    Md = cache.M.toarray()
    rng = np.random.default_rng(0)
    for _ in range(2):
        t = rng.normal(size=D.shape[0])
        assert rel(model.dpi_apply(t), D @ t) <= 1e-11
        assert rel(model.dpi_apply(t, transpose=True), D.T @ t) <= 1e-11
        T = rng.normal(size=Md.shape[0])
        assert rel(model.M_apply(T), Md @ T) <= 1e-11
        assert rel(model.M_apply(T, transpose=True), Md.T @ T) <= 1e-11


@pytest.mark.parametrize("psd_sides", [(), (6,)])
def test_conic_forward_reverse_match_oracle(ctx, psd_sides):
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4(n=200, n_zero=20, n_nonneg=160, n_soc=12, soc_dim=10, nnz_per_row=6, seed=21,
                                 psd_sides=psd_sides)
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    model.tolerances = dict(TIGHT, maxiter=20000)
    cache = _oracle_cache(d)
    kw = dict(TIGHT, maxiter=20000)
    model.reverse_differentiate(d["seed"])
    g = oconic.reverse(cache, d["seed"], **kw)
    _, db, dc = oconic.reverse_param_grads(cache, g, dense_dA=False)
    assert rel(model.back_grad_cache["g"], g) <= RTOL_LSQR
    assert rel(model.reverse_objective_function(), dc) <= RTOL_LSQR
    assert rel(model.get_db(), db) <= RTOL_LSQR
    rows = np.array([0, 25, 190])
    dA_ref = np.outer(g[200 + rows], d["x"]) - np.outer(cache.vp[rows], g[:200])
    assert rel(model.get_dA(rows), dA_ref) <= RTOL_LSQR
    rng = np.random.default_rng(5)
    dA = sp.random(*d["A"].shape, density=0.01, random_state=2).tocsc()
    dbv, dcv = rng.normal(size=d["A"].shape[0]), rng.normal(size=200)
    model.forward_differentiate(dA, dbv, dcv)
    dx, dz = oconic.forward(cache, dA, dbv, dcv, **kw)
    assert rel(model.forward_variable_primal(), dx) <= RTOL_LSQR
    # zero perturbation -> zeros (ConicProgram.jl:320-321), tiny seed -> zeros (:369-370)
    model.forward_differentiate(None, None, None)
    assert not model.forward_variable_primal().any()
    model.reverse_differentiate(np.full(200, 1e-7))
    assert not model.back_grad_cache["g"].any()


def test_conic_config4_full_size(ctx):
    """BASELINE config 4 at full size (n=5000, m=7500 = Zeros(500)+Nonneg(4000)+300xSOC(10)), reverse mode.

    This M is badly conditioned (LSQR's own estimate: cond ~ 4e7; the oracle needs ~10^4 iterations at the
    default tolerances and ~5e4 at 1e-12; rounding differences between two LSQR implementations grow ~10x per
    few iterations: 3e-16 after 1, 1e-11 after 10, 3e-2 after 50), so the comparison is (a) iterate by iterate at
    a matched SMALL iteration count and (b) through size-independent properties of the answer."""
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4()
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    cache = _oracle_cache(d)
    dz = np.concatenate([d["seed"], np.zeros(7500), [-(d["x"] @ d["seed"])]])
    for iters in (3, 10, 400):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        assert model.last_stats["itn"] == iters and model.last_stats["istop"] == 7
        if iters <= 10:
            g = oconic.reverse(cache, d["seed"], **tol)
            assert rel(model.back_grad_cache["g"], g) <= 1e-9
        # LSQR's running residual estimate is the true residual of the returned iterate
        r = model.M_apply(model.back_grad_cache["g"]) - dz
        assert abs(np.linalg.norm(r) - model.last_stats["rnorm"]) <= 1e-8 * np.linalg.norm(dz)
    # the operator itself at full size
    T = np.random.default_rng(0).normal(size=12501)
    assert rel(model.M_apply(T), cache.M @ T) <= 1e-12
    assert rel(model.M_apply(T, transpose=True), cache.M.T @ T) <= 1e-12
    assert rel(model.vp(), cache.vp) <= 1e-13


def test_conic_config4_conditioned_converged_parity(ctx):
    """BASELINE config 4 at full size (n=5000, m=7500) on the WELL-CONDITIONED generator (75 % of the nonnegative rows
    active, solution scaled; cond(M) ~ 1e4 instead of ~1e7, bench_data.conic_config4): LSQR runs to its own stopping
    rule on the GPU and in the oracle at MATCHED tolerances and the converged answers are compared (north_star: <= 1e-6
    at a matched residual tolerance).  (a) tight tolerances 1e-13: both stop with istop = 1 after ~2500 iterations,
    measured agreement 1e-12; (b) the reference's default tolerances (sqrt(eps)): ~1130 iterations, agreement ~6e-7."""
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4_conditioned()
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    cache = _oracle_cache(d)
    dz = np.concatenate([d["seed"], np.zeros(7500), [-(d["x"] @ d["seed"])]])
    for tol, bound in ((dict(atol=1e-13, btol=1e-13, conlim=0.0, maxiter=12501), 1e-9),
                       (dict(atol=olsqr.SQRT_EPS, btol=olsqr.SQRT_EPS, conlim=1 / olsqr.SQRT_EPS, maxiter=12501), 1e-6)):
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        g, info = olsqr.lsqr(cache.M, dz, return_info=True, **tol)
        st = model.last_stats
        assert st["istop"] == info.istop == 1                       # ||r|| small: both converged by the same test
        assert abs(st["itn"] - info.itn) <= max(5, info.itn // 100)
        assert abs(st["rnorm"] - info.rnorm) <= 0.02 * info.rnorm
        assert rel(model.back_grad_cache["g"], g) <= bound, (tol["atol"], st, info)
        # the getters the caller reads (ConicProgram.jl:396-428)
        _, db, dc = oconic.reverse_param_grads(cache, g, dense_dA=False)
        assert rel(model.reverse_objective_function(), dc) <= bound and rel(model.get_db(), db) <= bound
        r = model.M_apply(model.back_grad_cache["g"]) - dz
        assert abs(np.linalg.norm(r) - st["rnorm"]) <= 1e-6 * np.linalg.norm(dz)


def test_psd_maxcut_200_full_reverse(ctx):
    """BASELINE config 5: a full `reverse_differentiate!` (ConicProgram.jl:336-394) on the 200 x 200 max-cut SDP against
    the oracle's matrix-free LSQR (the reference's dense 20100^2 Dpi block is never formed).
    r = 20 (SURVEY 8d) is dual degenerate (r(r+1)/2 = 210 > 200 constraints): M is singular beyond the embedding's own
    null direction, LSQR does not converge within N iterations in either implementation and rounding differences
    between the two grow with the iteration count -- compared iterate by iterate while they are meaningful and by
    stopping state at the iteration limit.  r = 8 is nondegenerate: both run to istop = 1 at the reference's default
    tolerances and agree to 1e-4 (the answers of two LSQR runs differ by tolerance x cond(M) ~ 1.5e-8 x 7e5)."""
    cm = diffopt_b200.submodule("conic")
    for r, full_iters in ((20, 400), (8, None)):
        d = bench_data.maxcut_config5(r=r)
        model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
        model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
        args = [d[k] for k in ("A", "b", "c", "x", "s", "y", "cone_types", "cone_dims")]
        m, n = d["A"].shape
        dz = np.concatenate([d["seed"], np.zeros(m), [-(d["x"] @ d["seed"])]])
        for iters, bound in ((1, 1e-10), (2, 1e-10), (5, 1e-9)):
            tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
            model.tolerances = tol
            model.reverse_differentiate(d["seed"])
            g = oconic.reverse_matrix_free(*args, d["seed"], **tol)
            assert rel(model.back_grad_cache["g"], g) <= bound, (r, iters)
        tol = dict(atol=olsqr.SQRT_EPS, btol=olsqr.SQRT_EPS, conlim=1 / olsqr.SQRT_EPS, maxiter=full_iters or 3000)
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        st = model.last_stats
        g, info = olsqr.lsqr(oconic.matrix_free_ops(*args), dz, return_info=True, **tol)
        assert st["istop"] == info.istop == (7 if full_iters else 1)
        assert abs(st["itn"] - info.itn) <= max(5, info.itn // 50)
        assert abs(st["rnorm"] - info.rnorm) <= 0.02 * info.rnorm
        res = np.linalg.norm(model.M_apply(model.back_grad_cache["g"]) - dz)
        assert abs(res - st["rnorm"]) <= 1e-6 * np.linalg.norm(dz)        # the returned g really has that residual
        if not full_iters:
            assert rel(model.back_grad_cache["g"], g) <= 1e-4, (r, st, info)


def test_kat8_dispatch_lp_forward_directions(ctx, kat):
    """KAT 8 (test/jump.jl:473-638) through the reference-shaped model on the GPU: 13 successive forward directions on
    the degenerate-looking dispatch LP (Q = 0 -> LSQR on the KKT matrix, QuadraticProgram.jl:436-438) against column-wise
    LSQR on the hand-built KKT system with the reference's sign table and tolerance."""
    qpm = diffopt_b200.submodule("qp")
    c = kat["lp_dispatch_sensitivity"]
    n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
    a = lambda k, shape: np.array(c[k], float).reshape(shape)
    Q, G, A, z, lam = a("Q", (n, n)), a("G", (m, n)), a("A", (p, n)), a("z", n), a("lam", m)
    model = qpm.QPModel(ctx, Q, a("q", n), G, a("h", m), A, a("b", p))
    model.set_variable_primal(z); model.set_constraint_dual_le(-lam); model.set_constraint_dual_eq(-a("nu", p))
    K = np.block([[Q, G.T, A.T], [np.diag(lam) @ G, np.diag(G @ z - a("h", m)), np.zeros((m, p))],
                  [A, np.zeros((p, m)), np.zeros((p, p))]])
    R = np.block([[np.zeros((n, m)), np.zeros((n, p))], [np.diag(lam), np.zeros((m, p))], [np.zeros((p, m)), np.eye(p)]])
    for i, dct in enumerate(c["directions"]):
        dh, db = np.zeros(m), np.zeros(p)
        (dh if dct["kind"] == "dh" else db)[dct["index"]] = dct["value"]
        model.forward_differentiate(dh=dh, db=db)
        col = olsqr.lsqr(K, R[:, i])[:n]
        got = -model.forward_variable_primal()
        want = dct["kkt_sign"] * col
        assert np.linalg.norm(got - want) <= max(c["tol"], c["tol"] * max(np.linalg.norm(got), np.linalg.norm(want))), i


def test_kat14_qp_cases_through_the_conic_backend(ctx, kat):
    """KAT 14 (test/utils.jl:369-377: every qp_test also runs with ConicProgram.Model): each QP / LP known-answer case
    restated as a conic program (tests/qp_as_conic.py: Zeros + Nonnegatives + the SOC epigraph of the quadratic
    objective) runs forward and reverse through the GPU conic backend.  Checked (1) against the oracle's conic backend
    on every direction, coefficient directions included (<= 1e-6 at matched tight tolerances) and (2) against the QP
    backend's own answers where the reference's two backends agree (constants, linear objective; see the CPU twin
    of this test in test_oracle_kat.py for the sign of coefficient directions)."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from qp_as_conic import conic_forward_direction, qp_as_conic
    cm = diffopt_b200.submodule("conic")
    tight = dict(atol=1e-14, btol=1e-14, conlim=0.0, maxiter=5000)
    agree = {"qp_moi_examples_2": ["dq", "db"], "qp_moi_examples_1": ["dq", "dh"], "qp_ineq_eq": ["dh", "db"],
             "qp_trivial_1": ["dq", "dh"], "lp_simplex_example": ["dh"], "lp_fixed_variable": ["dh", "db"],
             "lp_nonactive": ["dh"], "lp_dispatch_sensitivity": ["dq", "dh", "db"]}
    rng = np.random.default_rng(14)
    for name, keys in agree.items():
        c = kat[name]
        n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
        a = lambda k, shape: np.array(c[k], float).reshape(shape)
        Q, q, G, h, A, b, z, lam, nu = (a("Q", (n, n)), a("q", n), a("G", (m, n)), a("h", m), a("A", (p, n)), a("b", p),
                                        a("z", n), a("lam", m), a("nu", p))
        cp = qp_as_conic(Q, q, G, h, A, b, z, lam, nu)
        model = cm.ConicModel(ctx, cp["A"], cp["b"], cp["c"], cp["cone_types"], cp["cone_dims"])
        model.set_variable_primal(cp["x"]); model.set_constraint_primal(cp["s"]); model.set_constraint_dual(cp["y"])
        model.tolerances = tight
        cache = oconic.gradient_cache(cp["A"], cp["b"], cp["c"], cp["x"], cp["s"], cp["y"], cp["cone_types"], cp["cone_dims"])
        kw_qp = tight if oqp.is_iterative(Q) else {}
        sizes = dict(dq=n, dh=m, db=p, dG=(m, n), dA=(p, n))
        for key in ("dq", "dh", "db", "dG", "dA"):
            if (key in ("dh", "dG") and m == 0) or (key in ("db", "dA") and p == 0):
                continue
            direction = {key: rng.standard_normal(sizes[key])}
            dAc, dbc, dcc = conic_forward_direction(cp, **direction)
            model.forward_differentiate(dAc, dbc, dcc)
            dx, _ = oconic.forward(cache, dAc, dbc, dcc, **tight)
            assert np.linalg.norm(model.forward_variable_primal() - dx) <= 1e-6 * np.linalg.norm(dx) + 1e-10, (name, key)
            if key in keys:
                if key == "dq" and cp["quad"]:
                    model.forward_differentiate(-dAc, dbc, dcc)   # un-negated dA of the reference flips q's SOC rows
                full = dict(dQ=np.zeros((n, n)), dq=np.zeros(n), dG=np.zeros((m, n)), dh=np.zeros(m),
                            dA=np.zeros((p, n)), db=np.zeros(p))
                full.update(direction)
                ref = oqp.forward(Q, G, h, A, z, lam, nu, **full, **kw_qp)[0]
                got = model.forward_variable_primal()[:n]
                assert np.linalg.norm(got - ref) <= 1e-6 * max(1.0, np.linalg.norm(ref)), (name, key, "vs QP backend")
        seed = np.concatenate([np.array(c.get("seed", np.ones(n)), float), np.zeros(cp["x"].size - n)])
        model.reverse_differentiate(seed)
        g = oconic.reverse(cache, seed, **tight)
        assert np.linalg.norm(model.back_grad_cache["g"] - g) <= 1e-6 * np.linalg.norm(g) + 1e-10, name


def test_psd_maxcut_200(ctx):
    """BASELINE config 5: 200 x 200 PSD cone (max-cut SDP shape).  pi and the Dpi operator vs the oracle
    (eigh + 4 GEMMs); the reference's literal dense 20100^2 Jacobian is never formed."""
    cm = diffopt_b200.submodule("conic")
    dd, r = 200, 20
    rng = np.random.default_rng(5)
    V = rng.normal(size=(dd, r)); V /= np.linalg.norm(V, axis=1, keepdims=True)
    X = V @ V.T
    Qf, _ = np.linalg.qr(np.hstack([V, rng.normal(size=(dd, dd - r))]))
    W = Qf[:, r:]
    Smat = (W * rng.uniform(0.5, 1.5, size=dd - r)) @ W.T
    k = dd * (dd + 1) // 2
    s = np.concatenate([np.zeros(dd), ocones.vec_symm(X)])
    y = np.concatenate([rng.normal(size=dd), ocones.vec_symm(Smat)])
    # rows: Zeros(200) (X_ii = 1) + PSD triangle; variables = the triangle
    iu = [(i * (i + 1) // 2 + i) for i in range(dd)]
    A = sp.vstack([sp.csc_matrix((np.ones(dd), (np.arange(dd), iu)), shape=(dd, k)), -sp.identity(k)]).tocsc()
    x = ocones.vec_symm(X)
    b = A @ x + s
    c = -(A.T @ y)
    model = cm.ConicModel(ctx, A, b, c, [ocones.ZERO, ocones.PSD], [dd, k])
    model.set_variable_primal(x); model.set_constraint_primal(s); model.set_constraint_dual(y)
    v = y - s
    assert rel(model.vp(), ocones.pi(v, [ocones.ZERO, ocones.PSD], [dd, k])) <= 1e-9
    t = rng.normal(size=dd + k)
    for tr in (False, True):
        want = ocones.Dpi_apply(v, [ocones.ZERO, ocones.PSD], [dd, k], t, transpose=tr)
        assert rel(model.dpi_apply(t, transpose=tr), want) <= 1e-8


@pytest.mark.parametrize("sort", ["0", "1"])
@pytest.mark.parametrize("col_window", [None, 150])
def test_streaming_lsqr_mid_size_operators(ctx, monkeypatch, col_window, sort):
    """The multi-kernel (streaming) LSQR with its row-block SpMV on operators of a few 10^4 rows -- uniformly random
    columns and a stage-structured pattern, with and without the column-ordered copy of the row blocks that large
    operators get -- against the oracle's explicit M at small iteration counts."""
    monkeypatch.setenv("DIFFOPT_B200_SPMV_SORT", sort)
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4(n=9000, n_zero=900, n_nonneg=7000, n_soc=500, soc_dim=8, nnz_per_row=7, seed=77,
                                 col_window=col_window)
    cache = _oracle_cache(d)
    monkeypatch.setenv("DIFFOPT_B200_LSQR", "stream")
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    for iters in (1, 2, 3):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        model.tolerances = tol
        model.reverse_differentiate(d["seed"])
        assert model.last_stats["itn"] == iters
        assert rel(model.back_grad_cache["g"], oconic.reverse(cache, d["seed"], **tol)) <= 1e-9


def _psd_only_model(ctx, mats):
    """One PSD cone per matrix in `mats`, A = -I (rows = variables), s = 0, y = vec(mat) => v = vec(mat)."""
    cm = diffopt_b200.submodule("conic")
    dims = [m.shape[0] * (m.shape[0] + 1) // 2 for m in mats]
    k = sum(dims)
    y = np.concatenate([ocones.vec_symm(m) for m in mats])
    A = (-sp.identity(k)).tocsc()
    model = cm.ConicModel(ctx, A, np.zeros(k), np.zeros(k), [ocones.PSD] * len(mats), dims)
    model.set_variable_primal(np.zeros(k)); model.set_constraint_primal(np.zeros(k)); model.set_constraint_dual(y)
    return model, y, dims


@pytest.mark.parametrize("case", ["pm_pairs", "degenerate", "zero_and_one", "odd_sizes", "block_path", "batch512"])
def test_psd_eigensolver_edge_cases(ctx, case):
    """The Jacobi eigensolver behind Dpi for PSD cones (diff_opt.jl:509-519 -> MOSD, eigen): spectra with +l/-l
    pairs (the reference's own 2x2 case has them), repeated eigenvalues, the zero matrix, side 1, odd sides, sides
    on both sides of the shared-memory / block-Jacobi switch, and a batch of 512 small cones in one launch."""
    rng = np.random.default_rng(17)

    def with_spectrum(lams):
        Qm, _ = np.linalg.qr(rng.normal(size=(len(lams), len(lams))))
        Xm = (Qm * np.asarray(lams, float)) @ Qm.T
        return (Xm + Xm.T) / 2

    if case == "pm_pairs":
        mats = [np.array([[0.0, 1.0], [1.0, 0.0]]), with_spectrum([3, -3, 2, -2, 1, -1, 0.5, -0.5]),
                with_spectrum([5, -5] * 10)]
    elif case == "degenerate":
        mats = [with_spectrum([2.0] * 5 + [-1.0] * 4), with_spectrum([1.0, 1.0, 1.0, -1.0, -1.0, 0.0, 0.0]),
                np.diag([1.0, -2.0, 3.0, -4.0])]
    elif case == "zero_and_one":
        mats = [np.zeros((3, 3)), np.array([[-2.0]]), np.array([[0.7]]), np.eye(4), -np.eye(5)]
    elif case == "odd_sizes":
        mats = [with_spectrum(rng.normal(size=d)) for d in (3, 5, 17, 33, 63)]
    elif case == "block_path":
        mats = [with_spectrum(rng.normal(size=d)) for d in (119, 121, 150)] + [with_spectrum([4, -4] * 64 + [1e-3, -1e-3])]
    else:
        mats = [with_spectrum(rng.normal(size=d)) for d in ([16] * 256 + [32] * 256)]
    model, v, dims = _psd_only_model(ctx, mats)
    types = [ocones.PSD] * len(mats)
    want_vp = ocones.pi(v, types, dims)
    assert np.linalg.norm(model.vp() - want_vp) <= 1e-11 * max(1.0, np.linalg.norm(want_vp))
    t = rng.normal(size=v.size)
    for tr in (False, True):
        want = ocones.Dpi_apply(v, types, dims, t, transpose=tr)
        got = model.dpi_apply(t, transpose=tr)
        # per cone: a +l/-l pair makes B entries depend on l1/(l1+l2) only, so the tolerance can stay tight
        o = 0
        for k_ in dims:
            assert np.linalg.norm(got[o:o + k_] - want[o:o + k_]) <= 1e-9 * max(1.0, np.linalg.norm(want[o:o + k_]))
            o += k_


def test_streaming_lsqr_matches_persistent_kernel(ctx, monkeypatch):
    """Large conic operators use the multi-kernel (streaming) LSQR; it must reproduce the persistent kernel and the
    oracle on the same problem.  This M is singular and LSQR's iterates are sensitive (the persistent kernel and the
    oracle already differ by 1e-13 / 1e-10 / 1e-5 after 4 / 5 / 7 iterations), so iterates are compared tightly at
    small counts and through the residual norm afterwards."""
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4(n=600, n_zero=60, n_nonneg=400, n_soc=40, soc_dim=7, nnz_per_row=6, seed=11)
    cache = _oracle_cache(d)
    out = {}
    for mode in ("persistent", "stream"):
        monkeypatch.setenv("DIFFOPT_B200_LSQR", mode)
        model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
        model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
        res = {}
        for iters in (1, 2, 3, 4, 10, 40):
            tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
            model.tolerances = tol
            model.reverse_differentiate(d["seed"])
            assert model.last_stats["itn"] == iters and model.last_stats["istop"] == 7
            if iters <= 3:
                assert rel(model.back_grad_cache["g"], oconic.reverse(cache, d["seed"], **tol)) <= 1e-9
            res[iters] = (model.back_grad_cache["g"].copy(), model.last_stats["rnorm"])
        model.forward_differentiate(db=np.ones(model.m))      # forward mode goes through the same solver (40 iterations)
        res["fwd"] = (model.forward_variable_primal().copy(), model.last_stats["rnorm"])
        out[mode] = res
    for k in out["persistent"]:
        a, b = out["persistent"][k], out["stream"][k]
        if k in (1, 2, 3, 4):
            assert rel(a[0], b[0]) <= 1e-9
        assert a[1] == pytest.approx(b[1], rel=1e-5 if k in (1, 2, 3, 4, 10) else 5e-2), (k, a[1], b[1])


@pytest.mark.parametrize("tol, istop", [(dict(atol=0.0, btol=1e-9, conlim=0.0), 1),
                                        (dict(atol=0.0, btol=0.0, conlim=100.0), 3)])
def test_lsqr_stop_tests_persistent_and_streaming(ctx, monkeypatch, tol, istop):
    """LSQR's own stopping rule -- ||r|| small (istop 1), cond(M) beyond conlim (istop 3) -- through the persistent and
    the streaming driver on a well-conditioned, consistent config-4 problem: both stop where the oracle stops, with the
    oracle's answer.  (The oracle's acond crosses conlim = 100 between 98.7 and 103.2, so rounding cannot move the stop.)"""
    cm = diffopt_b200.submodule("conic")
    d = bench_data.conic_config4_conditioned(n=150, n_zero=15, n_nonneg=130, n_soc=9, soc_dim=8, nnz_per_row=5, seed=100)
    cache = _oracle_cache(d)
    dz = np.concatenate([d["seed"], np.zeros(d["A"].shape[0]), [-(d["x"] @ d["seed"])]])
    kw = dict(tol, maxiter=4 * dz.size)
    g, info = olsqr.lsqr(cache.M, dz, return_info=True, **kw)
    assert info.istop == istop
    for mode in ("persistent", "stream"):
        monkeypatch.setenv("DIFFOPT_B200_LSQR", mode)
        model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
        model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
        model.tolerances = kw
        model.reverse_differentiate(d["seed"])
        st = model.last_stats
        assert st["istop"] == info.istop, (mode, st, info)
        assert abs(st["itn"] - info.itn) <= max(3, info.itn // 50), (mode, st, info)
        assert rel(model.back_grad_cache["g"], g) <= RTOL_LSQR, mode


@pytest.mark.parametrize("ctas", [1, 4])
@pytest.mark.parametrize("stage", ["1", "0"])
def test_conic_lockstep_batch_matches_single_problem_solves(ctx, monkeypatch, ctas, stage):
    """Lock-step batch (diffopt_b200_conic_batch_*): B problems of equal size but different sparsity, solutions and
    seeds, advanced by one persistent kernel -- one CTA per problem with the gather vectors staged in shared memory, or
    one 4-CTA cluster per problem.  Every problem must reproduce its own single-problem `reverse_differentiate!`
    (ConicProgram.jl:336-394): same iteration count and stop code as the oracle's LSQR, g / dc / db <= 1e-6; a problem
    whose seed is below the 1e-4 threshold (:369) returns zeros while its neighbours iterate."""
    monkeypatch.setenv("DIFFOPT_B200_CONIC_BATCH_STAGE", stage)
    cm = diffopt_b200.submodule("conic")
    B = 6
    kw = dict(TIGHT, maxiter=20000)
    ds, models = [], []
    for k in range(B):
        d = bench_data.conic_config4_conditioned(n=150, n_zero=15, n_nonneg=130, n_soc=9, soc_dim=8, nnz_per_row=5 + k % 3,
                                                 seed=100 + k)
        mdl = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
        mdl.set_variable_primal(d["x"]); mdl.set_constraint_primal(d["s"]); mdl.set_constraint_dual(d["y"])
        ds.append(d); models.append(mdl)
    seeds = np.stack([d["seed"] for d in ds])
    seeds[3] = 1e-7                                       # below the reverse zero test
    batch = cm.ConicBatch(ctx, models, ctas_per_problem=ctas)
    batch.tolerances = kw
    out = batch.reverse_differentiate(seeds)
    for k, d in enumerate(ds):
        if k == 3:
            assert not out["g"][k].any() and out["stats"][k][1] == 0
            continue
        cache = _oracle_cache(d)
        dz = np.concatenate([seeds[k], np.zeros(d["A"].shape[0]), [-(d["x"] @ seeds[k])]])
        g, info = olsqr.lsqr(cache.M, dz, return_info=True, **kw)
        _, db, dc = oconic.reverse_param_grads(cache, g, dense_dA=False)
        assert int(out["stats"][k][0]) == info.istop
        assert abs(int(out["stats"][k][1]) - info.itn) <= max(3, info.itn // 50)
        assert rel(out["g"][k], g) <= RTOL_LSQR
        assert rel(out["dc"][k], dc) <= RTOL_LSQR and rel(out["db"][k], db) <= RTOL_LSQR
    # a second call on the same batch (work area reused) gives the same answer bit for bit
    out2 = batch.reverse_differentiate(seeds)
    assert np.array_equal(out["g"], out2["g"])


@pytest.mark.parametrize("sides", [(121, 200), (230, 300)])
def test_psd_block_jacobi_sides(ctx, sides):
    """Sides beyond one CTA's shared memory (block Jacobi over a cooperative grid), with a rank-deficient part as max-cut
    solutions have: projection and Dpi must match the oracle's eigh-based ones."""
    rng = np.random.default_rng(23)
    for d in sides:
        Qm, _ = np.linalg.qr(rng.normal(size=(d, d)))
        lam = rng.normal(size=d)
        lam[: d // 10] = 0.0
        Xm = (Qm * lam) @ Qm.T
        model, v, dims = _psd_only_model(ctx, [(Xm + Xm.T) / 2])
        types = [ocones.PSD]
        want_vp = ocones.pi(v, types, dims)
        assert np.linalg.norm(model.vp() - want_vp) <= 1e-11 * max(1.0, np.linalg.norm(want_vp))
        t = rng.normal(size=v.size)
        for tr in (False, True):
            want = ocones.Dpi_apply(v, types, dims, t, transpose=tr)
            got = model.dpi_apply(t, transpose=tr)
            assert np.linalg.norm(got - want) <= 1e-9 * max(1.0, np.linalg.norm(want))


def test_kat13_psd_and_pos_forward(ctx):
    """test/conic_program.jl:378-579 (PSD + POS problem against diffcp): forward mode through the device vs the oracle
    (<= 1e-6 at matched tolerances) and vs the reference's literals at its own atol 0.3 / rtol 0.01."""
    from test_oracle_kat import kat13_psd_pos_problem
    cm = diffopt_b200.submodule("conic")
    d = kat13_psd_pos_problem()
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    model.tolerances = dict(TIGHT, maxiter=2000)
    model.forward_differentiate(d["dA"], d["db"], d["dc"])
    got = model.forward_variable_primal()
    cache = _oracle_cache(d)
    want, _ = oconic.forward(cache, d["dA"], d["db"], d["dc"], **dict(TIGHT, maxiter=2000))
    assert rel(got, want) <= RTOL_LSQR
    assert np.allclose(got, d["dx"], atol=0.3, rtol=0.01)


@pytest.mark.parametrize("route", ["tridiagonal", "jacobi"])
def test_psd_mid_size_routes_and_hard_spectra(ctx, route, monkeypatch):
    """Sides 112-218 have two eigensolvers: tridiagonalisation + multisection + inverse iteration (default) and the block
    Jacobi (DIFFOPT_B200_PSD=jacobi).  Both must reproduce the oracle's projection and Dpi on spectra that stress the direct
    route: exact multiplicities (clusters orthogonalised inside inverse iteration), eigenvalues 1e-10 and 1e-6 apart (close
    but separate shifts; the Newton-Schulz step restores orthogonality), +-pairs, a rank-one matrix, the zero matrix, an
    already diagonal matrix and a matrix that decouples into blocks (zero off-diagonals in T)."""
    if route == "jacobi":
        monkeypatch.setenv("DIFFOPT_B200_PSD", "jacobi")
    rng = np.random.default_rng(29)

    def with_spectrum(lams):
        Qm, _ = np.linalg.qr(rng.normal(size=(len(lams), len(lams))))
        Xm = (Qm * np.asarray(lams, float)) @ Qm.T
        return (Xm + Xm.T) / 2

    d = 128
    blocks = np.zeros((d, d))
    blocks[:60, :60] = with_spectrum(rng.normal(size=60))
    blocks[60:, 60:] = with_spectrum(rng.normal(size=d - 60))
    u = rng.normal(size=d)
    mats = [with_spectrum([2.0] * 50 + [-1.0] * 40 + list(rng.normal(size=d - 90))),
            with_spectrum(list(1.0 + 1e-10 * np.arange(30)) + list(-0.5 + 1e-6 * np.arange(30)) + list(rng.normal(size=d - 60))),
            with_spectrum([3, -3] * (d // 2)),
            np.outer(u, u) / (u @ u),
            np.zeros((d, d)),
            np.diag(rng.normal(size=d)),
            blocks,
            with_spectrum(rng.normal(size=218) * 10.0 ** rng.integers(-3, 3, size=218))]
    for X in mats:
        model, v, dims = _psd_only_model(ctx, [X])
        types = [ocones.PSD]
        want_vp = ocones.pi(v, types, dims)
        assert np.linalg.norm(model.vp() - want_vp) <= 1e-10 * max(1.0, np.linalg.norm(want_vp))
        t = rng.normal(size=v.size)
        for tr in (False, True):
            want = ocones.Dpi_apply(v, types, dims, t, transpose=tr)
            got = model.dpi_apply(t, transpose=tr)
            assert np.linalg.norm(got - want) <= 1e-8 * max(1.0, np.linalg.norm(want))
