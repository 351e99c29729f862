"""GPU parity tests for the QuadraticProgram hot path: CUDA (through the C ABI) vs the CPU oracle.

Tolerance (BASELINE.json north_star): relative error <= 1e-8 for direct KKT sensitivities,
measured per instance as ||x_gpu - x_oracle||_2 / ||x_oracle||_2.
"""
import numpy as np
import pytest

import bench_data
import diffopt_b200
from oracle import qp as oqp

pytestmark = pytest.mark.gpu
RTOL_DIRECT = 1e-8


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


def rel_err(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm(a - b, axis=-1) / np.maximum(np.linalg.norm(b, axis=-1), 1e-300)


def _oracle_batch(d):
    return oqp.batch_forward_reverse(d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], d["seed"],
                                     d["dQ"], d["dq"], d["dG"], d["dh"], d["dA"], d["db"])


@pytest.mark.parametrize("n,m,p,na", [(64, 64, 16, 16), (10, 25, 10, 0), (5, 0, 2, 0), (7, 9, 0, 3), (3, 0, 0, 0),
                                      (33, 47, 5, 11), (1, 1, 0, 1), (80, 60, 20, 30)])
def test_fused_solve_matches_oracle(ctx, n, m, p, na):
    qpm = diffopt_b200.submodule("qp")
    B = 24
    d = bench_data.qp_batch(B, n, m, p, n_active=na, seed0=100 + n)
    fwd, rev, info = qpm.solve_batch(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"],
                                     fwd_dir=(d["dQ"], d["dq"], d["dG"], d["dh"], d["dA"], d["db"]), seed=d["seed"])
    assert not info.any()
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


def test_setup_forward_reverse_and_param_grads(ctx):
    qpm = diffopt_b200.submodule("qp")
    B, n, m, p = 40, 64, 64, 16
    d = bench_data.qp_batch(B, n, m, p)
    batch = qpm.QPBatch(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"])
    dz, dl, dn = batch.reverse(d["seed"])
    fz, fl, fn = batch.forward(d["dQ"], d["dq"], d["dG"], d["dh"], d["dA"], d["db"])
    of, orv = _oracle_batch(d)
    assert rel_err(np.hstack([dz, dl, dn]), orv).max() <= RTOL_DIRECT
    assert rel_err(np.hstack([fz, fl, fn]), of).max() <= RTOL_DIRECT
    # partial forward direction (only dh), as in docs/src/examples/matrix-inversion-manual.jl
    fz2, _, _ = batch.forward(dh=d["dh"])
    for b in range(0, B, 13):
        z0 = np.zeros
        ref = oqp.forward(d["Q"][b], d["G"][b], d["h"][b], d["A"][b], d["z"][b], d["lam"][b], d["nu"][b],
                          z0((n, n)), z0(n), z0((m, n)), d["dh"][b], z0((p, n)), z0(p))[0]
        assert rel_err(fz2[b], ref) <= RTOL_DIRECT
    rev = np.hstack([dz, dl, dn])
    g = batch.param_grads(rev)
    gsum = batch.param_grads(rev, reduce_over_batch=True)
    for b in range(0, B, 7):
        ref = oqp.reverse_param_grads(d["z"][b], d["lam"][b], d["nu"][b], orv[b, :n], orv[b, n:n + m], orv[b, n + m:])
        for got, want in zip(g, ref):
            assert np.allclose(got[b], want, rtol=1e-8, atol=1e-10)
    refs = [oqp.reverse_param_grads(d["z"][b], d["lam"][b], d["nu"][b], orv[b, :n], orv[b, n:n + m], orv[b, n + m:])
            for b in range(B)]
    for k in range(6):
        assert np.allclose(gsum[k], sum(r[k] for r in refs), rtol=1e-8, atol=1e-9)


def test_reference_known_answers_through_qpmodel(ctx, kat):
    """The reference's own QP literals (direct-solve cases) through the reference-shaped model."""
    qpm = diffopt_b200.submodule("qp")
    for name in ["qp_moi_examples_2", "qp_moi_examples_1", "qp_ineq_eq", "qp_trivial_1", "qp_fixture_data"]:
        c = kat[name]
        n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
        a = lambda k, shape: np.array(c[k], float).reshape(shape)
        model = qpm.QPModel(ctx, a("Q", (n, n)), a("q", n), a("G", (m, n)), a("h", m), a("A", (p, n)), a("b", p))
        model.set_variable_primal(c["z"])
        model.set_constraint_dual_le(-a("lam", m))   # MOI duals; the model negates them like the reference
        model.set_constraint_dual_eq(-a("nu", p))
        model.reverse_differentiate(c["seed"])
        assert model.diff_time == model.diff_time
        dq, dQ = model.reverse_objective_function()
        got = dict(dq=dq, dQ=dQ, grad_z=dq, grad_lam=model.back_grad_cache[1], grad_nu=model.back_grad_cache[2],
                   dh=-np.array([model.get_db_le(i) for i in range(m)]),
                   db=-np.array([model.get_db_eq(i) for i in range(p)]),
                   dG=np.array([model.get_dA_le(i) for i in range(m)]).reshape(m, n),
                   dA=np.array([model.get_dA_eq(i) for i in range(p)]).reshape(p, n))
        keys = ["dq", "dh", "db"] if name == "qp_fixture_data" else c["exp"].keys()
        tol = c["tol"]
        for k in keys:
            e = np.array(c["exp"][k], float).ravel()
            g = np.asarray(got[k]).ravel()
            assert np.linalg.norm(g - e) <= max(tol, tol * max(np.linalg.norm(g), np.linalg.norm(e))), (name, k)
        if "fwd" in c:
            f = c["fwd"]
            fa = lambda k, shape: np.array(f[k], float).reshape(shape)
            model.forward_differentiate(fa("dQ", (n, n)), fa("dq", n), fa("dG", (m, n)), fa("dh", m),
                                        fa("dA", (p, n)), fa("db", p))
            assert np.allclose(model.forward_variable_primal(), c["exp_fwd"]["dz"], atol=tol)


def test_singular_kkt_reports_info(ctx):
    """test/conic_program.jl:846+ `test_singular_exception`-style: duplicated equality rows -> exact zero pivot."""
    qpm = diffopt_b200.submodule("qp")
    Q = np.eye(2)[None]
    A = np.array([[[1.0, 1.0], [1.0, 1.0]]])
    z = np.array([[0.5, 0.5]])
    fwd, rev, info = qpm.solve_batch(ctx, Q, None, A, None, z, None, np.zeros((1, 2)), seed=np.ones((1, 2)))
    assert info[0] > 0
    model = qpm.QPModel(ctx, np.eye(2), np.zeros(2), np.zeros((0, 2)), np.zeros(0), A[0], np.ones(2))
    model.set_variable_primal(z[0]); model.set_constraint_dual_le(np.zeros(0)); model.set_constraint_dual_eq(np.zeros(2))
    with pytest.raises(diffopt_b200.SingularException):
        model.reverse_differentiate(np.ones(2))


def test_full_size_batch_properties(ctx):
    """Config 2 at full size (4096 x n=64): size-independent properties instead of a 4096-instance oracle run.
    (a) residuals K x_b = -r_b and K' x_f = -r_f; (b) forward/reverse inner-product identity
    (test/utils.jl:331-337); (c) a 64-instance slice against the oracle."""
    qpm = diffopt_b200.submodule("qp")
    B = 4096
    d = bench_data.qp_batch_fast(B)
    n, m, p = 64, 64, 16
    fwd, rev, info = qpm.solve_batch(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"],
                                     fwd_dir=(d["dQ"], d["dq"], d["dG"], d["dh"], d["dA"], d["db"]), seed=d["seed"])
    assert not info.any()
    N = n + m + p
    K = np.zeros((B, N, N))
    K[:, :n, :n] = d["Q"]
    K[:, :n, n:n + m] = d["G"].transpose(0, 2, 1) * d["lam"][:, None, :]
    K[:, :n, n + m:] = d["A"].transpose(0, 2, 1)
    K[:, n:n + m, :n] = d["G"]
    K[:, n + m:, :n] = d["A"]
    idx = np.arange(m)
    K[:, n + idx, n + idx] = np.einsum("bij,bj->bi", d["G"], d["z"]) - d["h"]
    rb = np.zeros((B, N)); rb[:, :n] = d["seed"]
    rf = np.concatenate([
        np.einsum("bij,bj->bi", d["dQ"], d["z"]) + d["dq"] + np.einsum("bij,bi->bj", d["dG"], d["lam"]) +
        np.einsum("bij,bi->bj", d["dA"], d["nu"]),
        d["lam"] * (np.einsum("bij,bj->bi", d["dG"], d["z"]) - d["dh"]),
        np.einsum("bij,bj->bi", d["dA"], d["z"]) - d["db"]], axis=1)
    res_b = np.einsum("bij,bj->bi", K, rev) + rb
    res_f = np.einsum("bji,bj->bi", K, fwd) + rf
    scale_b = np.linalg.norm(K, axis=(1, 2)) * np.linalg.norm(rev, axis=1)
    scale_f = np.linalg.norm(K, axis=(1, 2)) * np.linalg.norm(fwd, axis=1)
    assert (np.linalg.norm(res_b, axis=1) / scale_b).max() < 1e-13
    assert (np.linalg.norm(res_f, axis=1) / scale_f).max() < 1e-13
    lhs = np.einsum("bi,bi->b", fwd[:, :n], d["seed"])
    rhs = np.einsum("bi,bi->b", rf, rev)
    assert np.abs(lhs - rhs).max() <= 1e-9 * np.abs(lhs).max()
    sl = slice(1000, 1064)
    sub = {k: v[sl] for k, v in d.items()}
    of, orv = _oracle_batch(sub)
    assert rel_err(fwd[sl], of).max() <= RTOL_DIRECT
    assert rel_err(rev[sl], orv).max() <= RTOL_DIRECT


# ---- the n=64, m=64, p=16 shape has three kernels: pivot-free LDL' fast path (default), pivoted LU
# (fallback and DIFFOPT_B200_QP_KERNEL=lu), generic LU (DIFFOPT_B200_QP_KERNEL=generic).

def _solve(ctx, d):
    qpm = diffopt_b200.submodule("qp")
    return qpm.solve_batch(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"],
                           fwd_dir=(d["dQ"], d["dq"], d["dG"], d["dh"], d["dA"], d["db"]), seed=d["seed"])


@pytest.mark.parametrize("kernel", ["ldl", "lu", "generic"])
def test_each_headline_kernel_matches_oracle(ctx, kernel, monkeypatch):
    monkeypatch.setenv("DIFFOPT_B200_QP_KERNEL", kernel)
    d = bench_data.qp_batch(48, seed0=4242)
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


@pytest.mark.parametrize("na", [0, 1, 7, 8, 9, 31, 40, 48])
def test_active_set_sizes(ctx, na):
    """Reduced-system order 80 + na: tile padding, pad pivots, every shared-memory configuration (na + 16 <= 64)."""
    d = bench_data.qp_batch(20, n_active=na, seed0=900 + na)
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


@pytest.mark.parametrize("na", [16, 41, 48, 50, 55, 57, 63])
def test_ldl_fast_path_serves_every_active_set_size(ctx, na, monkeypatch):
    """The pivot-free LDL' kernel itself (not its pivoted-LU safety net) must serve regular instances of every
    active-set size, including reduced orders 80 + na >= 128 that are not multiples of 8 (the identity padding rows
    are then indexed beyond the CTA size).  40 rows are active with slack 0 (with the 16 equalities: 56 < n = 64
    constraints, a well-conditioned KKT matrix); the other na - 40 rows of the reduced system carry lam > 0 with
    slack < 0, which keeps it quasi-definite at order 80 + na."""
    monkeypatch.setenv("DIFFOPT_B200_QP_KERNEL", "ldl")
    d = bench_data.qp_batch(12, n_active=min(na, 40), seed0=4100 + na)
    for b in range(12):
        idle = np.flatnonzero(d["lam"][b] == 0)[:max(0, na - 40)]
        d["lam"][b, idle] = 0.7
    _solve(ctx, d)                      # first call of this size: configures the launch for it
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    nfb, hint, kern = ctx.qp_last_stats()
    assert kern == 2 and nfb == 0, (nfb, hint, kern)
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


def test_ragged_active_sets_in_one_batch(ctx):
    parts = [bench_data.qp_batch(6, n_active=na, seed0=300 + na) for na in (0, 3, 16, 29, 45)]
    d = {k: np.concatenate([q[k] for q in parts]) for k in parts[0]}
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


def test_interior_point_style_duals(ctx):
    """Solver output instead of exact complementarity: inactive rows carry lam = 1e-9 (no exact zeros, so nothing is
    eliminated and the full N = 144 system is factorised), active rows carry slack -1e-9."""
    d = bench_data.qp_batch(16, seed0=77)
    act = d["lam"] > 0
    d["lam"] = np.where(act, d["lam"], 1e-9)
    slack = np.einsum("bij,bj->bi", d["G"], d["z"]) - d["h"]
    d["h"] = np.einsum("bij,bj->bi", d["G"], d["z"]) - np.where(act, -1e-9, slack)
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


def test_ldl_rejects_go_to_pivoted_lu(ctx):
    """Instances outside the LDL' path's assumptions must come back identical to the oracle through the fallback:
    (a) Q only positive SEMIdefinite (rank 40) but K nonsingular, (b) negative duals (wrong sign: K_s not
    quasi-definite), mixed with regular instances in one batch."""
    d = bench_data.qp_batch(24, seed0=555)
    rng = np.random.default_rng(5)
    for b in range(0, 24, 3):       # (a)
        L = rng.standard_normal((64, 40))
        d["Q"][b] = L @ L.T / 40
    for b in range(1, 24, 3):       # (b)
        d["lam"][b] = -d["lam"][b]
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


def test_singular_instance_inside_headline_batch(ctx):
    """LICQ violated in one instance (two identical active rows, K numerically singular): the LDL' path rejects it
    and the pivoted LU treats it like LAPACK would (info > 0 on an exactly zero pivot, otherwise a huge solution);
    the other instances of the batch are unaffected."""
    d = bench_data.qp_batch(8, seed0=31)
    act = np.flatnonzero(d["lam"][3] > 0)
    d["G"][3, act[1]] = d["G"][3, act[0]]
    d["h"][3, act[1]] = d["h"][3, act[0]]
    fwd, rev, info = _solve(ctx, d)
    assert not np.delete(info, 3).any()
    assert info[3] > 0 or not np.isfinite(rev[3]).all() or np.abs(rev[3]).max() > 1e8
    keep = np.arange(8) != 3
    of, orv = _oracle_batch({k: v[keep] for k, v in d.items()})
    assert rel_err(fwd[keep], of).max() <= RTOL_DIRECT
    assert rel_err(rev[keep], orv).max() <= RTOL_DIRECT


def test_stream_ordered_batch_calls(ctx):
    """diffopt_b200_qp_batch_solve_async + diffopt_b200_synchronize (device pointers, no host round trip between
    batches): three different batches enqueued back to back give the blocking call's results; the status of the last
    call (a batch with an exactly singular instance) surfaces at synchronize."""
    import torch
    capi = diffopt_b200.submodule("_capi")
    qpm = diffopt_b200.submodule("qp")
    lib = ctx.lib
    dev = torch.device("cuda", 0)
    fields = ["Q", "G", "A", "h", "z", "lam", "nu", "dQ", "dq", "dG", "dh", "dA", "db", "seed"]
    batches, outs = [], []
    for k in range(3):
        d = bench_data.qp_batch(40 + 8 * k, seed0=7000 + 100 * k)
        B = d["z"].shape[0]
        rows = {"Q": 64, "G": 64, "A": 16, "dQ": 64, "dG": 64, "dA": 16}   # matrices go column-major per instance
        t = {f: torch.from_numpy(qpm.colmajor(d[f], rows[f], 64, B) if f in rows else np.ascontiguousarray(d[f])).to(dev)
             for f in fields}
        o = dict(fwd=torch.empty((B, 144), dtype=torch.float64, device=dev),
                 rev=torch.empty((B, 144), dtype=torch.float64, device=dev),
                 info=torch.zeros(B, dtype=torch.int32, device=dev))
        batches.append((d, t, B))
        outs.append(o)
    torch.cuda.synchronize()
    for (d, t, B), o in zip(batches, outs):
        rc = lib.diffopt_b200_qp_batch_solve_async(ctx.h, B, 64, 64, 16, *[capi.vp(t[f].data_ptr()) for f in fields],
                                                   capi.vp(o["fwd"].data_ptr()), capi.vp(o["rev"].data_ptr()),
                                                   capi.vp(o["info"].data_ptr()))
        assert rc == 0
    assert lib.diffopt_b200_synchronize(ctx.h) == 0
    assert lib.diffopt_b200_synchronize(ctx.h) == 0      # idempotent
    for (d, t, B), o in zip(batches, outs):
        of, orv = _oracle_batch(d)
        assert not o["info"].cpu().numpy().any()
        assert rel_err(o["fwd"].cpu().numpy(), of).max() <= RTOL_DIRECT
        assert rel_err(o["rev"].cpu().numpy(), orv).max() <= RTOL_DIRECT
    # a singular instance: lam_i = D_i = 0 and a zero row of G make column n+i of LHS exactly zero
    d, t, B = batches[0]
    G = d["G"].copy(); h = d["h"].copy(); lam = d["lam"].copy()
    G[5, 2, :] = 0.0; lam[5, 2] = 0.0; h[5, 2] = 0.0
    tG, th, tl = (torch.from_numpy(x).to(dev) for x in (qpm.colmajor(G, 64, 64, B), h, lam))
    ptrs = {f: capi.vp(t[f].data_ptr()) for f in fields}
    ptrs.update(G=capi.vp(tG.data_ptr()), h=capi.vp(th.data_ptr()), lam=capi.vp(tl.data_ptr()))
    o = outs[0]
    assert lib.diffopt_b200_qp_batch_solve_async(ctx.h, B, 64, 64, 16, *[ptrs[f] for f in fields],
                                                 capi.vp(o["fwd"].data_ptr()), capi.vp(o["rev"].data_ptr()),
                                                 capi.vp(o["info"].data_ptr())) == 0
    assert lib.diffopt_b200_synchronize(ctx.h) == 6      # first failing instance + 1
    assert o["info"].cpu().numpy()[5] > 0
    # a failure in an EARLIER queued call is not lost behind later clean calls (info = NULL: every call shares the
    # library's own info buffer, the device-side sticky word carries the status)
    null = capi.vp(None)
    assert lib.diffopt_b200_qp_batch_solve_async(ctx.h, B, 64, 64, 16, *[ptrs[f] for f in fields],
                                                 capi.vp(o["fwd"].data_ptr()), capi.vp(o["rev"].data_ptr()), null) == 0
    for (d2, t2, B2), o2 in zip(batches[1:], outs[1:]):
        assert lib.diffopt_b200_qp_batch_solve_async(ctx.h, B2, 64, 64, 16, *[capi.vp(t2[f].data_ptr()) for f in fields],
                                                     capi.vp(o2["fwd"].data_ptr()), capi.vp(o2["rev"].data_ptr()), null) == 0
    assert lib.diffopt_b200_synchronize(ctx.h) == 6
    assert b"call 0" in lib.diffopt_b200_last_error(ctx.h)
    assert lib.diffopt_b200_synchronize(ctx.h) == 0


@pytest.mark.parametrize("N,nrhs", [(1, 1), (9, 1), (70, 3), (300, 16), (1100, 5)])
def test_direct_solve_system_csc(ctx, N, nrhs):
    """`LHS \\ RHS` drop-in (QuadraticProgram.jl:490): CSC and Adjoint{CSC}, one and many right-hand sides."""
    import scipy.sparse as sp
    lsq = diffopt_b200.submodule("lsqr")
    rng = np.random.default_rng(N)
    M = sp.random(N, N, density=min(1.0, 8.0 / N), random_state=N, format="csc") + sp.diags(rng.uniform(1, 2, N) * rng.choice([-1, 1], N))
    M = sp.csc_matrix(M)
    R = rng.standard_normal((N, nrhs))
    for trans in (False, True):
        X = lsq.solve_csc(ctx, M, R, trans=trans)
        ref = np.linalg.solve(M.toarray().T if trans else M.toarray(), R)
        assert (np.linalg.norm(X - ref, axis=0) / np.linalg.norm(ref, axis=0)).max() <= RTOL_DIRECT
    x1 = lsq.solve_csc(ctx, M, R[:, 0])
    assert np.allclose(x1, np.linalg.solve(M.toarray(), R[:, 0]), rtol=1e-9, atol=1e-12)


def test_direct_solve_system_kkt_and_singular(ctx, kat):
    """The reference's KKT matrix (create_LHS_matrix) of a known-answer case through the direct drop-in, both
    orientations as reverse (:335) and forward (:438) use them; exactly singular LHS -> SingularException."""
    lsq = diffopt_b200.submodule("lsqr")
    import scipy.sparse as sp
    c = kat["qp_moi_examples_2"]
    n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
    a = lambda k, shape: np.array(c[k], float).reshape(shape)
    K = oqp.create_lhs(a("z", n), a("lam", m), a("Q", (n, n)), a("G", (m, n)), a("h", m), a("A", (p, n)))
    rb = np.zeros(n + m + p); rb[:n] = c["seed"]
    x = -lsq.solve_csc(ctx, sp.csc_matrix(K), rb)
    dz, dl, dn = oqp.reverse(a("Q", (n, n)), a("G", (m, n)), a("h", m), a("A", (p, n)), a("z", n), a("lam", m), a("nu", p),
                             np.array(c["seed"], float))
    assert np.allclose(x, np.concatenate([dz, dl, dn]), rtol=1e-9, atol=1e-12)
    S = sp.csc_matrix(np.array([[1.0, 1.0, 0.0], [1.0, 1.0, 0.0], [0.0, 0.0, 1.0]]))
    with pytest.raises(diffopt_b200.SingularException):
        lsq.solve_csc(ctx, S, np.ones(3))


def test_extended_entry_shared_matrices_and_packed_triangles(ctx):
    """diffopt_b200_qp_batch_solve_ex: (a) Q, G, A (and the direction dQ, dG, dA) given once for the whole batch
    (OptNet layer with shared weights, SURVEY 8d) and (b) Q / dQ as packed lower triangles give exactly the results of
    the plain call on the expanded data -- headline shape (tuned kernels) and a generic shape."""
    qpm = diffopt_b200.submodule("qp")
    for (n, m, p, na) in ((64, 64, 16, 16), (12, 9, 3, 4)):
        d = bench_data.qp_batch(20, n, m, p, n_active=na, seed0=8800 + n, shared=True)
        fd = (d["dQ"], d["dq"], d["dG"], d["dh"], d["dA"], d["db"])
        # (twice: the first call of a new batch is configured with the previous batch's active-set size and may serve
        # instances from the pivoted-LU kernel, whose rounding differs; the bit-for-bit comparisons below are between calls
        # configured alike)
        for _ in range(2):
            f0, r0, i0 = qpm.solve_batch(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fd, seed=d["seed"])
        st0 = ctx.qp_last_stats()
        assert not i0.any()
        of, orv = _oracle_batch(d)
        assert rel_err(f0, of).max() <= RTOL_DIRECT and rel_err(r0, orv).max() <= RTOL_DIRECT
        # (a) one instance of Q, G, A
        f1, r1, i1 = qpm.solve_batch_ex(ctx, d["Q"][0], d["G"][0], d["A"][0], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fd,
                                        seed=d["seed"], shared_matrices=True)
        assert not i1.any() and np.array_equal(f1, f0) and np.array_equal(r1, r0), (st0, ctx.qp_last_stats())
        # (b) packed triangles (per instance), and both together with a shared direction
        f2, r2, _ = qpm.solve_batch_ex(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fd,
                                       seed=d["seed"], packed_q=True)
        assert np.array_equal(f2, f0) and np.array_equal(r2, r0)
        fd_sh = (d["dQ"][0], d["dq"], d["dG"][0], d["dh"], d["dA"][0], d["db"])
        f3, r3, _ = qpm.solve_batch_ex(ctx, d["Q"][0], d["G"][0], d["A"][0], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fd_sh,
                                       seed=d["seed"], shared_matrices=True, shared_direction=True, packed_q=True)
        B = d["z"].shape[0]
        d3 = dict(d, dQ=np.repeat(d["dQ"][:1], B, 0), dG=np.repeat(d["dG"][:1], B, 0), dA=np.repeat(d["dA"][:1], B, 0))
        of3, orv3 = _oracle_batch(d3)
        assert rel_err(f3, of3).max() <= RTOL_DIRECT and rel_err(r3, orv3).max() <= RTOL_DIRECT


@pytest.mark.parametrize("B,n,m,p", [(1, 3, 2, 1), (37, 64, 64, 16), (700, 10, 25, 0), (5, 7, 0, 2)])
def test_shared_parameter_gradients_batch_sum(ctx, B, n, m, p):
    """diffopt_b200_qp_batch_shared_grads (no collective: one rank): the device batch sum of the getters
    (QuadraticProgram.jl:307-314, :448-473) equals the sum of the oracle's per-instance gradients, and is bitwise
    reproducible from call to call (fixed summation order)."""
    qpm = diffopt_b200.submodule("qp")
    rng = np.random.default_rng(B + n)
    z, lam, nu = rng.standard_normal((B, n)), rng.uniform(0, 1, (B, m)), rng.standard_normal((B, p))
    rev = rng.standard_normal((B, n + m + p))
    got = qpm.shared_param_grads(ctx, z, lam if m else None, nu if p else None, rev)
    again = qpm.shared_param_grads(ctx, z, lam if m else None, nu if p else None, rev)
    refs = [oqp.reverse_param_grads(z[b], lam[b], nu[b], rev[b, :n], rev[b, n:n + m], rev[b, n + m:]) for b in range(B)]
    for k in range(6):
        want = sum(r[k] for r in refs)
        assert np.allclose(got[k], want, rtol=1e-10, atol=1e-10 * max(1.0, np.abs(want).max(initial=0.0))), k
        assert np.array_equal(got[k], again[k])


def test_nccl_path_on_a_single_rank_communicator(ctx):
    """The ctx-owned NCCL communicator (diffopt_b200_nccl_unique_id / _nccl_init) and the device-resident all-reduce of
    the shared-parameter gradients, exercised on ONE GPU (communicator of size 1: the all-reduce is the identity, but
    NCCL is bound, initialised and launched on the ctx stream exactly as with N ranks; the N = 2 check against the
    oracle is tests/test_multi_gpu.py and bench.py --gpus N)."""
    qpm = diffopt_b200.submodule("qp")
    sharding = diffopt_b200.submodule("sharding")
    d = bench_data.qp_batch(24, shared=True, seed0=99)
    sharding.nccl_init(ctx, 0, 1)
    try:
        rev, total = sharding.sharded_reverse_shared_params_device(ctx, d["Q"][0], d["G"][0], d["A"][0], d["h"], d["z"], d["lam"],
                                                                   d["nu"], d["seed"], 0, 1)
        plain = qpm.shared_param_grads(ctx, d["z"], d["lam"], d["nu"], rev, allreduce=True)
    finally:
        assert ctx.lib.diffopt_b200_nccl_destroy(ctx.h) == 0
    want = [0.0] * 6
    for b in range(24):
        dz, dl, dn = oqp.reverse(d["Q"][b], d["G"][b], d["h"][b], d["A"][b], d["z"][b], d["lam"][b], d["nu"][b], d["seed"][b])
        assert rel_err(rev[b], np.concatenate([dz, dl, dn])) <= RTOL_DIRECT
        want = [w + x for w, x in zip(want, oqp.reverse_param_grads(d["z"][b], d["lam"][b], d["nu"][b], dz, dl, dn))]
    for got, again, w in zip(total, plain, want):
        assert np.allclose(got, w, rtol=1e-8, atol=1e-9) and np.array_equal(got, again)
    # without a communicator the flag is refused, not ignored
    with pytest.raises(diffopt_b200.DiffOptB200Error):
        qpm.shared_param_grads(ctx, d["z"], d["lam"], d["nu"], rev, allreduce=True)


def test_c99_client_runs_the_reference_known_answer(tmp_path):
    """The plain-C client of tests/c_abi/c99_client.c (gcc -std=c99) drives create -> qp_batch_solve -> destroy on the GPU
    and reproduces the reference's literals of test/quadratic_program.jl:232-293."""
    import subprocess
    from test_abi_cpu import _build_c99_client
    exe = _build_c99_client(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "(ok)" in r.stdout, r.stdout + r.stderr


# ---- every other shape: the shape-generic LDL' fast path (qp_batch_sqd_any.cu) with the generic pivoted LU behind it

ANY_SHAPES = [(10, 25, 10, 0), (5, 0, 2, 0), (7, 9, 0, 3), (3, 0, 0, 0), (33, 47, 5, 11), (1, 1, 0, 1), (80, 60, 20, 30),
              (100, 50, 0, 12), (32, 32, 8, 8), (50, 100, 10, 20), (17, 130, 3, 9), (64, 64, 8, 16)]


@pytest.mark.parametrize("n,m,p,na", ANY_SHAPES)
def test_any_shape_ldl_fast_path_matches_oracle(ctx, n, m, p, na):
    """Regular instances of any (n, m, p) are served by the pivot-free LDL' kernel itself (kernel id 2, nothing handed to
    the pivoted LU): n not a multiple of 8 (identity padding of the z block), no inequalities, no equalities, m > 128."""
    B = 37
    d = bench_data.qp_batch(B, n, m, p, n_active=na, seed0=7000 + n + m)
    _solve(ctx, d)                      # first call of this shape: measures the active sets, configures the launch
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    nfb, hint, kern = ctx.qp_last_stats()
    assert kern == 2 and nfb == 0 and hint == na, (nfb, hint, kern)
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


def test_any_shape_growing_active_set_and_interior_point_duals(ctx):
    """A batch whose active sets outgrow the configuration of the previous call is still solved correctly (the oversize
    instances go to the pivoted LU), the next call is configured for it; duals without exact zeros make every row active."""
    n, m, p = 40, 30, 6
    small = bench_data.qp_batch(16, n, m, p, n_active=4, seed0=8100)
    large = bench_data.qp_batch(16, n, m, p, n_active=20, seed0=8200)
    _solve(ctx, small); _solve(ctx, small)
    for d in (large, large):
        fwd, rev, info = _solve(ctx, d)
        assert not info.any()
        of, orv = _oracle_batch(d)
        assert rel_err(fwd, of).max() <= RTOL_DIRECT and rel_err(rev, orv).max() <= RTOL_DIRECT
    nfb, hint, kern = ctx.qp_last_stats()
    assert kern == 2 and nfb == 0 and hint == 20, (nfb, hint, kern)
    ipm = {k: v.copy() for k, v in large.items()}
    ipm["lam"][ipm["lam"] == 0] = 1e-9
    for _ in range(2):
        fwd, rev, info = _solve(ctx, ipm)
    assert not info.any()
    nfb, hint, kern = ctx.qp_last_stats()
    assert kern == 2 and hint == m, (nfb, hint, kern)
    of, orv = _oracle_batch(ipm)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT and rel_err(rev, orv).max() <= RTOL_DIRECT


def test_any_shape_rejects_go_to_the_pivoted_lu(ctx):
    """Instances outside the fast path's assumptions (indefinite Q, singular KKT) inside a regular batch: the regular ones
    keep their fast-path results, the indefinite one is re-solved by the pivoted LU, the singular one reports info > 0."""
    n, m, p = 12, 10, 4
    d = bench_data.qp_batch(9, n, m, p, n_active=3, seed0=8300)
    d["Q"][2] = np.diag(np.r_[-1.0, np.ones(n - 1)]) + 0.0     # indefinite but nonsingular KKT
    d["A"][5][1] = d["A"][5][0]                                  # duplicated equality row: exactly singular
    _solve(ctx, d)
    fwd, rev, info = _solve(ctx, d)
    nfb, hint, kern = ctx.qp_last_stats()
    assert kern == 2 and nfb >= 2
    assert info[5] > 0 and not np.delete(info, 5).any()
    keep = np.delete(np.arange(9), 5)
    sub = {k: v[keep] for k, v in d.items()}
    of, orv = _oracle_batch(sub)
    assert rel_err(fwd[keep], of).max() <= RTOL_DIRECT
    assert rel_err(rev[keep], orv).max() <= RTOL_DIRECT


# ---- forward directions as sparse triplets (diffopt_b200_qp_batch_solve_coo): the reference's own packing of dQ, dG, dA

def _sparse_direction(d, density, seed):
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    out = {}
    for k in ("dQ", "dG", "dA"):
        X = d[k] * (rng.random(d[k].shape) < density)
        if k == "dQ":
            X = (X + X.transpose(0, 2, 1)) / 2
        out[k] = X
    return out, {k: [sp.coo_matrix(M) for M in X] for k, X in out.items()}


@pytest.mark.parametrize("n,m,p,na", [(64, 64, 16, 16), (33, 47, 5, 11), (5, 0, 2, 0), (80, 60, 20, 30)])
def test_sparse_triplet_directions_match_dense_call_and_oracle(ctx, n, m, p, na):
    """Sparse (I, J, V) directions (src/diff_opt.jl:594-656, QuadraticProgram.jl:396-424) give the dense call's answer."""
    qpm = diffopt_b200.submodule("qp")
    d = bench_data.qp_batch(19, n, m, p, n_active=na, seed0=9100 + n)
    dense, coo = _sparse_direction(d, 0.05, 1 + n)
    d.update(dense)
    for _ in range(2):
        fwd, rev, info = qpm.solve_batch_coo(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], dQ=coo["dQ"],
                                             dq=d["dq"], dG=coo["dG"], dh=d["dh"], dA=coo["dA"], db=d["db"], seed=d["seed"])
    assert not info.any()
    nfb, hint, kern = ctx.qp_last_stats()
    assert kern == 2 and nfb == 0
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT
    f2, _, _ = _solve(ctx, d)
    assert rel_err(fwd, f2).max() <= 1e-12


def test_sparse_triplet_edge_cases(ctx, monkeypatch):
    """Empty directions, duplicated triplets (added up like SparseArrays.sparse), one direction shared by the batch, an
    out-of-range index (argument error), and the generic pivoted-LU kernel consuming the assembled right-hand side."""
    import scipy.sparse as sp
    qpm = diffopt_b200.submodule("qp")
    n, m, p = 12, 9, 3
    d = bench_data.qp_batch(6, n, m, p, n_active=3, seed0=9300)
    z0 = {k: np.zeros_like(d[k]) for k in ("dQ", "dG", "dA")}
    base = dict(d); base.update(z0)
    fwd, _, _ = qpm.solve_batch_coo(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], dq=d["dq"], dh=d["dh"], db=d["db"])
    of, _ = _oracle_batch(base)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    # duplicates: the same entry twice with half the value each
    dG1 = np.zeros((m, n)); dG1[2, 5] = 1.5; dG1[7, 0] = -2.0
    dup = sp.coo_matrix((np.array([0.75, 0.75, -2.0]), (np.array([2, 2, 7]), np.array([5, 5, 0]))), shape=(m, n))
    shared = dict(base); shared["dG"] = np.broadcast_to(dG1, (6, m, n)).copy()
    fwd, _, _ = qpm.solve_batch_coo(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], dq=d["dq"], dG=dup, dh=d["dh"],
                                    db=d["db"], shared_direction=True)
    of, _ = _oracle_batch(shared)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    monkeypatch.setenv("DIFFOPT_B200_QP_KERNEL", "generic")
    f3, _, _ = qpm.solve_batch_coo(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], dq=d["dq"], dG=dup, dh=d["dh"],
                                   db=d["db"], shared_direction=True)
    monkeypatch.delenv("DIFFOPT_B200_QP_KERNEL")
    assert ctx.qp_last_stats()[2] == 0 and rel_err(f3, of).max() <= RTOL_DIRECT
    bad = (np.array([0, 1], np.int64), np.array([m + 1], np.int64), np.array([1], np.int64), np.array([1.0]))
    capi = diffopt_b200.submodule("_capi")
    st = capi.CooBatch(*[a.ctypes.data for a in bad])
    B = 6
    cm = lambda X, r: qpm.colmajor(X, r, n, B)
    out = np.empty((B, n + m + p)); info = np.zeros(B, np.int32)
    rc = ctx.lib.diffopt_b200_qp_batch_solve_coo(
        ctx.h, B, n, m, p, capi.ptr(cm(d["Q"], n)), capi.ptr(cm(d["G"], m)), capi.ptr(cm(d["A"], p)), capi.ptr(d["h"]), capi.ptr(d["z"]),
        capi.ptr(d["lam"]), capi.ptr(d["nu"]), None, None, capi.C.addressof(st), None, None, None, None, capi.ptr(out), None,
        capi.ptr(info), capi.HOST, capi.QP_SHARED_DIRECTION)
    assert rc == -1
    with pytest.raises(diffopt_b200.DiffOptB200Error, match="outside"):
        ctx.check(rc)


def test_qpmodel_takes_sparse_directions(ctx):
    import scipy.sparse as sp
    qpm = diffopt_b200.submodule("qp")
    n, m, p = 10, 7, 2
    d = bench_data.qp_batch(1, n, m, p, n_active=2, seed0=9400)
    model = qpm.QPModel(ctx, d["Q"][0], d["q"][0], d["G"][0], d["h"][0], d["A"][0], d["b"][0])
    model.set_variable_primal(d["z"][0]); model.set_constraint_dual_le(-d["lam"][0]); model.set_constraint_dual_eq(-d["nu"][0])
    dG = np.zeros((m, n)); dG[1, 3] = 1.0
    model.forward_differentiate(dG=sp.csr_matrix(dG), dh=d["dh"][0])
    got = model.forward_variable_primal().copy()
    model.forward_differentiate(dG=dG, dh=d["dh"][0])
    assert np.allclose(got, model.forward_variable_primal(), rtol=1e-10, atol=1e-13)


@pytest.mark.parametrize("n,m,p,na,fast", [(100, 100, 10, 15, True), (150, 60, 20, 25, True), (200, 150, 0, 10, True),
                                           (200, 150, 0, 40, False), (120, 260, 4, 12, False)])
def test_problems_beyond_the_shared_memory_lu(ctx, n, m, p, na, fast):
    """N = n + m + p > 165: the pivoted-LU kernel keeps its matrix in global memory (the safety net), the LDL' fast path still
    serves instances whose reduced system fits shared memory.  `fast`: every instance is expected on the fast path; otherwise
    the active set (or m > 255) is beyond it and the whole batch runs the global-memory LU -- same answers either way."""
    B = 6
    d = bench_data.qp_batch(B, n, m, p, n_active=na, seed0=9700 + n + m)
    _solve(ctx, d)
    fwd, rev, info = _solve(ctx, d)
    assert not info.any()
    nfb, hint, kern = ctx.qp_last_stats()
    if fast:
        assert kern == 2 and nfb == 0, (nfb, hint, kern)
    else:
        assert kern == 0 or nfb == B, (nfb, hint, kern)
    of, orv = _oracle_batch(d)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT


@pytest.mark.parametrize("n,m,p,na,nrhs", [(60, 60, 15, 15, 3), (120, 120, 31, 30, 1), (250, 250, 60, 60, 40), (400, 400, 100, 100, 5)])
def test_direct_solve_of_one_dense_kkt_system_blocked_lu(ctx, n, m, p, na, nrhs):
    """`LHS \\ RHS` for ONE QP with dense Q, G, A (N = 135 .. 900: block sizes that are and are not multiples of 32): the
    blocked partially pivoted LU over the whole GPU (kkt_dense.cu), both orientations, one and many right-hand sides, against
    a dense LAPACK solve; a structurally singular matrix of that size raises SingularException (numerically singular ones give a
    rounding-level pivot in any blocked LU, LAPACK's included)."""
    import scipy.sparse as sp
    lsq = diffopt_b200.submodule("lsqr")
    d = bench_data.qp_batch(1, n, m, p, n_active=na, seed0=9900 + n)
    K = oqp.create_lhs(d["z"][0], d["lam"][0], d["Q"][0], d["G"][0], d["h"][0], d["A"][0])
    N = K.shape[0]
    R = np.random.default_rng(n).standard_normal((N, nrhs))
    Kc = sp.csc_matrix(K)
    for trans in (False, True):
        X = lsq.solve_csc(ctx, Kc, R, trans=trans)
        ref = np.linalg.solve(K.T if trans else K, R)
        assert (np.linalg.norm(X - ref, axis=0) / np.linalg.norm(ref, axis=0)).max() <= RTOL_DIRECT
    Ks = K.copy()
    Ks[n + m + 1] = 0.0                # an equality row without entries: structurally singular, the zero pivot is exact
    with pytest.raises(diffopt_b200.SingularException):
        lsq.solve_csc(ctx, sp.csc_matrix(Ks), R)


def test_qpmodel_routes_one_large_dense_qp_to_the_blocked_lu(ctx):
    """A single QP beyond the batched kernels' shared-memory order (n = 300, m = 200, p = 40: N = 540) through the
    reference-shaped model: reverse and forward mode against the oracle."""
    qpm = diffopt_b200.submodule("qp")
    n, m, p = 300, 200, 40
    d = bench_data.qp_batch(1, n, m, p, n_active=30, seed0=9950)
    model = qpm.QPModel(ctx, d["Q"][0], d["q"][0], d["G"][0], d["h"][0], d["A"][0], d["b"][0])
    model.set_variable_primal(d["z"][0]); model.set_constraint_dual_le(-d["lam"][0]); model.set_constraint_dual_eq(-d["nu"][0])
    launches = ctx.launch_count
    model.reverse_differentiate(d["seed"][0])
    assert ctx.launch_count - launches > 20      # the blocked factorisation, not one batched launch
    of, orv = _oracle_batch(d)
    got = np.concatenate(model.back_grad_cache)
    assert rel_err(got, orv[0]) <= RTOL_DIRECT
    model.forward_differentiate(d["dQ"][0], d["dq"][0], d["dG"][0], d["dh"][0], d["dA"][0], d["db"][0])
    assert rel_err(np.concatenate(model.forw_grad_cache), of[0]) <= RTOL_DIRECT
