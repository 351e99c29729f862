"""Batched LSQR branch of the QP backend for LPs (Q = 0): ``diffopt_b200_qp_batch_solve_lsqr`` against the oracle, against
the single-instance ``lsqr_csc`` route QPModel takes, against the LP known answers, and the entry point's semantics."""
import ctypes as C

import numpy as np
import pytest

import bench_data
import diffopt_b200
from oracle import lsqr as olsqr
from oracle import qp as oqp

pytestmark = pytest.mark.gpu
TIGHT = dict(atol=1e-12, btol=1e-12, conlim=1e14, maxiter=5000)


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


@pytest.fixture(scope="module")
def qpm():
    return diffopt_b200.submodule("qp")


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


def lp_batch(B, n, m, p, n_active, seed0):
    """B random LPs with their own seeds: ``n_active`` active rows (lam ~ U(.5, 1.5), zero slack), the rest inactive;
    equality rows with nu ~ N(0, 1); a dense forward direction and a reverse seed per instance."""
    d = {k: np.zeros(s) for k, s in dict(G=(B, m, n), A=(B, p, n), h=(B, m), z=(B, n), lam=(B, m), nu=(B, p),
                                         dQ=(B, n, n), dq=(B, n), dG=(B, m, n), dh=(B, m), dA=(B, p, n), db=(B, p),
                                         seed=(B, n)).items()}
    for b in range(B):
        rng = np.random.default_rng(seed0 + b)
        G, A, z = rng.standard_normal((m, n)), rng.standard_normal((p, n)), rng.standard_normal(n)
        act = rng.permutation(m)[:n_active]
        lam = np.zeros(m)
        lam[act] = rng.uniform(0.5, 1.5, size=act.size)
        slack = -rng.uniform(0.5, 1.5, size=m)
        slack[act] = 0.0
        S = rng.standard_normal((n, n))
        d["G"][b], d["A"][b], d["z"][b], d["lam"][b], d["nu"][b] = G, A, z, lam, rng.standard_normal(p)
        d["h"][b] = G @ z - slack
        d["dQ"][b] = (S + S.T) / 2
        d["dq"][b], d["dG"][b], d["dh"][b] = rng.standard_normal(n), rng.standard_normal((m, n)), rng.standard_normal(m)
        d["dA"][b], d["db"][b], d["seed"][b] = rng.standard_normal((p, n)), rng.standard_normal(p), rng.standard_normal(n)
    return d


def fwd_dir(d, b=None):
    keys = ("dQ", "dq", "dG", "dh", "dA", "db")
    return tuple(d[k] if b is None else d[k][b] for k in keys)


def run(qpm, ctx, d, shared=False, **tol):
    return qpm.solve_batch_lsqr(ctx, d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fwd_dir(d),
                                seed=d["seed"], shared_matrices=shared, **tol)


def oracle(d, b, **tol):
    n = d["z"].shape[1]
    Q = np.zeros((n, n))
    args = (Q, d["G"][b], d["h"][b], d["A"][b], d["z"][b], d["lam"][b], d["nu"][b])
    f = np.concatenate(oqp.forward(*args, *fwd_dir(d, b), **tol))
    r = np.concatenate(oqp.reverse(*args, d["seed"][b], **tol))
    return f, r


SHAPES = [(200, 100, 0, 60), (64, 64, 16, 40), (30, 0, 10, 0), (40, 25, 0, 10), (400, 200, 8, 120)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[:3])))
@pytest.mark.parametrize("B", [1, 7, 300])
def test_parity_with_oracle_at_convergence(ctx, qpm, shape, B):
    n, m, p, na = shape
    d = lp_batch(B, n, m, p, na, seed0=1000 * B + n)
    fwd, rev, st = run(qpm, ctx, d, **TIGHT)
    assert fwd.shape == rev.shape == (B, n + m + p) and st.shape == (B, 2, 4)
    check = range(B) if B <= 7 else np.linspace(0, B - 1, 6).astype(int)
    for b in check:
        f, r = oracle(d, b, **TIGHT)
        assert rel(fwd[b], f) <= 1e-6, (b, rel(fwd[b], f), st[b])
        assert rel(rev[b], r) <= 1e-6, (b, rel(rev[b], r), st[b])
        assert st[b, :, 0].min() >= 1 and st[b, :, 0].max() <= 3


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[:3])))
def test_fixed_iteration_counts_match_oracle_iterates(ctx, qpm, shape):
    n, m, p, na = shape
    d = lp_batch(3, n, m, p, na, seed0=77)
    for mi in (1, 3, 6):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=mi)
        fwd, rev, st = run(qpm, ctx, d, **tol)
        assert (st[:, :, 0] == 7).all() and (st[:, :, 1] == mi).all()
        for b in range(3):
            f, r = oracle(d, b, **tol)
            assert rel(fwd[b], f) <= 1e-10 and rel(rev[b], r) <= 1e-10, (mi, b)


# (shape, iteration slack, tolerance on the answer of a solve that stopped on a convergence test)
SINGLE = [(SHAPES[0], 0.05, 1e-6), (SHAPES[1], 0.15, 1e-4), (SHAPES[2], 0.05, 1e-6), (SHAPES[3], 0.05, 1e-6),
          (SHAPES[4], 0.05, 1e-6)]


@pytest.mark.parametrize("shape,slack,tol", SINGLE, ids=["x".join(map(str, c[0][:3])) for c in SINGLE])
def test_against_single_instance_lsqr_csc(ctx, qpm, shape, slack, tol):
    """Each instance against the route QPModel takes (host-built KKT CSC, lsqr_csc) at default tolerances: the same stop
    code, the iteration count within max(2, 5 %) (the ||M'r|| test is sensitive to summation order), the same answer to
    1e-6.  The 64/64/16 shape is the exception: its forward solves reach the cap of N iterations (istop 7), where both
    routes stop at the same count and their unconverged iterates differ by up to 2.2e-3 (checked to 1e-2), and the ||M'r||
    estimate of its reverse solves is flat near the stop (81 against 72 iterations seen for one instance), so it gets
    15 % and 1e-4."""
    lsqr = diffopt_b200.submodule("lsqr")
    n, m, p, na = shape
    d = lp_batch(4, n, m, p, na, seed0=5)
    fwd, rev, st = run(qpm, ctx, d)
    for b in range(4):
        model = qpm.QPModel(ctx, np.zeros((n, n)), np.zeros(n), d["G"][b], d["h"][b], d["A"][b], np.zeros(p))
        model.set_variable_primal(d["z"][b]); model.set_constraint_dual_le(-d["lam"][b])
        model.set_constraint_dual_eq(-d["nu"][b])
        K = model._lhs_csc()
        rr = np.zeros(n + m + p); rr[:n] = d["seed"][b]
        for k, (trans, rhs, got) in enumerate([(True, model._forward_rhs(*fwd_dir(d, b)), fwd[b]), (False, rr, rev[b])]):
            x, s = lsqr.lsqr_csc(ctx, K, rhs, trans=trans)
            assert st[b, k, 0] == s["istop"], (n, b, k, st[b, k], s)
            assert abs(st[b, k, 1] - s["itn"]) <= max(2, slack * s["itn"]), (n, b, k, st[b, k], s)
            assert rel(got, -x) <= (1e-2 if s["istop"] == 7 else tol), (n, b, k, rel(got, -x), st[b, k], s)


def test_config1_min_norm_and_iteration_counts(ctx, qpm):
    d = bench_data.lp_config1()
    n, m = 200, 100
    one = lambda v: np.asarray(v, float)[None]
    _, rev, st = qpm.solve_batch_lsqr(ctx, one(d["G"]), None, one(d["h"]), one(d["z"]), one(d["lam"]), None,
                                      seed=one(d["seed"]), **TIGHT)
    K = oqp.create_lhs(d["z"], d["lam"], d["Q"], d["G"], d["h"], d["A"])
    rhs = np.zeros(n + m); rhs[:n] = d["seed"]
    assert rel(rev[0], -np.linalg.pinv(K) @ rhs) <= 1e-5
    _, _, st = qpm.solve_batch_lsqr(ctx, one(d["G"]), None, one(d["h"]), one(d["z"]), one(d["lam"]), None,
                                    seed=one(d["seed"]))
    _, info = olsqr.lsqr(K, rhs, return_info=True)
    assert st[0, 1, 0] == info.istop == 2 and abs(st[0, 1, 1] - info.itn) <= max(2, 0.05 * info.itn)


def test_lp_known_answers_through_the_batch(ctx, qpm, kat):
    for name in ["lp_simplex_example", "lp_fixed_variable", "lp_nonactive"]:
        c = kat[name]
        n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
        a = lambda k, shape: np.array(c[k], float).reshape(shape)
        assert not a("Q", (n, n)).any()
        z, lam, nu = a("z", n), a("lam", m), a("nu", p)
        fd = None
        if "fwd" in c:
            f = c["fwd"]
            fa = lambda k, shape: np.array(f[k], float).reshape((1,) + shape)
            fd = (fa("dQ", (n, n)), fa("dq", (n,)), fa("dG", (m, n)), fa("dh", (m,)), fa("dA", (p, n)), fa("db", (p,)))
        fwd, rev, _ = qpm.solve_batch_lsqr(ctx, a("G", (1, m, n)), a("A", (1, p, n)) if p else None, a("h", (1, m)),
                                           z[None], lam[None], nu[None] if p else None, fwd_dir=fd,
                                           seed=np.array(c["seed"], float)[None])
        dz, dlam, dnu = rev[0, :n], rev[0, n:n + m], rev[0, n + m:]
        _, dq, dG, dh, dA, db = oqp.reverse_param_grads(z, lam, nu, dz, dlam, dnu)
        got = dict(dq=dq, grad_z=dq, grad_lam=dlam, dh=dh, db=db, dG=dG, dA=dA)
        for k, e in c["exp"].items():
            e = np.array(e, float).ravel(); g = np.asarray(got[k]).ravel()
            assert np.linalg.norm(g - e) <= max(c["tol"], c["tol"] * max(np.linalg.norm(g), np.linalg.norm(e))), (name, k)
        if fd is not None:
            assert np.allclose(fwd[0, :n], c["exp_fwd"]["dz"], atol=c["tol"])


def test_kat8_dispatch_lp_forward_directions_as_one_shared_batch(ctx, qpm, kat):
    c = kat["lp_dispatch_sensitivity"]
    n, m, p = len(c["z"]), len(c["lam"]), len(c["nu"])
    a = lambda k, shape: np.array(c[k], float).reshape(shape)
    Q, G, A, z, lam = a("Q", (n, n)), a("G", (m, n)), a("A", (p, n)), a("z", n), a("lam", m)
    K = np.block([[Q, G.T, A.T], [np.diag(lam) @ G, np.diag(G @ z - a("h", m)), np.zeros((m, p))],
                  [A, np.zeros((p, m)), np.zeros((p, p))]])
    R = np.block([[np.zeros((n, m)), np.zeros((n, p))], [np.diag(lam), np.zeros((m, p))], [np.zeros((p, m)), np.eye(p)]])
    k = len(c["directions"])
    dh, db = np.zeros((k, m)), np.zeros((k, p))
    for i, dct in enumerate(c["directions"]):
        (dh if dct["kind"] == "dh" else db)[i, dct["index"]] = dct["value"]
    rep = lambda v: np.repeat(v[None], k, axis=0)
    fwd, _, _ = qpm.solve_batch_lsqr(ctx, G, A, rep(a("h", m)), rep(z), rep(lam), rep(a("nu", p)),
                                     fwd_dir=(None, None, None, dh, None, db), shared_matrices=True)
    for i, dct in enumerate(c["directions"]):
        col = olsqr.lsqr(K, R[:, i])[:n]
        got = -fwd[i, :n]
        want = dct["kkt_sign"] * col
        assert np.linalg.norm(got - want) <= max(c["tol"], c["tol"] * max(np.linalg.norm(got), np.linalg.norm(want))), i


def test_bitwise_semantics(ctx, qpm):
    n, m, p = 64, 64, 16
    d = lp_batch(300, n, m, p, 40, seed0=900)
    # shared G, A: the same as repeating them per instance
    ds = dict(d)
    ds["G"], ds["A"] = np.repeat(d["G"][:1], 300, axis=0), np.repeat(d["A"][:1], 300, axis=0)
    f1, r1, s1 = run(qpm, ctx, ds)
    f2, r2, s2 = qpm.solve_batch_lsqr(ctx, d["G"][0], d["A"][0], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fwd_dir(ds),
                                      seed=d["seed"], shared_matrices=True)
    assert np.array_equal(f1, f2) and np.array_equal(r1, r2) and np.array_equal(s1, s2)
    # reproducible, and instance b alone equals instance b inside the batch
    fa, ra, sa = run(qpm, ctx, d)
    fb, rb, sb = run(qpm, ctx, d)
    assert np.array_equal(fa, fb) and np.array_equal(ra, rb) and np.array_equal(sa, sb)
    for b in (0, 123, 299):
        one = {k: v[b:b + 1] for k, v in d.items()}
        f, r, s = run(qpm, ctx, one)
        assert np.array_equal(f[0], fa[b]) and np.array_equal(r[0], ra[b]) and np.array_equal(s[0], sa[b])
    # one mode alone gives the same bits as both modes together; the skipped mode reports zero statistics
    f, r, s = qpm.solve_batch_lsqr(ctx, d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=fwd_dir(d))
    assert r is None and np.array_equal(f, fa) and np.array_equal(s[:, 0], sa[:, 0]) and not s[:, 1].any()
    f, r, s = qpm.solve_batch_lsqr(ctx, d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], seed=d["seed"])
    assert f is None and np.array_equal(r, ra) and np.array_equal(s[:, 1], sa[:, 1]) and not s[:, 0].any()


def test_zero_directions_and_default_maxiter(ctx, qpm):
    n, m, p = 40, 25, 5
    d = lp_batch(4, n, m, p, 10, seed0=3)
    zero = tuple(np.zeros_like(v) for v in fwd_dir(d))
    f, r, s = qpm.solve_batch_lsqr(ctx, d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], fwd_dir=zero,
                                   seed=np.zeros((4, n)))
    assert not f.any() and not r.any() and (s[:, :, 1] == 0).all()
    f, r, s = qpm.solve_batch_lsqr(ctx, d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"],
                                   fwd_dir=(None, None, None, None, None, None), seed=None)
    assert not f.any() and not s.any()
    # maxiter = 0 (None) means N = n + m + p: with zero tolerances every solve runs exactly N iterations
    _, _, s = run(qpm, ctx, d, atol=0.0, btol=0.0, conlim=0.0, maxiter=None)
    _, _, s2 = run(qpm, ctx, d, atol=0.0, btol=0.0, conlim=0.0, maxiter=n + m + p)
    assert np.array_equal(s, s2) and (s[:, :, 1] <= n + m + p).all()
    assert (s[:, :, 1][s[:, :, 0] == 7] == n + m + p).all()


def test_device_memspace_with_torch_tensors(ctx, qpm):
    torch = pytest.importorskip("torch")
    _capi = diffopt_b200.submodule("_capi")
    n, m, p = 64, 64, 16
    B = 9
    d = lp_batch(B, n, m, p, 40, seed0=42)
    fh, rh, sh = run(qpm, ctx, d)
    cm = lambda X, r: torch.from_numpy(qpm.colmajor(X, r, n, B)).cuda()
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).cuda()
    dev = [cm(d["G"], m), cm(d["A"], p), t(d["h"]), t(d["z"]), t(d["lam"]), t(d["nu"]), cm(d["dQ"], n), t(d["dq"]),
           cm(d["dG"], m), t(d["dh"]), cm(d["dA"], p), t(d["db"]), t(d["seed"])]
    fwd = torch.empty((B, n + m + p), dtype=torch.float64, device="cuda")
    rev = torch.empty_like(fwd)
    st = torch.empty((B, 2, 4), dtype=torch.float64, device="cuda")
    L = olsqr
    torch.cuda.synchronize()
    rc = ctx.lib.diffopt_b200_qp_batch_solve_lsqr(ctx.h, B, n, m, p, *[_capi.ptr(x) for x in dev], L.SQRT_EPS, L.SQRT_EPS,
                                                  1 / L.SQRT_EPS, 0, _capi.ptr(fwd), _capi.ptr(rev), _capi.ptr(st),
                                                  _capi.DEVICE, 0)
    ctx.check(rc)
    assert np.array_equal(fwd.cpu().numpy(), fh) and np.array_equal(rev.cpu().numpy(), rh)
    assert np.array_equal(st.cpu().numpy(), sh)
    assert ctx.last_kernel_ms > 0


def test_bad_arguments_and_oversize(ctx, qpm):
    lib, h = ctx.lib, ctx.h
    z = np.zeros(4)
    out = np.zeros(4)
    call = lambda B, n, zz, flags, m=0: lib.diffopt_b200_qp_batch_solve_lsqr(
        h, B, n, m, 0, *([None] * 3), None if zz is None else zz.ctypes.data_as(C.c_void_p), *([None] * 9),
        1e-8, 1e-8, 1e8, 0, None, out.ctypes.data_as(C.c_void_p), None, 0, flags)
    assert call(-1, 4, z, 0) == -1
    assert call(1, 0, z, 0) == -1
    assert call(1, 4, None, 0) == -1
    assert call(1, 4, z, 2) == -1 and call(1, 4, z, 1 << 8) == -1
    assert call(1, 4, z, 0) == 0 and call(0, 4, z, 0) == 0
    # an instance whose LSQR vectors alone exceed one CTA's shared memory
    n = 4000
    zb = np.zeros(n)
    rc = lib.diffopt_b200_qp_batch_solve_lsqr(h, 1, n, 0, 0, *([None] * 3), zb.ctypes.data_as(C.c_void_p),
                                              *([None] * 9), 1e-8, 1e-8, 1e8, 0, None, None, None, 0, 0)
    assert rc == -3
