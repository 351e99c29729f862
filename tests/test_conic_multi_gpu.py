"""Many sensitivity directions per LSQR launch (diffopt_b200_conic_forward_multi / _reverse_multi): every direction of a
multi call against the oracle and against its own single-direction call, the zero tests inside a group, independence
of the other directions and reproducibility (bitwise), full size, each launch route by kernel name, and bad input."""
import re

import numpy as np
import pytest
import scipy.sparse as sp

import bench_data
import diffopt_b200
import pow_cone_oracle
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
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"], d.get("cone_params"))
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    return model


def _cache(d):
    return pow_cone_oracle.gradient_cache(d["A"], d["b"], d["c"], d["x"], d["s"], d["y"], d["cone_types"],
                                          d["cone_dims"], d.get("cone_params"))


def _directions(d, k, seed):
    """k forward directions (dA, db, dc) and k reverse seeds, reproducible from `seed`."""
    m, n = d["A"].shape
    rng = np.random.default_rng(seed)
    dAs = [sp.random(m, n, density=0.01, random_state=seed * 100 + j).tocsc() for j in range(k)]
    return dAs, rng.normal(size=(k, m)), rng.normal(size=(k, n)), rng.normal(size=(k, n))


def _fwd_rhs(cache, dA, db, dc):
    return np.concatenate([dA.T @ cache.vp + dc, -(dA @ cache.x) + db, [-(dc @ cache.x) - db @ cache.vp]])


def _rev_rhs(cache, seed):
    return np.concatenate([seed, np.zeros(cache.b.size), [-(cache.x @ seed)]])


def _oracle(cache, rhs, **tol):
    return olsqr.lsqr(cache.M, rhs, return_info=True, **tol)


def kernels_run(fn):
    """(names of the CUDA kernels `fn` launched, fn's result); fails when the profiler records no kernel."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    kernels = {n for n in names if not n.startswith(("Memcpy", "Memset"))}
    assert kernels, f"the profiler recorded no kernel (events: {sorted(names)})"
    return kernels, out


def ran(names, pattern):
    return any(re.search(pattern, n) for n in names)


PROBLEMS = {
    "psd6": lambda: bench_data.conic_config4(n=200, n_zero=20, n_nonneg=160, n_soc=12, soc_dim=10, nnz_per_row=6, seed=21,
                                             psd_sides=(6,)),
    "psd4_7": lambda: bench_data.conic_config4(n=200, n_zero=20, n_nonneg=160, n_soc=12, soc_dim=10, nnz_per_row=6,
                                               seed=22, psd_sides=(4, 7)),
    "exp_pow": lambda: bench_data.conic_exp_problem(n=200, n_zero=20, n_nonneg=120, n_soc=6, soc_dim=5, n_exp=6,
                                                    n_dual_exp=4, nnz_per_row=6, seed=34, n_pow=16, n_dual_pow=14),
}


def _itn_slack(info):
    return max(3, info.itn // (50 if info.istop == 1 else 20))


@pytest.mark.parametrize("name", sorted(PROBLEMS))
def test_multi_matches_oracle_every_cone_kind(ctx, name):
    """Every direction of forward and reverse multi calls with k = 1, 3, 8, 13 (across the group boundaries of 4 and 8
    directions) against the oracle at matched tight tolerances: the solution, the getters, istop and itn.  Directions
    whose right-hand side is not in the range of M stop on ||M'r|| (istop 2); that estimate is flat there, and two
    summation orders move the stop by up to a few percent of the iterations, so their itn is held to 5 %."""
    d = PROBLEMS[name]()
    model = _model(ctx, d)
    cache = _cache(d)
    m, n = d["A"].shape
    kw = dict(TIGHT, maxiter=20000)
    model.tolerances = kw
    K = 13
    dAs, dbs, dcs, seeds = _directions(d, K, 3)
    fwd = [_oracle(cache, _fwd_rhs(cache, dAs[j], dbs[j], dcs[j]), **kw) for j in range(K)]
    rev = [_oracle(cache, _rev_rhs(cache, seeds[j]), **kw) for j in range(K)]
    for k in (1, 3, 8, 13):
        f = model.forward_differentiate_multi(dAs[:k], dbs[:k], dcs[:k])
        r = model.reverse_differentiate_multi(seeds[:k])
        for j in range(k):
            dz, info = fwd[j]
            assert rel(f["dz"][j], dz) <= RTOL_LSQR, (name, k, j)
            assert rel(f["dx"][j], -(dz[:n] - cache.x * dz[n + m])) <= RTOL_LSQR
            assert f["stats"][j, 0] == info.istop and abs(f["stats"][j, 1] - info.itn) <= _itn_slack(info)
            g, info = rev[j]
            _, db, dc = oconic.reverse_param_grads(cache, g, dense_dA=False)
            assert rel(r["g"][j], g) <= RTOL_LSQR, (name, k, j)
            assert rel(r["dc"][j], dc) <= RTOL_LSQR and rel(r["db"][j], db) <= RTOL_LSQR
            assert r["stats"][j, 0] == info.istop and abs(r["stats"][j, 1] - info.itn) <= _itn_slack(info)


def _conditioned(n=400, seed=4):
    return bench_data.conic_config4_conditioned(n=n, n_zero=40, n_nonneg=320, n_soc=24, soc_dim=10, nnz_per_row=8,
                                                seed=seed)


def test_multi_matches_single_calls(ctx):
    """Each direction of a multi call equals its own conic_forward / conic_reverse on the same setup (<= 1e-9, same
    istop).  Directions of very different scales stop after different iteration counts: the ones that stop first are
    frozen while their group goes on."""
    d = _conditioned()
    model = _model(ctx, d)
    model.tolerances = dict(atol=1e-13, btol=1e-13, conlim=0.0, maxiter=20000)
    k = 11
    dAs, dbs, dcs, seeds = _directions(d, k, 5)
    scale = np.logspace(-3, 3, k)
    dbs *= scale[:, None]
    seeds[:, : seeds.shape[1] // 2] *= scale[:, None]
    f = model.forward_differentiate_multi(dAs, dbs, dcs)
    r = model.reverse_differentiate_multi(seeds)
    itns = set()
    for j in range(k):
        model.forward_differentiate(dAs[j], dbs[j], dcs[j])
        assert rel(f["dx"][j], model.forward_variable_primal()) <= 1e-9, j
        assert rel(f["dz"][j], np.concatenate(model.forw_grad_cache[:3])) <= 1e-9
        assert f["stats"][j, 0] == model.last_stats["istop"]
        model.reverse_differentiate(seeds[j])
        assert rel(r["g"][j], model.back_grad_cache["g"]) <= 1e-9, j
        assert rel(r["dc"][j], model.back_grad_cache["dc"]) <= 1e-9 and rel(r["db"][j], model.back_grad_cache["db"]) <= 1e-9
        assert r["stats"][j, 0] == model.last_stats["istop"]
        itns |= {f["stats"][j, 1], r["stats"][j, 1]}
    assert len(itns) > 2


def test_multi_zero_tests_inside_a_group(ctx):
    """An all-zero forward direction (:320) and a reverse seed of norm below 1e-4 (:369) in the middle of a group return
    exact zeros and zero statistics; their neighbours still match the oracle."""
    d = PROBLEMS["exp_pow"]()
    model = _model(ctx, d)
    cache = _cache(d)
    m, n = d["A"].shape
    kw = dict(TIGHT, maxiter=20000)
    model.tolerances = kw
    k, z = 8, 3
    dAs, dbs, dcs, seeds = _directions(d, k, 7)
    dAs[z] = None
    dbs[z] = 0.0
    dcs[z] = 0.0
    seeds[z] = 1e-6
    f = model.forward_differentiate_multi(dAs, dbs, dcs)
    r = model.reverse_differentiate_multi(seeds)
    assert not f["dx"][z].any() and not f["dz"][z].any() and not f["stats"][z].any()
    assert not r["g"][z].any() and not r["dc"][z].any() and not r["db"][z].any() and not r["stats"][z].any()
    for j in (z - 1, z + 1):
        dz, _ = _oracle(cache, _fwd_rhs(cache, dAs[j], dbs[j], dcs[j]), **kw)
        assert rel(f["dz"][j], dz) <= RTOL_LSQR
        g, _ = _oracle(cache, _rev_rhs(cache, seeds[j]), **kw)
        assert rel(r["g"][j], g) <= RTOL_LSQR


def test_multi_independent_reproducible_and_device_memory(ctx):
    """Direction j gives the same bits when the other directions are replaced or the directions permuted, a repeated
    call gives the same bits, and a device-memory call gives the bits of the host-memory call."""
    import torch
    capi = diffopt_b200.submodule("_capi")
    d = _conditioned(n=300, seed=9)
    model = _model(ctx, d)
    model.tolerances = dict(atol=1e-10, btol=1e-10, conlim=0.0, maxiter=20000)
    m, n = d["A"].shape
    k = 13
    dAs, dbs, dcs, seeds = _directions(d, k, 11)
    oA, ob, oc, os_ = _directions(d, k, 12)
    f = model.forward_differentiate_multi(dAs, dbs, dcs)
    r = model.reverse_differentiate_multi(seeds)
    perm = np.random.default_rng(0).permutation(k)
    for sel in ([0, 5, 12], [1, 7]):
        # keep the selected directions, permute them into other slots, replace every other direction
        A2, b2, c2, s2 = list(oA), ob.copy(), oc.copy(), os_.copy()
        for j in sel:
            q = int(perm[j])
            A2[q], b2[q], c2[q], s2[q] = dAs[j], dbs[j], dcs[j], seeds[j]
        f2 = model.forward_differentiate_multi(A2, b2, c2)
        r2 = model.reverse_differentiate_multi(s2)
        for j in sel:
            q = int(perm[j])
            assert np.array_equal(f2["dz"][q], f["dz"][j]) and np.array_equal(f2["stats"][q], f["stats"][j])
            assert np.array_equal(r2["g"][q], r["g"][j]) and np.array_equal(r2["stats"][q], r["stats"][j])
    f3 = model.forward_differentiate_multi(dAs, dbs, dcs)
    r3 = model.reverse_differentiate_multi(seeds)
    for key in f:
        assert np.array_equal(f3[key], f[key])
    for key in r:
        assert np.array_equal(r3[key], r[key])
    # device memory: the same call with every pointer on the device
    keep = []

    def dev(a):
        keep.append(torch.from_numpy(np.ascontiguousarray(a)).cuda())
        return keep[-1]
    tol = model._tol()
    g, dc, db, st = (torch.empty((k, L), dtype=torch.float64, device="cuda") for L in (n + m + 1, n, m, 4))
    rc = ctx.lib.diffopt_b200_conic_reverse_multi(ctx.h, k, capi.ptr(dev(seeds)), *tol, capi.ptr(g), capi.ptr(dc),
                                                  capi.ptr(db), capi.ptr(st), capi.DEVICE)
    ctx.check(rc)
    torch.cuda.synchronize()
    for a, key in ((g, "g"), (dc, "dc"), (db, "db"), (st, "stats")):
        assert np.array_equal(a.cpu().numpy(), r[key])
    arrs = diffopt_b200.submodule("qp").coo_batch(dAs, k)
    darrs = [dev(a) for a in arrs]
    coo = capi.CooBatch(*[capi.ptr(a) for a in darrs])
    dx, dz, st = (torch.empty((k, L), dtype=torch.float64, device="cuda") for L in (n, n + m + 1, 4))
    rc = ctx.lib.diffopt_b200_conic_forward_multi(ctx.h, k, capi.C.addressof(coo), capi.ptr(dev(dbs)), capi.ptr(dev(dcs)),
                                                  *tol, capi.ptr(dx), capi.ptr(dz), capi.ptr(st), capi.DEVICE)
    ctx.check(rc)
    torch.cuda.synchronize()
    for a, key in ((dx, "dx"), (dz, "dz"), (st, "stats")):
        assert np.array_equal(a.cpu().numpy(), f[key])


def test_multi_config4_full_size(ctx):
    """BASELINE config 4 (n = 5000, m = 7500): reverse with k = 8 iterate by iterate against the oracle at 3 and 10
    iterations, LSQR's residual estimate per direction against the true residual; the conditioned generator converged at
    the default tolerances with k = 4 against the oracle."""
    d = bench_data.conic_config4()
    model = _model(ctx, d)
    cache = _cache(d)
    m, n = d["A"].shape
    seeds = np.random.default_rng(2).normal(size=(8, n))
    seeds[0] = d["seed"]
    for iters in (3, 10):
        tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        model.tolerances = tol
        r = model.reverse_differentiate_multi(seeds)
        assert (r["stats"][:, 1] == iters).all() and (r["stats"][:, 0] == 7).all()
        for j in range(8):
            assert rel(r["g"][j], oconic.reverse(cache, seeds[j], **tol)) <= 1e-9, (iters, j)
            dz = _rev_rhs(cache, seeds[j])
            res = model.M_apply(r["g"][j]) - dz
            assert abs(np.linalg.norm(res) - r["stats"][j, 2]) <= 1e-8 * np.linalg.norm(dz)
    d = bench_data.conic_config4_conditioned()
    model = _model(ctx, d)
    cache = _cache(d)
    tol = dict(atol=olsqr.SQRT_EPS, btol=olsqr.SQRT_EPS, conlim=1 / olsqr.SQRT_EPS, maxiter=12501)
    model.tolerances = tol
    seeds = np.random.default_rng(3).normal(size=(4, n))
    seeds[0] = d["seed"]
    r = model.reverse_differentiate_multi(seeds)
    for j in range(4):
        g, info = _oracle(cache, _rev_rhs(cache, seeds[j]), **tol)
        assert r["stats"][j, 0] == info.istop == 1
        assert rel(r["g"][j], g) <= RTOL_LSQR, j


def _single_parity(model, r, seeds, js, bound=1e-9):
    for j in js:
        model.reverse_differentiate(seeds[j])
        assert rel(r["g"][j], model.back_grad_cache["g"]) <= bound, j


def test_multi_routes_by_kernel_name(ctx):
    """Cluster per group (small operator, no PSD cones), including more groups than clusters fit on the GPU at once;
    the cooperative grid per group (an operator above the cluster route's size limit, and a problem with PSD cones)."""
    tol = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=3)
    # small operator: one cluster per group, KB = 4 and 8
    d = PROBLEMS["exp_pow"]()
    model = _model(ctx, d)
    model.tolerances = tol
    n = d["A"].shape[1]
    seeds = np.random.default_rng(4).normal(size=(640, n))
    names, r = kernels_run(lambda: model.reverse_differentiate_multi(seeds[:3]))
    assert ran(names, r"lsqr_multi_kernel<4, true>") and not ran(names, r"lsqr_kernel_t|lsqr_batch_kernel"), names
    _single_parity(model, r, seeds, range(3))
    # 80 groups of 8: more 16-CTA clusters than 148 SMs hold at once
    names, r = kernels_run(lambda: model.reverse_differentiate_multi(seeds))
    assert ran(names, r"lsqr_multi_kernel<8, true>"), names
    assert (r["stats"][:, 1] == 3).all()
    _single_parity(model, r, seeds, (0, 333, 639))
    # operator above the cluster route's limit (work = 2 nnz + n + 2 m > 512 Ki)
    d = bench_data.conic_config4(n=20000, n_zero=2000, n_nonneg=16000, n_soc=1200, soc_dim=10, nnz_per_row=10, seed=6)
    assert 2 * d["A"].nnz + d["A"].shape[1] + 2 * d["A"].shape[0] > 512 * 1024
    model = _model(ctx, d)
    model.tolerances = tol
    seeds = np.random.default_rng(5).normal(size=(8, d["A"].shape[1]))
    names, r = kernels_run(lambda: model.reverse_differentiate_multi(seeds))
    assert ran(names, r"lsqr_multi_kernel<8, false>") and not ran(names, r"lsqr_multi_kernel<\d, true>"), names
    _single_parity(model, r, seeds, (0, 7))
    # PSD cones
    d = PROBLEMS["psd4_7"]()
    model = _model(ctx, d)
    model.tolerances = tol
    dAs, dbs, dcs, seeds = _directions(d, 5, 8)
    names, f = kernels_run(lambda: model.forward_differentiate_multi(dAs, dbs, dcs))
    assert ran(names, r"lsqr_multi_kernel<8, false>") and not ran(names, r"lsqr_multi_kernel<\d, true>"), names
    for j in range(5):
        model.forward_differentiate(dAs[j], dbs[j], dcs[j])
        assert rel(f["dx"][j], model.forward_variable_primal()) <= 1e-9


def test_multi_bad_input(ctx):
    capi = diffopt_b200.submodule("_capi")
    fresh = diffopt_b200.Context(0)
    seeds = np.ones((2, 5))
    out = np.empty((2, 100))
    rc = fresh.lib.diffopt_b200_conic_reverse_multi(fresh.h, 2, capi.ptr(seeds), 1e-8, 1e-8, 1e8, 0, capi.ptr(out), None,
                                                    None, None, capi.HOST)
    assert rc == -1 and "conic_setup" in fresh.lib.diffopt_b200_last_error(fresh.h).decode()
    rc = fresh.lib.diffopt_b200_conic_forward_multi(fresh.h, 2, None, None, None, 1e-8, 1e-8, 1e8, 0, capi.ptr(out), None,
                                                    None, capi.HOST)
    assert rc == -1 and "conic_setup" in fresh.lib.diffopt_b200_last_error(fresh.h).decode()
    d = PROBLEMS["exp_pow"]()
    model = _model(ctx, d)
    model.vp()
    m, n = d["A"].shape
    assert ctx.lib.diffopt_b200_conic_reverse_multi(ctx.h, -1, capi.ptr(seeds), 1e-8, 1e-8, 1e8, 0, None, None, None, None,
                                                    capi.HOST) == -1
    assert ctx.lib.diffopt_b200_conic_forward_multi(ctx.h, -1, None, None, None, 1e-8, 1e-8, 1e8, 0, None, None, None,
                                                    capi.HOST) == -1
    assert ctx.lib.diffopt_b200_conic_reverse_multi(ctx.h, 0, None, 1e-8, 1e-8, 1e8, 0, None, None, None, None, capi.HOST) == 0
    assert ctx.lib.diffopt_b200_conic_forward_multi(ctx.h, 0, None, None, None, 1e-8, 1e-8, 1e8, 0, None, None, None,
                                                    capi.HOST) == 0
    for i, j in ((m + 1, 1), (1, n + 1), (0, 1), (1, 0)):
        arrs = (np.array([0, 0, 1], np.int64), np.array([i], np.int64), np.array([j], np.int64), np.array([1.0]))
        coo = capi.CooBatch(*[a.ctypes.data for a in arrs])
        dx = np.empty((2, n))
        rc = ctx.lib.diffopt_b200_conic_forward_multi(ctx.h, 2, capi.C.addressof(coo), None, None, 1e-8, 1e-8, 1e8, 0,
                                                      capi.ptr(dx), None, None, capi.HOST)
        assert rc == -1 and "outside" in ctx.lib.diffopt_b200_last_error(ctx.h).decode(), (i, j)
    # the model is still usable after the refusals
    f = model.forward_differentiate_multi([None, sp.eye(m, n).tocsc()], k=2)
    assert not f["dx"][0].any() and f["dx"][1].any()
