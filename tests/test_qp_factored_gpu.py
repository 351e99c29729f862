"""Factorise once, solve many directions: diffopt_b200_qp_batch_factorize + qp_batch_reverse_multi / qp_batch_forward_multi.

Every (instance, direction) of a multi call must match the oracle (relative error <= 1e-8, as every direct solve here) and
the per-direction qp_batch_forward / qp_batch_reverse result on the same setup (<= 1e-12: the stored-factor sweeps sum in
another order than the fused kernels).
"""
import numpy as np
import pytest
import scipy.sparse as sp

import bench_data
import diffopt_b200
from oracle import qp as oqp

pytestmark = pytest.mark.gpu
RTOL_DIRECT = 1e-8
RTOL_SAME_SETUP = 1e-12


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


def rel_err(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm(a - b, axis=-1) / np.maximum(np.linalg.norm(b, axis=-1), 1e-300)


def _batch(ctx, d):
    return diffopt_b200.submodule("qp").QPBatch(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"])


def _directions(B, k, n, m, p, seed, density=0.1, duplicates=False):
    """k random forward directions per instance: sparse dQ (symmetric), dG, dA as B*k scipy matrices in slot order b*k + j,
    dense dq, dh, db (B, k, .); `duplicates`: every matrix also carries one entry twice, split in two halves."""
    rng = np.random.default_rng(seed)

    def mats(rows, sym):
        out = []
        for _ in range(B * k):
            X = rng.standard_normal((rows, n)) * (rng.random((rows, n)) < density)
            if sym:
                X = (X + X.T) / 2
            M = sp.coo_matrix(X)
            if duplicates and rows:
                i, j, v = int(rng.integers(rows)), int(rng.integers(n)), float(rng.standard_normal())
                extra = [(i, j, v / 2), (i, j, v / 2)] + ([(j, i, v / 2), (j, i, v / 2)] if sym else [])
                M = sp.coo_matrix((np.r_[M.data, [e[2] for e in extra]], (np.r_[M.row, [e[0] for e in extra]],
                                                                         np.r_[M.col, [e[1] for e in extra]])), shape=(rows, n))
            out.append(M)
        return out
    return dict(dQ=mats(n, True), dG=mats(m, False) if m else None, dA=mats(p, False) if p else None,
                dq=rng.standard_normal((B, k, n)), dh=rng.standard_normal((B, k, m)), db=rng.standard_normal((B, k, p)))


def _dense(mats, B, k, j, rows, n):
    """direction j of every instance as a dense (B, rows, n) array"""
    if mats is None or rows == 0:
        return np.zeros((B, rows, n))
    return np.stack([mats[b * k + j].toarray() for b in range(B)])


def _forward_multi(batch, k, dirs):
    return np.concatenate(batch.forward_multi(k, dQ=dirs["dQ"], dq=dirs["dq"], dG=dirs["dG"], dh=dirs["dh"], dA=dirs["dA"],
                                              db=dirs["db"]), axis=-1)


def _per_direction(batch, k, dirs, seeds):
    """the same k directions through qp_batch_forward / qp_batch_reverse, one call each: (fwd, rev) [B][k][N]"""
    B, n, m, p = batch.B, batch.n, batch.m, batch.p
    fwd, rev = [], []
    for j in range(k):
        f = batch.forward(_dense(dirs["dQ"], B, k, j, n, n), dirs["dq"][:, j], _dense(dirs["dG"], B, k, j, m, n), dirs["dh"][:, j],
                          _dense(dirs["dA"], B, k, j, p, n), dirs["db"][:, j])
        fwd.append(np.concatenate(f, axis=1))
        rev.append(np.concatenate(batch.reverse(seeds[:, j]), axis=1))
    return np.stack(fwd, axis=1), np.stack(rev, axis=1)


def _oracle(d, k, dirs, seeds):
    B, n = d["z"].shape
    m, p = d["lam"].shape[1], d["nu"].shape[1]
    fwd, rev = np.empty((B, k, n + m + p)), np.empty((B, k, n + m + p))
    for j in range(k):
        dQ, dG, dA = (_dense(dirs["dQ"], B, k, j, n, n), _dense(dirs["dG"], B, k, j, m, n), _dense(dirs["dA"], B, k, j, p, n))
        f, r = oqp.batch_forward_reverse(d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], seeds[:, j], dQ, dirs["dq"][:, j],
                                         dG, dirs["dh"][:, j], dA, dirs["db"][:, j])
        fwd[:, j], rev[:, j] = f, r
    return fwd, rev


SHAPES = [(64, 64, 16, 16), (16, 16, 4, 4), (100, 50, 0, 10), (50, 100, 10, 20), (7, 9, 0, 3), (5, 0, 2, 0), (3, 0, 0, 0),
          (1, 1, 0, 1), (100, 100, 10, 15)]


@pytest.mark.parametrize("k", [1, 5, 8, 33])
@pytest.mark.parametrize("n,m,p,na", SHAPES)
def test_multi_directions_match_oracle_and_per_direction_calls(ctx, n, m, p, na, k):
    B = 5
    d = bench_data.qp_batch(B, n, m, p, n_active=na, seed0=11000 + n + m + k)
    batch = _batch(ctx, d)
    batch.factorize()
    nrej, nt_cap, kern = ctx.qp_last_stats()
    assert kern == 3 and nrej == 0 and nt_cap == (((n + 7) // 8) * 8 + na + p + 7) // 8, (nrej, nt_cap, kern)
    dirs = _directions(B, k, n, m, p, seed=k + n)
    seeds = np.random.default_rng(k + m).standard_normal((B, k, n))
    fwd = _forward_multi(batch, k, dirs)
    rev = np.concatenate(batch.reverse_multi(seeds), axis=-1)
    of, orv = _oracle(d, k, dirs, seeds)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT
    assert rel_err(rev, orv).max() <= RTOL_DIRECT
    pf, pr = _per_direction(batch, k, dirs, seeds)
    assert rel_err(fwd, pf).max() <= RTOL_SAME_SETUP
    assert rel_err(rev, pr).max() <= RTOL_SAME_SETUP


@pytest.mark.parametrize("n,m,p,na", [(64, 64, 16, 16), (100, 50, 0, 10)])
def test_many_instances_per_cta(ctx, n, m, p, na):
    """A batch larger than the grid: every CTA of the store and solve kernels serves several instances in turn."""
    B, k = 1500, 3
    d = bench_data.qp_batch_fast(B, n, m, p, n_active=na, seed=16000 + n)
    batch = _batch(ctx, d)
    batch.factorize()
    assert ctx.qp_last_stats()[0] == 0
    dirs = _directions(B, k, n, m, p, seed=17, density=0.02)
    seeds = np.random.default_rng(18).standard_normal((B, k, n))
    fwd = _forward_multi(batch, k, dirs)
    rev = np.concatenate(batch.reverse_multi(seeds), axis=-1)
    pf, pr = _per_direction(batch, k, dirs, seeds)
    assert rel_err(fwd, pf).max() <= RTOL_SAME_SETUP
    assert rel_err(rev, pr).max() <= RTOL_SAME_SETUP
    sl = np.r_[0:3, 700:703, B - 3:B]
    sub = {kk: v[sl] for kk, v in d.items()}
    sdirs = {kk: (None if dirs[kk] is None else [dirs[kk][b * k + j] for b in sl for j in range(k)] if kk in ("dQ", "dG", "dA")
                  else dirs[kk][sl]) for kk in dirs}
    of, orv = _oracle(sub, k, sdirs, seeds[sl])
    assert rel_err(fwd[sl], of).max() <= RTOL_DIRECT and rel_err(rev[sl], orv).max() <= RTOL_DIRECT


def test_largest_reduced_system_is_served_from_the_stored_factor(ctx):
    """n=100, m=100, p=10 with interior-point-style duals (no exact zeros: every inequality is in the reduced system, order
    214): the stored factor still fits shared memory next to the right-hand-side blocks (fewer blocks per CTA)."""
    B, k, n, m, p = 4, 17, 100, 100, 10
    d = bench_data.qp_batch(B, n, m, p, n_active=15, seed0=11500)
    act = d["lam"] > 0
    d["lam"] = np.where(act, d["lam"], 1e-9)
    slack = np.einsum("bij,bj->bi", d["G"], d["z"]) - d["h"]
    d["h"] = np.einsum("bij,bj->bi", d["G"], d["z"]) - np.where(act, -1e-9, slack)
    batch = _batch(ctx, d)
    batch.factorize()
    assert ctx.qp_last_stats() == (0, 27, 3)
    dirs = _directions(B, k, n, m, p, seed=5)
    seeds = np.random.default_rng(6).standard_normal((B, k, n))
    fwd = _forward_multi(batch, k, dirs)
    rev = np.concatenate(batch.reverse_multi(seeds), axis=-1)
    of, orv = _oracle(d, k, dirs, seeds)
    assert rel_err(fwd, of).max() <= RTOL_DIRECT and rel_err(rev, orv).max() <= RTOL_DIRECT
    pf, pr = _per_direction(batch, k, dirs, seeds)
    assert rel_err(fwd, pf).max() <= RTOL_SAME_SETUP and rel_err(rev, pr).max() <= RTOL_SAME_SETUP


def test_jacobian_transpose_identity(ctx):
    """Forward mode solves with LHS', reverse mode with LHS: with unit dq directions and unit seeds,
    fwd(e_i).dz[j] == rev(e_j).dz[i]."""
    B, n, m, p = 6, 64, 64, 16
    d = bench_data.qp_batch(B, n, m, p, seed0=12000)
    batch = _batch(ctx, d)
    batch.factorize()
    E = np.broadcast_to(np.eye(n), (B, n, n)).copy()
    fz = batch.forward_multi(n, dq=E)[0]       # [b][i][j] = fwd(e_i).dz[j]
    rz = batch.reverse_multi(E)[0]             # [b][j][i] = rev(e_j).dz[i]
    diff = np.abs(fz - rz.transpose(0, 2, 1)).max(axis=(1, 2)) / np.abs(fz).max(axis=(1, 2))
    assert diff.max() <= RTOL_SAME_SETUP


def test_forward_reverse_inner_product_identity(ctx):
    """test/utils.jl:331-337: <dz_fwd, seed> = <rhs_fwd, x_rev> for random triplet directions with duplicated triplets."""
    B, k, n, m, p = 8, 6, 33, 47, 5
    d = bench_data.qp_batch(B, n, m, p, n_active=11, seed0=12500)
    batch = _batch(ctx, d)
    batch.factorize()
    dirs = _directions(B, k, n, m, p, seed=9, density=0.05, duplicates=True)
    seeds = np.random.default_rng(10).standard_normal((B, k, n))
    fwd = _forward_multi(batch, k, dirs)
    rev = np.concatenate(batch.reverse_multi(seeds), axis=-1)
    for j in range(k):
        dQ, dG, dA = (_dense(dirs["dQ"], B, k, j, n, n), _dense(dirs["dG"], B, k, j, m, n), _dense(dirs["dA"], B, k, j, p, n))
        for b in range(B):
            rf = oqp.forward_rhs(d["z"][b], d["lam"][b], d["nu"][b], dQ[b], dirs["dq"][b, j], dG[b], dirs["dh"][b, j], dA[b],
                                 dirs["db"][b, j])
            lhs = fwd[b, j, :n] @ seeds[b, j]
            rhs = rf @ rev[b, j]
            assert abs(lhs - rhs) <= 1e-9 * max(abs(lhs), 1.0)


def test_mixed_batch_rejects_singular_instances_and_stats(ctx):
    """Regular instances next to instances the pivot-free factorisation cannot take -- semidefinite Q, a rank-deficient
    active set (two identical active rows: singular up to rounding), an active set beyond shared memory, interior-point-style
    duals (every row in the reduced system, beyond shared memory at m = 120) -- and one exactly singular instance (a zero
    equality row).  Wrong-sign duals on rows with zero slack leave the symmetric form quasi-definite: that instance stays on
    the stored factor.  The rejects are solved by the pivoted LU, the singular ones are reported by factorize and by the multi
    calls, every other instance gives its per-direction result."""
    B, k, n, m, p = 10, 5, 100, 120, 10
    d = bench_data.qp_batch(B, n, m, p, n_active=15, seed0=13000)
    rng = np.random.default_rng(13)
    L = rng.standard_normal((n, 90))
    d["Q"][2] = L @ L.T / 90                                     # positive semidefinite, rank 90
    act = np.flatnonzero(d["lam"][3] > 0)
    d["G"][3, act[1]] = d["G"][3, act[0]]                        # rank-deficient active set
    d["h"][3, act[1]] = d["h"][3, act[0]]
    d["lam"][4][d["lam"][4] == 0] = 0.7                          # every row in the reduced system (slack < 0 keeps K regular)
    a5 = d["lam"][5] > 0
    slack = np.einsum("ij,j->i", d["G"][5], d["z"][5]) - d["h"][5]
    d["lam"][5] = np.where(a5, d["lam"][5], 1e-9)
    d["h"][5] = d["G"][5] @ d["z"][5] - np.where(a5, -1e-9, slack)
    d["A"][6][1] = 0.0                                           # a zero equality row: exactly singular
    d["lam"][7] = -d["lam"][7]                                   # wrong-sign duals
    batch = _batch(ctx, d)
    with pytest.raises(diffopt_b200.SingularException) as e:
        batch.factorize()
    info = batch.info.copy()
    # the rank-deficient active set is singular only up to rounding: the pivoted LU may or may not meet an exact zero
    assert info[6] > 0 and not np.delete(info, [3, 6]).any()
    first = 3 if info[3] else 6
    assert e.value.instance == first
    nrej, nt_cap, kern = ctx.qp_last_stats()
    assert kern == 3 and nrej == 5 and nt_cap == 28, (nrej, nt_cap, kern)
    dirs = _directions(B, k, n, m, p, seed=14)
    seeds = np.random.default_rng(15).standard_normal((B, k, n))
    with pytest.raises(diffopt_b200.SingularException) as e:
        batch.reverse_multi(seeds)
    assert e.value.instance == first
    # the raw calls return first singular instance + 1 and still fill in every other instance
    capi = diffopt_b200.submodule("_capi")
    qpm = diffopt_b200.submodule("qp")
    N = n + m + p
    keep = []
    fm, rm = np.empty((B, k, N)), np.empty((B, k, N))
    assert ctx.lib.diffopt_b200_qp_batch_forward_multi(ctx.h, k, *_coo_args(qpm, capi, dirs, B * k, n, m, p, keep), capi.ptr(fm),
                                                       capi.HOST) == first + 1
    assert ctx.lib.diffopt_b200_qp_batch_reverse_multi(ctx.h, k, capi.ptr(np.ascontiguousarray(seeds)), capi.ptr(rm), capi.HOST) == first + 1
    # per direction on the same data: qp_batch_reverse, and qp_batch_solve_coo with the same triplets
    pf, pr = np.empty((B, k, N)), np.empty((B, k, N))
    for j in range(k):
        one = {kk: dirs[kk][j::k] for kk in ("dQ", "dG", "dA")}
        pf[:, j], _, _ = qpm.solve_batch_coo(ctx, d["Q"], d["G"], d["A"], d["h"], d["z"], d["lam"], d["nu"], dQ=one["dQ"],
                                             dq=dirs["dq"][:, j], dG=one["dG"], dh=dirs["dh"][:, j], dA=one["dA"], db=dirs["db"][:, j])
        out, inf = np.empty((B, N)), np.zeros(B, np.int32)
        rc = ctx.lib.diffopt_b200_qp_batch_reverse(ctx.h, capi.ptr(np.ascontiguousarray(seeds[:, j])), capi.ptr(out), capi.ptr(inf),
                                                   capi.HOST)
        assert rc == first + 1
        pr[:, j] = out
    ok = np.array([b for b in range(B) if b not in (3, 6)])
    assert rel_err(fm[ok], pf[ok]).max() <= RTOL_SAME_SETUP
    assert rel_err(rm[ok], pr[ok]).max() <= RTOL_SAME_SETUP
    sub = {kk: v[ok] for kk, v in d.items()}
    sdirs = {kk: ([dirs[kk][b * k + j] for b in ok for j in range(k)] if kk in ("dQ", "dG", "dA") else dirs[kk][ok]) for kk in dirs}
    of, orv = _oracle(sub, k, sdirs, seeds[ok])
    assert rel_err(fm[ok], of).max() <= RTOL_DIRECT and rel_err(rm[ok], orv).max() <= RTOL_DIRECT


def _coo_args(qpm, capi, dirs, slots, n, m, p, keep):
    """(dQ, dq, dG, dh, dA, db) pointers of qp_batch_forward_multi for host arrays; `keep` holds the buffers alive"""
    def coo(mats, rows):
        if mats is None or rows == 0:
            return None
        arrs = qpm.coo_batch(mats, slots)
        st = capi.CooBatch(*[a.ctypes.data for a in arrs])
        keep.append((arrs, st))
        return capi.C.addressof(st)

    def vec(v):
        if v is None or v.shape[-1] == 0:
            return None
        a = np.ascontiguousarray(v)
        keep.append(a)
        return capi.ptr(a)
    return (coo(dirs["dQ"], n), vec(dirs["dq"]), coo(dirs["dG"], m), vec(dirs["dh"]), coo(dirs["dA"], p), vec(dirs["db"]))


def test_lifecycle_errors(ctx):
    """A multi call before factorize, or after a new setup, is an argument error that names the missing step; k = 0 returns
    nothing; an out-of-range triplet is an argument error."""
    B, n, m, p = 4, 12, 9, 3
    d = bench_data.qp_batch(B, n, m, p, n_active=3, seed0=14000)
    capi = diffopt_b200.submodule("_capi")
    batch = _batch(ctx, d)
    seeds = np.ones((B, 2, n))
    with pytest.raises(diffopt_b200.DiffOptB200Error, match="factorize"):
        batch.reverse_multi(seeds)
    with pytest.raises(diffopt_b200.DiffOptB200Error, match="factorize"):
        batch.forward_multi(2, dq=seeds)
    batch.factorize()
    assert batch.reverse_multi(np.zeros((B, 0, n)))[0].shape == (B, 0, n)
    assert ctx.lib.diffopt_b200_qp_batch_reverse_multi(ctx.h, 0, None, None, capi.HOST) == 0
    assert ctx.lib.diffopt_b200_qp_batch_forward_multi(ctx.h, 0, None, None, None, None, None, None, None, capi.HOST) == 0
    bad = sp.coo_matrix((np.array([1.0]), (np.array([m]), np.array([0]))), shape=(m + 1, n))   # row m + 1 of an m-row matrix
    with pytest.raises(diffopt_b200.DiffOptB200Error, match="outside") as e:
        batch.forward_multi(1, dG=[bad] + [sp.coo_matrix((m, n))] * (B - 1))
    assert e.value.code == -1
    batch.reverse_multi(seeds)
    _batch(ctx, d)                                              # a new setup drops the stored factor
    with pytest.raises(diffopt_b200.DiffOptB200Error, match="factorize"):
        batch.reverse_multi(seeds)


def test_multi_calls_are_bitwise_reproducible(ctx):
    B, k, n, m, p = 64, 12, 64, 64, 16
    d = bench_data.qp_batch_fast(B)
    batch = _batch(ctx, d)
    batch.factorize()
    dirs = _directions(B, k, n, m, p, seed=21, density=0.05)
    seeds = np.random.default_rng(22).standard_normal((B, k, n))
    f1, r1 = _forward_multi(batch, k, dirs), np.concatenate(batch.reverse_multi(seeds), axis=-1)
    f2, r2 = _forward_multi(batch, k, dirs), np.concatenate(batch.reverse_multi(seeds), axis=-1)
    assert np.array_equal(f1, f2) and np.array_equal(r1, r2)


def test_device_memory_gives_the_host_results(ctx):
    """memspace = DEVICE: info, seeds, directions (triplets included) and outputs in device memory, consumed in place."""
    import torch
    capi = diffopt_b200.submodule("_capi")
    qpm = diffopt_b200.submodule("qp")
    B, k, n, m, p = 16, 9, 33, 47, 5
    d = bench_data.qp_batch(B, n, m, p, n_active=11, seed0=15000)
    batch = _batch(ctx, d)
    batch.factorize()
    dirs = _directions(B, k, n, m, p, seed=23)
    seeds = np.random.default_rng(24).standard_normal((B, k, n))
    fh = _forward_multi(batch, k, dirs)
    rh = np.concatenate(batch.reverse_multi(seeds), axis=-1)
    dev = torch.device("cuda", 0)
    info = torch.full((B,), 7, dtype=torch.int32, device=dev)
    assert ctx.lib.diffopt_b200_qp_batch_factorize(ctx.h, capi.ptr(info), capi.DEVICE) == 0
    assert not info.any()
    N = n + m + p
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    out = torch.empty((B, k, N), dtype=torch.float64, device=dev)
    sd = T(seeds)
    assert ctx.lib.diffopt_b200_qp_batch_reverse_multi(ctx.h, k, capi.ptr(sd), capi.ptr(out), capi.DEVICE) == 0
    assert np.array_equal(out.cpu().numpy(), rh)
    keep = []

    def coo(mats):
        arrs = [T(a) for a in qpm.coo_batch(mats, B * k)]
        st = capi.CooBatch(*[a.data_ptr() for a in arrs])
        keep.append((arrs, st))
        return capi.C.addressof(st)
    dq, dh, db = T(dirs["dq"]), T(dirs["dh"]), T(dirs["db"])
    rc = ctx.lib.diffopt_b200_qp_batch_forward_multi(ctx.h, k, coo(dirs["dQ"]), capi.ptr(dq), coo(dirs["dG"]), capi.ptr(dh),
                                                     coo(dirs["dA"]), capi.ptr(db), capi.ptr(out), capi.DEVICE)
    assert rc == 0
    assert np.array_equal(out.cpu().numpy(), fh)
